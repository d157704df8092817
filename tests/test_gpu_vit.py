"""GPU numerics for the tensor-core path: GEMM and attention against float64 truth computed from the exact 16-bit
operands, at error bounds derived from the kernels' rounding steps; the whole ViT-L/14 tower + heads vs the fp32 oracle
(north_star: cosine >= 0.999, aesthetic +-0.01).  tests/test_gpu_vit_f64.py checks the tower's whole residual stream
against float64; tests/test_gpu_vit_heads_f64.py the tail, the stored-embedding heads, LayerNorm and im2col."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _rand_bf16(shape, seed, scale=1.0, dtype=None):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(shape, device="cuda", generator=g) * scale).to(dtype or torch.bfloat16)


U32 = 2.0 ** -24          # unit roundoff of fp32
# fp32 accumulation bound |err| <= C_ACC * u32 * sqrt(K) * (|A| @ |B|^T).  tcgen05 (kind::f16) adds the exact products of
# 16 k-values per instruction into the fp32 accumulator, so an output sees K / 16 accumulator additions.  Each errs by at
# most one ulp (2 u32, truncating adders included) of a partial sum bounded by G = (|A| @ |B|^T); independent errors give a
# standard deviation of at most 2 u32 sqrt(K / 16) G = 0.5 u32 sqrt(K) G, and the rounding inside each 16-product block
# adds at most a same-size term.  C_ACC = 4 is four such standard deviations of the sum of both: a kernel that drops or
# repeats one k-block of 64 is off by ~G / sqrt(K / 64), orders of magnitude outside.
C_ACC = 4.0
ERF_AS = 1.5e-7          # |error| of the Abramowitz & Stegun 7.1.26 erf the GELU epilogue evaluates


def _half_ulp16(x, dtype):
    """Half an ulp of the 16-bit format at |x| (float64 tensor), subnormals included."""
    import torch
    p, emin = (11, -14) if dtype == torch.float16 else (8, -126)
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** emin)))
    return torch.exp2(e - p)


def _gelu64(x):
    import torch
    return 0.5 * x * (1.0 + torch.special.erf(x * 0.5 ** 0.5))


def _gemm_bound(g, k, pre, extra_abs):
    """fp32-level bound of one output: accumulation (C_ACC) + one rounding per epilogue add (pre = |acc| + |bias|,
    extra_abs = |residual| or 0; each add rounds once in fp32)."""
    return C_ACC * U32 * k ** 0.5 * g + 2 * U32 * (pre + extra_abs)


def _check_gemm(got, truth, bound, what):
    import torch
    err = (got.double() - truth).abs()
    ratio = float((err / bound.clamp_min(1e-300)).max())
    assert bool((err <= bound).all()), f"{what}: max err/bound {ratio:.3g}, max err {float(err.max()):.3g}"
    print(f"gemm {what} {got.dtype} {tuple(got.shape)}: max err/bound {ratio:.3g}")
    return ratio


def _gemm_truth(a, b, bias):
    """float64 truth from the exact 16-bit operands: acc = A B^T, G = |A| |B|^T, and acc + bias."""
    a64, b64 = a.double(), b.double()
    acc = a64 @ b64.T
    g = a64.abs() @ b64.abs().T
    return acc, g, acc + bias.double()


def _check_all_epilogues(a, b, bias, res, out_views=None):
    """Every epilogue of ops.gemm_bf16 on (a, b) against float64 truth.  out_views: optional factory of output tensors
    (a window into a larger buffer) per output dtype; returns the largest err/bound ratio."""
    import torch
    from facet_b200 import ops
    k = a.shape[1]
    t16 = a.dtype
    acc, g, pre = _gemm_truth(a, b, bias)
    mk = out_views or (lambda dt: None)
    ratios = []
    b_f32 = _gemm_bound(g, k, g, 0)
    ratios.append(_check_gemm(ops.gemm_bf16(a, b, ops.GEMM_F32, out=mk(torch.float32)), acc, b_f32, "F32"))
    b_bias = _gemm_bound(g, k, g + bias.double().abs(), 0)
    ratios.append(_check_gemm(ops.gemm_bf16(a, b, ops.GEMM_F32, bias=bias, out=mk(torch.float32)), pre, b_bias, "F32+bias"))
    got = ops.gemm_bf16(a, b, ops.GEMM_BIAS_BF16, bias=bias, out=mk(t16))
    ratios.append(_check_gemm(got, pre, b_bias + _half_ulp16(torch.maximum(pre.abs(), got.double().abs()), t16), "BIAS_16"))
    # GELU: the fp32 pre-activation error passes through gelu' (|gelu'| <= 1.13), then the erf approximation
    # (0.5 |x| * ERF_AS), its fp32 evaluation (rcp / ex2 approximations and nine FMAs, 16 u32 of 0.5 |x|), one rounding
    # of the result, and the 16-bit output rounding
    got = ops.gemm_bf16(a, b, ops.GEMM_BIAS_GELU_BF16, bias=bias, out=mk(t16))
    gt = _gelu64(pre)
    bound = 1.13 * b_bias + 0.5 * pre.abs() * (ERF_AS + 16 * U32) + U32 * gt.abs() + _half_ulp16(torch.maximum(gt.abs(), got.double().abs()), t16)
    ratios.append(_check_gemm(got, gt, bound, "BIAS_GELU_16"))
    out = mk(torch.float32)
    if out is None:
        out = res.clone()
    else:
        out.copy_(res)
    ops.gemm_bf16(a, b, ops.GEMM_BIAS_RESIDUAL_F32, bias=bias, residual=out, out=out)   # in place
    ratios.append(_check_gemm(out, pre + res.double(), _gemm_bound(g, k, g + bias.double().abs(), res.double().abs()), "BIAS_RESIDUAL_F32"))
    return max(ratios)


# ViT-L/14 tower GEMMs at batch 128 and 512 (M = 257 B rows; the patch GEMM has 256 B rows, K padded to 640).  At these
# sizes every persistent CTA / CTA pair walks many tiles: the TMEM accumulator double buffer is reused with both
# phases, and 257 B is odd in 128-row tiles, so each tile column ends on a CTA-pair rank whose rows all lie past M.
TOWER_GEMMS = [(257 * bt, n, k) for bt in (128, 512) for (n, k) in ((3072, 1024), (1024, 1024), (4096, 1024), (1024, 4096))] + \
              [(256 * 128, 1024, 640), (256 * 512, 1024, 640)]


@pytest.mark.parametrize("m,n,k", [(128, 256, 64), (300, 256, 128), (1000, 768, 1024), (257 * 8, 3072, 1024),
                                   (2056, 1024, 4096), (129, 32, 640), (4096, 1024, 640),
                                   # CTA-pair form (M >= 512, N % 256 == 0): exactly two pairs, an odd number of row
                                   # tiles with a ragged last one, many column tiles, a single k-block, a long K
                                   (512, 256, 64), (513, 512, 128), (640, 4096, 1024), (1283, 256, 64), (768, 256, 8192),
                                   # 57 row tiles (the last odd and ragged: 37 rows) x 8 column tiles = 232 tile pairs, at
                                   # least 3 per CTA pair on 148 SMs; 5 k-blocks against 6 stages, so the ring wraps mid-tile
                                   (7205, 2048, 320)] + TOWER_GEMMS)
@pytest.mark.parametrize("dt", ["bf16", "fp16"])
def test_gemm_all_epilogues(m, n, k, dt):
    """Every epilogue against float64 truth from the exact 16-bit operands, at bounds derived from the kernel's rounding
    steps (see C_ACC): fp32 accumulation, one rounding per epilogue add, the erf approximation, the 16-bit output."""
    import torch
    dtype = torch.float16 if dt == "fp16" else torch.bfloat16
    a, b = _rand_bf16((m, k), 1, dtype=dtype), _rand_bf16((n, k), 2, scale=k ** -0.5, dtype=dtype)
    bias = torch.randn(n, device="cuda")
    res = torch.randn(m, n, device="cuda")
    _check_all_epilogues(a, b, bias, res)


@pytest.mark.parametrize("m,n", [(300, 512), (1283, 512)], ids=["single-cta", "cta-pair"])
@pytest.mark.parametrize("dt", ["bf16", "fp16"])
def test_gemm_windows(m, n, dt):
    """Strided operands: A is a column slice (lda > K, base 16 bytes into its row) and every output is a window
    (ldo > N) into a canary-filled buffer with rows before and after it.  Nothing outside the [M, N] window may change.
    M = 300 runs the single-CTA form for every epilogue; M = 1283 runs the CTA-pair form for the 16-bit and residual
    epilogues (and the single-CTA form for the fp32 ones)."""
    import torch
    dtype = torch.float16 if dt == "fp16" else torch.bfloat16
    k = 192
    a_big = _rand_bf16((m, k + 72), 11, dtype=dtype)
    a = a_big[:, 8:8 + k]
    assert a.stride(0) == k + 72 and not a.is_contiguous()
    b = _rand_bf16((n, k), 12, scale=k ** -0.5, dtype=dtype)
    bias = torch.randn(n, device="cuda")
    res = torch.randn(m, n, device="cuda")
    bufs = []

    def window(odt):
        pad_r, pad_c = 3, 40          # rows before / after, extra columns: ldo = N + 40 (16-byte multiple for both widths)
        big = torch.full((m + 2 * pad_r, n + pad_c), -7.25, dtype=odt, device="cuda")
        view = big[pad_r:pad_r + m, 8:8 + n]
        bufs.append((big, big.clone(), pad_r))
        return view

    _check_all_epilogues(a, b, bias, res, out_views=window)
    for big, before, pad_r in bufs:
        inside = torch.zeros_like(big, dtype=torch.bool)
        inside[pad_r:pad_r + m, 8:8 + n] = True
        iv = torch.int16 if big.element_size() == 2 else torch.int32
        assert torch.equal(big.view(iv)[~inside], before.view(iv)[~inside]), "a GEMM wrote outside its output window"


def test_gemm_pair_kernel_on_two_devices():
    """Kernel attributes and the co-resident cluster count are per device: the same CTA-pair GEMM (every 16-bit and
    residual epilogue) on cuda:0 and then on cuda:1 in one process gives identical results."""
    import torch
    from facet_b200 import ops
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    outs = []
    for dev in ("cuda:0", "cuda:1"):
        g = torch.Generator(device="cpu").manual_seed(9)
        a = torch.randn((1283, 1024), generator=g).to(dev, torch.float16)
        b = (torch.randn((3072, 1024), generator=g) / 32).to(dev, torch.float16)
        bias = torch.randn(3072, generator=g).to(dev)
        res = torch.randn((1283, 3072), generator=g).to(dev)
        got = [ops.gemm_bf16(a, b, mode, bias=bias) for mode in (ops.GEMM_BIAS_BF16, ops.GEMM_BIAS_GELU_BF16)]
        out = res.clone()
        ops.gemm_bf16(a, b, ops.GEMM_BIAS_RESIDUAL_F32, bias=bias, residual=out, out=out)
        outs.append([t.cpu() for t in got + [out]])
    for x0, x1 in zip(*outs):
        assert torch.equal(x0, x1)


def _attn_truth(qkv, bsz):
    """float64 softmax(Q K^T / 8) V per (image, head) from the exact 16-bit qkv rows, and the scale of the bound,
    sum_j p_j |v_j| / l.  Both [bsz*257, 1024]."""
    import torch
    o, sv = [], []
    for b0 in range(0, bsz, 32):
        q, k, v = qkv[b0 * 257:min(bsz, b0 + 32) * 257].double().reshape(-1, 257, 3, 16, 64).unbind(2)
        p = torch.softmax(torch.einsum("bqhd,bkhd->bhqk", q, k) * 0.125, dim=-1)
        o.append(torch.einsum("bhqk,bkhd->bqhd", p, v).reshape(-1, 1024))
        sv.append(torch.einsum("bhqk,bkhd->bqhd", p, v.abs()).reshape(-1, 1024))
    return torch.cat(o), torch.cat(sv)


def _check_attention(got, qkv, bsz):
    """Per element: half an ulp of the 16-bit output + 2 u16 sum_j p_j |v_j| / l.  P is rounded to 16 bits before the
    P V product (relative error u16 per term, against a row sum l taken before rounding); the second u16 covers the fp32
    score / exponential / accumulation errors, which are orders of magnitude smaller."""
    import torch
    u16 = 2.0 ** -11 if qkv.dtype == torch.float16 else 2.0 ** -8
    o, sv = _attn_truth(qkv, bsz)
    got = got.reshape(bsz * 257, 1024).double()
    bound = _half_ulp16(torch.maximum(o.abs(), got.abs()), qkv.dtype) + 2 * u16 * sv
    err = (got - o).abs()
    bad = ~(err <= bound)
    if bool(bad.any()):
        r, c = (int(i) for i in bad.nonzero()[0])
        raise AssertionError(f"attention: {int(bad.sum())} elements out of bound, first at token {r % 257} of image "
                             f"{r // 257}, head {c // 64}, dim {c % 64}: got {float(got[r, c])}, truth {float(o[r, c])}, "
                             f"max err/bound {float((err / bound).max()):.3g}")
    print(f"attention {qkv.dtype} batch {bsz}: max err/bound {float((err / bound).max()):.3g}")
    return float((err / bound).max())


def _check_attention_unbiased(got, qkv, bsz):
    """Round-to-nearest errors have zero mean.  The error towards larger |o|, in units of u16 sum_j p_j |v_j| / l,
    averages to ~0 (measured within 0.003 on B200 at every batch >= 3); a biased rounding step, such as truncating P to
    16 bits, moves it to about -0.5."""
    import torch
    u16 = 2.0 ** -11 if qkv.dtype == torch.float16 else 2.0 ** -8
    o, sv = _attn_truth(qkv, bsz)
    bias = float(((got.reshape(bsz * 257, 1024).double() - o) * torch.sign(o) / (u16 * sv)).mean())
    print(f"attention {qkv.dtype} batch {bsz}: mean signed error {bias:.3g} u16 units")
    assert abs(bias) <= 0.1, f"attention error is biased: mean {bias:.3g} u16 units"
    return bias


def _qkv_with_v_offsets(bsz, seed, dtype, scale=1.5):
    """Random qkv whose V block of each (image, head) pair carries its own offset (-4 .. 4 in steps of 0.5): a tile or
    phase leaking in from another pair then shows as an O(1) error instead of averaging away."""
    import torch
    qkv = _rand_bf16((bsz * 257, 3072), seed, scale=scale, dtype=torch.float32)
    pair = torch.arange(bsz * 16, device="cuda")
    off = 0.5 * ((pair * 5) % 17 - 8).float()
    qkv.view(bsz, 257, 3, 16, 64)[:, :, 2] += off.view(bsz, 1, 16, 1)
    return qkv.to(dtype)


def _attention_case(bsz, dtype):
    import torch
    from facet_b200 import ops
    qkv = _qkv_with_v_offsets(bsz, 5 + bsz, dtype)
    got = ops.vit_attention(qkv, bsz)
    _check_attention(got, qkv, bsz)
    if bsz >= 3:
        _check_attention_unbiased(got, qkv, bsz)


@pytest.mark.parametrize("variant", ["tcgen05-bf16", "tcgen05-fp16"])
def test_attention_vs_torch(variant):
    """float64 truth at batch 3: 48 (image, head) pairs, one per persistent group."""
    import torch
    _attention_case(3, torch.float16 if variant.endswith("fp16") else torch.bfloat16)


@pytest.mark.parametrize("bsz", [1, 19, 128, 512])
@pytest.mark.parametrize("dt", ["bf16", "fp16"])
def test_attention_batches(bsz, dt):
    """float64 truth at batches where each persistent group handles 1 pair (1), 1 or 2 (19: only 8 groups take a
    second pair), 6-7 (128) and 27-28 (512): later trips round the loop flip the TMA / score / PV barrier phases and
    prefetch the next pair into tiles that are still being read."""
    import torch
    _attention_case(bsz, torch.float16 if dt == "fp16" else torch.bfloat16)


CRAFT_POS = [0, 127, 128, 255, 256]     # half 0 / half 1 of the keys (tile 0 / tile 1 of the queries), and token 256


def _crafted_qkv(kind, dtype):
    """One image per position in CRAFT_POS, all 16 heads alike up to the per-pair V offsets.
    key:   every query row aligned with one dominant key, 64 * 4 * 4 = 1024 above the rest: after the / 8 scale the others
           are 2^-180 of it and ex2.approx.ftz flushes them to zero, so each output row is that key's V row;
    query: one dominant query row, aligned with key (pos + 77) % 257 only; the other rows stay near uniform;
    zero:  q = 0, so every output row is the plain mean of the 257 V rows (key 256 counted exactly once)."""
    import torch
    n = len(CRAFT_POS)
    qkv = _qkv_with_v_offsets(n, 23, torch.float32).float()
    q = qkv.view(n, 257, 3, 16, 64)[:, :, 0]
    k = qkv.view(n, 257, 3, 16, 64)[:, :, 1]
    if kind == "zero":
        q.zero_()
    else:
        q.mul_(0.1 / 1.5)
        k.mul_(0.1 / 1.5)
        for i, pos in enumerate(CRAFT_POS):
            if kind == "key":
                q[i] = 4.0
                k[i, pos] = 4.0
            else:
                q[i, pos] = 4.0
                k[i, (pos + 77) % 257] = 4.0
    return qkv.to(dtype)


@pytest.mark.parametrize("kind", ["key", "query", "zero"])
@pytest.mark.parametrize("dt", ["bf16", "fp16"])
def test_attention_crafted_scores(kind, dt):
    import torch
    from facet_b200 import ops
    dtype = torch.float16 if dt == "fp16" else torch.bfloat16
    qkv = _crafted_qkv(kind, dtype)
    n = len(CRAFT_POS)
    got = ops.vit_attention(qkv, n)
    _check_attention(got, qkv, n)
    v = qkv.view(n, 257, 3, 16, 64)[:, :, 2].reshape(n, 257, 1024)
    if kind == "key":
        # one-hot softmax: the output row is the dominant key's V row, exactly
        for i, pos in enumerate(CRAFT_POS):
            assert torch.equal(got.view(n, 257, 1024)[i], v[i, pos].expand(257, 1024)), f"dominant key {pos}"
    elif kind == "query":
        for i, pos in enumerate(CRAFT_POS):
            assert torch.equal(got.view(n, 257, 1024)[i, pos], v[i, (pos + 77) % 257]), f"dominant query row {pos}"


@pytest.mark.parametrize("dt", ["bf16", "fp16"])
def test_attention_output_window(dt):
    """fb_vit_attention[_f16] writes exactly batch * 257 rows of 1024: a canary-filled buffer with rows before and after
    the output keeps them."""
    import ctypes as C
    import torch
    from facet_b200 import _lib
    dtype = torch.float16 if dt == "fp16" else torch.bfloat16
    bsz, before, after = 19, 3, 5
    qkv = _qkv_with_v_offsets(bsz, 31, dtype)
    buf = torch.full(((bsz * 257) + before + after, 1024), -3.5, dtype=dtype, device="cuda")
    ref = buf.clone()
    lib = _lib.load()
    fn = lib.fb_vit_attention_f16 if dtype == torch.float16 else lib.fb_vit_attention
    out = buf[before:before + bsz * 257]
    _lib.check(fn(C.c_void_p(qkv.data_ptr()), bsz, C.c_void_p(out.data_ptr()), _lib.stream_ptr()), "fb_vit_attention")
    torch.cuda.synchronize()
    assert torch.equal(buf[:before].view(torch.int16), ref[:before].view(torch.int16))
    assert torch.equal(buf[before + bsz * 257:].view(torch.int16), ref[before + bsz * 257:].view(torch.int16))
    _check_attention(out, qkv, bsz)


@pytest.mark.parametrize("dt,aest_tol", [
    ("fp16", 0.01),
    # bf16 operands: cosine 0.999999 but 0.004 mean / 0.013 max aesthetic error on this random-init head (measured,
    # DESIGN.md §7) — outside the north_star's 0.01, so the bound is NOT loosened and the case is an expected failure.
    # The default (and everything the bench measures) is fp16, the precision the reference itself runs on CUDA
    # (`self.model.half()`, processing/scorer.py:515).
    pytest.param("bf16", 0.01, marks=pytest.mark.xfail(reason="bf16 activations: aesthetic max error 0.013 > 0.01", strict=False)),
])
def test_vit_tower_vs_fp32_oracle(dt, aest_tol):
    """north_star tolerances: cosine >= 0.999 and aesthetic within 0.01 of the fp32 oracle."""
    import torch
    from facet_b200.models.clip_vit import ClipVitL14, random_state_dict
    from oracle import vit_torch
    sd = random_state_dict(0)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(8, 3, 224, 224, generator=g)
    tags = torch.nn.functional.normalize(torch.randn(240, 768, generator=torch.Generator().manual_seed(7)), dim=-1)
    sd_gpu = {k: v.cuda() for k, v in sd.items()}
    ref = vit_torch.score_batch(sd_gpu, x.cuda(), tags.cuda())       # fp32 oracle (TF32 off by default)
    model = ClipVitL14(sd, tag_embeddings=tags.numpy(), dtype=dt)
    out = model.encode(x.cuda())
    cos = torch.nn.functional.cosine_similarity(out["embedding"], ref["embedding"], dim=-1)
    assert float(cos.min()) >= 0.999, cos
    aest = ((out["aesthetic_raw"] + 1) * 5).clamp(0, 10)
    assert float((aest - ref["aesthetic"]).abs().max()) <= aest_tol, (aest, ref["aesthetic"])
    assert float((out["tag_sims"] - ref["tag_sims"]).abs().max()) <= 5e-3
    nrm = out["embedding"].norm(dim=-1)
    torch.testing.assert_close(nrm, torch.ones_like(nrm), rtol=1e-5, atol=1e-5)
