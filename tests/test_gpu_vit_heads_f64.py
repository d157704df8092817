"""GPU: the kernels that turn the residual stream into what the pass stores for every photo, against float64.

vit_tail_kernel (ln_post on the class token, projection to 768, F.normalize, the MLP aesthetic head, the tag
similarities), embedding_heads_kernel (the same heads on stored vectors), layernorm_kernel (every output format and the
assembly mode) and im2col_patch14_kernel.  Truth is float64 computed from the exact fp32 inputs the kernel read.  Every
output gets two checks:

1. Per element, |kernel - truth| <= a bound derived from the kernel's rounding steps (below).  A correct kernel cannot
   fail it.
2. Over the call, the kernel's RMS error is at most K_FP32 times that of the same formula in fp32 PyTorch (TF32 off),
   or of u32 x RMS of the output's scale (the absolute-value evaluation the bound multiplies) where that is larger.
   Check 1 is a worst case and cannot tell an fp32 sum from one whose input was rounded to 16 bits first; that rounding
   is ~1e4 x larger than fp32 rounding and fails check 2.  The floor is there because, when every row is alike (one
   image, a constant row, the zero vector), the fp32 evaluation can be exact by chance.

Bound.  gamma(n) = n u / (1 - n u), u = 2^-24, bounds a chain of n fp32 roundings (Higham 2002, Lemma 3.1): a sum
or dot product whose every term passes through at most n roundings errs by at most gamma(n) sum |terms|.  The chains,
read off csrc/vit.cu:
  layernorm_kernel (one warp per row)    mean and sum of squares: 32 values per lane serially + 5-step butterfly (N_LN)
  vit_tail_kernel  (24 warps)            LayerNorm sums: 2 values per thread (the squares: product + add), a 5-step
                                         butterfly, 24 warp partials serially (N_TAIL_LN); the norm the same (N_NORM);
                                         projection: 8 accumulators of 128 FMAs + a 3-level tree (N_PROJ)
  both head kernels                      hidden units and prompts: 24 FMAs per lane + 5-step butterfly (N_DOT);
                                         final head sum: 8 per lane + 5 + b2 (N_HEAD)
The library is built without --use_fast_math, so sqrtf and the division are correctly rounded (relative error <= u);
rsqrtf errs by up to 2 ulp (relative <= 4u), its CUDA Math API bound.  Each stage's input error propagates through the
next stage's absolute weights: |proj|^T |dy|, |W1| |dfeat| (then through ReLU, 1-Lipschitz), |w2|, |T| |demb|.
LayerNorm: sum_j (x_j - mean) = 0 exactly, so a mean error dm enters the sum of squares only through
sum_j (d_hat_j - d_j)^2, i.e. at second order; the first-order term is the subtraction's own rounding.  The kernel adds
1e-5f, which is 1e-5 rounded to fp32, and that add rounds again: two roundings of their own.
"""
import ctypes as C
import functools

import pytest

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24
EPS = 1e-5
K_FP32 = 4.0
WIDTH, TOKENS, DIM = 1024, 257, 768
N_LN, N_TAIL_LN, N_PROJ, N_NORM, N_DOT, N_HEAD = 37, 31, 131, 30, 29, 14


def _gamma(n):
    return n * U32 / (1 - n * U32)


def _half_ulp16(x, dtype):
    """Half an ulp of the 16-bit format at |x| (float64 tensor), subnormals included."""
    import torch
    p, emin = (11, -14) if dtype == torch.float16 else (8, -126)
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** emin)))
    return torch.exp2(e - p)


class _Fp32:
    """fp32 matmuls without TF32 for the plain fp32 evaluation of check 2."""

    def __enter__(self):
        import torch
        self.prec = torch.get_float32_matmul_precision()
        torch.set_float32_matmul_precision("highest")

    def __exit__(self, *exc):
        import torch
        torch.set_float32_matmul_precision(self.prec)


def _check(what, got, truth, bound, fp32, scale):
    """Check 1 (per element, |got - truth| <= bound) and check 2 (RMS error <= K_FP32 x that of the fp32 evaluation,
    floored at u32 RMS(scale)).  Returns the largest err / bound."""
    import torch
    err = (got.double() - truth).abs()
    bad = ~(err <= bound)
    q = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, float("inf"), 0.0))
    ratio = float(q.max()) if q.numel() else 0.0
    if bool(bad.any()):
        i = tuple(int(t) for t in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements out of bound, first at {i}: got "
                             f"{float(got[i])}, truth {float(truth[i])}, bound {float(bound[i]):.3g}; max err/bound {ratio:.3g}")
    rms_k = float(err.pow(2).mean().sqrt())
    rms_32 = float((fp32.double() - truth).pow(2).mean().sqrt())
    floor = U32 * float(scale.pow(2).mean().sqrt())
    ref = max(rms_32, floor)
    print(f"{what}: max err/bound {ratio:.3g}, RMS error kernel/fp32 {rms_k / rms_32 if rms_32 else 0.0:.3g}, "
          f"kernel/floor {rms_k / floor if floor else 0.0:.3g}")
    assert rms_k <= K_FP32 * ref, f"{what}: RMS error {rms_k:.3g} > {K_FP32} x max(fp32 evaluation's, floor) {ref:.3g}"
    return ratio


# ------------------------------------------------------------------------------------------------------------------
# float64 truth and bounds


def _layernorm_truth(x, g, b, n_sum):
    """LayerNorm of the rows of x (float64, the exact fp32 inputs), eps 1e-5: (truth, bound of an fp32 output, scale).
    n_sum: rounding chain of the kernel's mean and sum of squares."""
    import torch
    n = x.shape[1]
    mean = x.mean(1, keepdim=True)
    d = x - mean
    s2 = d.pow(2).sum(1, keepdim=True)
    big_d = s2 / n + EPS
    rstd = big_d.rsqrt()
    y = d * rstd * g + b
    dm = _gamma(n_sum) * x.abs().mean(1, keepdim=True)            # |mean_hat - mean|
    dd = dm * (1 + U32) + U32 * d.abs()                             # |d_hat - d|: the mean error + the subtraction's rounding
    # sum d_hat^2 - sum d^2 = 2 sum d r + sum (d_hat - d)^2 (r: rounding of the subtraction, |r| <= u |d_hat|), plus the
    # summation's own gamma(n_sum) sum d_hat^2
    dvar = (_gamma(n_sum) * (d.abs() + dd).pow(2).sum(1, keepdim=True) + 2 * U32 * s2
            + 2 * U32 * dm * d.abs().sum(1, keepdim=True) + dd.pow(2).sum(1, keepdim=True)) / n
    d_big_d = dvar + U32 * EPS + U32 * (big_d + dvar + U32 * EPS)     # 1e-5f and the add each round once
    r = d_big_d / big_d
    assert bool((r < 0.5).all())
    rel = (1 - r).rsqrt() * (1 + 4 * U32) - 1                       # rstd: the variance's error + 2 ulp of rsqrtf
    # (d_hat * rstd_hat) * g + b: three roundings
    k = (1 + rel) * (1 + U32) ** 2
    e1 = g.abs() * rstd * (dd * k + d.abs() * (k - 1))
    bound = e1 + U32 * (y.abs() + e1)
    return y, bound, g.abs() * d.abs() * rstd + b.abs()


def _dot_truth(e, ee, t):
    """e @ t^T with e known to within ee per element: (truth, bound, scale); prompts chain N_DOT."""
    at = t.abs().T
    return e @ t.T, ee @ at + _gamma(N_DOT) * ((e.abs() + ee) @ at), e.abs() @ at


def _head_truth(f, ef, w1, b1, w2, b2):
    """raw = w2 . relu(W1 f + b1) + b2 with f known to within ef per element: (truth, bound, scale)."""
    import torch
    aw1 = w1.abs().T
    h = f @ w1.T + b1
    eh = ef @ aw1 + _gamma(N_DOT) * ((f.abs() + ef) @ aw1)
    ehb = eh + U32 * (h.abs() + eh)                                 # + b1
    hid = torch.relu(h) * w2
    ehid = w2.abs() * ehb * (1 + U32) + U32 * hid.abs()             # ReLU is 1-Lipschitz; * w2 rounds once
    raw = hid.sum(1) + b2
    eraw = ehid.sum(1) + _gamma(N_HEAD) * (hid.abs().sum(1) + ehid.sum(1) + b2.abs())
    return raw, eraw, ((f.abs() @ aw1 + b1.abs()) * w2.abs()).sum(1) + b2.abs()


def _head_fp32(f, w1, b1, w2, b2):
    import torch
    return torch.relu(f @ w1.T + b1) @ w2 + b2


# ------------------------------------------------------------------------------------------------------------------
# vit_tail_kernel, through ClipVitL14.encode


@functools.lru_cache(maxsize=2)
def _state_dict(layers):
    from facet_b200.models.clip_vit import random_state_dict
    return random_state_dict(0, layers=layers)


def _quiet_blocks(sd):
    """out_proj and c_proj weights and biases zero: every block adds exactly 0 to the residual stream, so the final
    stream is the ln_pre output bit for bit."""
    import torch
    sd = dict(sd)
    for k in sd:
        if k.startswith("transformer.resblocks.") and (".attn.out_proj." in k or ".mlp.c_proj." in k):
            sd[k] = torch.zeros_like(sd[k])
    return sd


def _tags(n):
    import torch
    if n == 0:
        return None
    return torch.nn.functional.normalize(torch.randn(n, DIM, generator=torch.Generator().manual_seed(7)), dim=-1).cuda()


def _tower_tail(sd, batch, dt, tags, seed=3):
    """Run the tower; returns the tail's input (the class rows of the final fp32 residual stream, read from offset 0 of
    the workspace) and the heads."""
    import torch
    from facet_b200.models.clip_vit import ClipVitL14
    model = ClipVitL14(sd, tag_embeddings=tags.cpu().numpy() if tags is not None else None, dtype=dt)
    x = torch.randn(batch, 3, 224, 224, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))
    out = model.encode(x)
    cls = model._ws[: batch * TOKENS * WIDTH * 4].view(torch.float32).view(batch, TOKENS, WIDTH)[:, 0].clone()
    return cls, out


def _check_tail(sd, cls, out, tags, what):
    """Every output of vit_tail_kernel against float64 from its input rows cls [B, 1024]."""
    import torch
    import torch.nn.functional as F
    w = {k: sd[k].to("cuda", torch.float64) for k in ("ln_post.weight", "ln_post.bias", "proj", "aesthetic_head.0.weight",
                                                       "aesthetic_head.0.bias", "aesthetic_head.2.weight", "aesthetic_head.2.bias")}
    head = (w["aesthetic_head.0.weight"], w["aesthetic_head.0.bias"], w["aesthetic_head.2.weight"].reshape(-1),
            w["aesthetic_head.2.bias"])
    y, ey, _ = _layernorm_truth(cls.double(), w["ln_post.weight"], w["ln_post.bias"], N_TAIL_LN)
    ap = w["proj"].abs()
    f = y @ w["proj"]
    ef = ey @ ap + _gamma(N_PROJ) * ((y.abs() + ey) @ ap)
    fs = y.abs() @ ap
    tot = f.pow(2).sum(1, keepdim=True)
    inv = 1 / tot.sqrt().clamp_min(1e-12)
    emb = f * inv
    # inv_hat / inv = (1 + theta)^(-1/2) / (1 + sqrt's rounding) * (1 + division's rounding), |theta| <= rt
    dtot = _gamma(N_NORM) * (f.abs() + ef).pow(2).sum(1, keepdim=True) + (2 * f.abs() * ef + ef.pow(2)).sum(1, keepdim=True)
    zero = tot == 0
    rt = torch.where(zero, 0.0, dtot / torch.where(zero, 1.0, tot))
    assert bool((rt < 0.5).all())
    rel = torch.where(zero, 0.0, (1 - rt).rsqrt() / (1 - U32) * (1 + U32) - 1)
    k = (1 + rel) * (1 + U32)                                       # f_hat * inv_hat rounds once
    eemb = inv * (ef * k + f.abs() * (k - 1))
    raw, eraw, raws = _head_truth(f, ef, *head)
    with _Fp32(), torch.no_grad():
        w32 = {k: v.float() for k, v in w.items()}
        y32 = F.layer_norm(cls, (WIDTH,), w32["ln_post.weight"], w32["ln_post.bias"], EPS)
        f32 = y32 @ w32["proj"]
        e32 = F.normalize(f32, dim=-1)
        raw32 = _head_fp32(f32, *(t.float() for t in head))
        sims32 = e32 @ tags.T if tags is not None else None
    r = [_check(f"tail {what} features", out["features"], f, ef, f32, fs),
         _check(f"tail {what} embedding", out["embedding"], emb, eemb, e32, fs * inv),
         _check(f"tail {what} aesthetic_raw", out["aesthetic_raw"], raw, eraw, raw32, raws)]
    if tags is None:
        assert out["tag_sims"] is None
    else:
        s, es, ss = _dot_truth(emb, eemb, tags.double())
        r.append(_check(f"tail {what} tag_sims", out["tag_sims"], s, es, sims32, ss))
    return r


@pytest.mark.parametrize("batch", [1, 3, 129, 512])
@pytest.mark.parametrize("dt", ["fp16", "bf16"])
def test_tail_batches(dt, batch):
    """A 2-layer tower at the batch sizes of a single photo, a ragged small batch and the pass's large batches; the tail
    is fp32 whatever the tower's 16-bit format."""
    tags = _tags(240)
    sd = _state_dict(2)
    cls, out = _tower_tail(sd, batch, dt, tags)
    _check_tail(sd, cls, out, tags, f"{dt} batch {batch}")


@pytest.mark.parametrize("ntags", [0, 1, 23, 24, 25, 1000])
def test_tail_prompt_counts(ntags):
    """The prompt loop strides by the 24 warps: no prompt, one, one warp short of / exactly / one past a full stride,
    and 1000 (42 trips, the last partial)."""
    tags = _tags(ntags)
    sd = _state_dict(1)
    cls, out = _tower_tail(sd, 3, "fp16", tags)
    _check_tail(sd, cls, out, tags, f"{ntags} prompts")


# Value of the constant rows.  A power of two, so every partial sum of the mean is exact too: an M with a full mantissa
# leaves the two-pass mean an ulp off, which rsqrt(eps) = 316 magnifies, inside check 1's bound but not comparable with
# fp32 PyTorch (Welford), whose mean of a constant row is exact.  Small, because check 1 must allow a mean error of
# gamma(n) M, and 316 gamma(31) M has to stay small against ln_post's bias (~0.02) for the norm's bound to hold.
CONST_ROW = 2.0 ** -6

# ln_pre.weight = s * w, ln_pre.bias = M + s * b (w ~ 1, b ~ 0.02 from the random init): with the blocks quiet, the class
# row the tail reads is that affine map of a unit-variance row
CRAFTED = {
    "eps": (1e-3, 0.0),        # row std ~1e-3: variance 1e-6 against eps = 1e-5
    "cancel": (1.0, 16.0),     # mean / std = 16: the cancellation case of the two-pass variance
    "const": (0.0, CONST_ROW),  # variance exactly 0

}


@pytest.mark.parametrize("kind", sorted(CRAFTED))
@pytest.mark.parametrize("dt", ["fp16", "bf16"])
def test_tail_crafted_rows(dt, kind):
    s, m = CRAFTED[kind]
    sd = _quiet_blocks(_state_dict(1))
    sd["ln_pre.weight"] = sd["ln_pre.weight"] * s
    sd["ln_pre.bias"] = sd["ln_pre.bias"] * s + m
    tags = _tags(240)
    cls, out = _tower_tail(sd, 3, dt, tags)
    std, mean = cls.double().std(1), cls.double().mean(1)
    if kind == "const":
        assert bool((cls == m).all()), "the quiet blocks changed the residual stream"
    elif kind == "eps":
        assert float(std.max()) < 2e-3
    else:
        assert float((mean / std).min()) > 12
    _check_tail(sd, cls, out, tags, f"{dt} {kind} row")


def test_tail_zero_features():
    """proj = 0: the features are exactly 0.  F.normalize's floor max(||f||, 1e-12) keeps the embedding and the tag
    similarities exactly 0 (the bound is 0 there), and the head sees the zero vector."""
    import torch
    sd = dict(_state_dict(1))
    sd["proj"] = torch.zeros_like(sd["proj"])
    tags = _tags(240)
    cls, out = _tower_tail(sd, 3, "fp16", tags)
    for k in ("features", "embedding", "tag_sims"):
        assert bool((out[k] == 0).all()), k
    _check_tail(sd, cls, out, tags, "zero features")


# ------------------------------------------------------------------------------------------------------------------
# embedding_heads_kernel (ops.embedding_heads)


def _head_weights():
    import torch
    g = torch.Generator(device="cuda").manual_seed(4)
    w1, b1 = torch.randn(256, DIM, device="cuda", generator=g) * DIM ** -0.5, torch.randn(256, device="cuda", generator=g) * 0.02
    w2, b2 = torch.randn(256, device="cuda", generator=g) * 256 ** -0.5, torch.randn(1, device="cuda", generator=g) * 0.02
    return w1, b1, w2, b2


def _stored_vectors(n, kind):
    """unit: L2-normalised rows as the pass stores them, through the clip_embedding BLOB format and back; nonunit: norms
    0.1 .. 10; zero: the zero vector."""
    import numpy as np
    import torch
    from facet_b200.utils.embedding import bytes_to_embedding, embedding_to_bytes
    g = torch.Generator(device="cuda").manual_seed(11 + n)
    v = torch.randn(n, DIM, device="cuda", generator=g)
    if kind == "zero":
        return torch.zeros_like(v)
    if kind == "nonunit":
        return v * torch.logspace(-1, 1, n, device="cuda")[:, None] / DIM ** 0.5
    rows = [bytes_to_embedding(embedding_to_bytes(r), dim=DIM) for r in torch.nn.functional.normalize(v, dim=-1).cpu().numpy()]
    return torch.from_numpy(np.stack(rows)).cuda()


@pytest.mark.parametrize("kind", ["unit", "nonunit", "zero"])
@pytest.mark.parametrize("n", [1, 7, 5000])
def test_embedding_heads(n, kind):
    """Head only, prompts only and both, at prompt counts around the 8-warp stride (1, 7, 8, 9) and 240."""
    import torch
    from facet_b200 import ops
    v = _stored_vectors(n, kind)
    head = _head_weights()
    tags = _tags(240)
    v64, z = v.double(), torch.zeros_like(v, dtype=torch.float64)
    raw, eraw, raws = _head_truth(v64, z, *(t.double() for t in head))
    s, es, ss = _dot_truth(v64, z, tags.double())
    with _Fp32():
        raw32, sims32 = _head_fp32(v, *head), v @ tags.T
    got_raw, got_sims = ops.embedding_heads(v, head=head)
    assert got_sims is None
    _check(f"heads n={n} {kind} head only: aesthetic_raw", got_raw, raw, eraw, raw32, raws)
    for nt in (1, 7, 8, 9, 240):
        t = tags[:nt].contiguous()
        for with_head in (False, True):
            got_raw, got_sims = ops.embedding_heads(v, head=head if with_head else None, tag_embeddings=t)
            what = f"heads n={n} {kind} {nt} prompts{' + head' if with_head else ''}"
            if with_head:
                _check(f"{what}: aesthetic_raw", got_raw, raw, eraw, raw32, raws)
            else:
                assert got_raw is None
            _check(f"{what}: tag_sims", got_sims, s[:, :nt], es[:, :nt], sims32[:, :nt], ss[:, :nt])
    if kind == "zero":
        assert bool((got_sims == 0).all())


# ------------------------------------------------------------------------------------------------------------------
# layernorm_kernel (ops.vit_layernorm)


def _ln_rows(kind, rows, seed):
    import torch
    r = torch.randn(rows, WIDTH, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))
    if kind == "plain":
        return r * 3 + 0.5
    if kind == "eps":
        return r * 1e-3                    # variance 1e-6 against eps = 1e-5
    if kind == "cancel":
        return r + 16                      # mean / std = 16
    return torch.full_like(r, CONST_ROW)


def _ln_params():
    import torch
    g = torch.Generator(device="cuda").manual_seed(21)
    return 1 + 0.5 * torch.randn(WIDTH, device="cuda", generator=g), torch.randn(WIDTH, device="cuda", generator=g)


def _check_layernorm(x, got, fmt, what, tok=None):
    """tok: the assembled rows when they differ from x."""
    import torch
    import torch.nn.functional as F
    g, b = _ln_params()
    src = x if tok is None else tok
    y, bound, scale = _layernorm_truth(src.double(), g.double(), b.double(), N_LN)
    y32 = F.layer_norm(src, (WIDTH,), g, b, EPS)
    if fmt != torch.float32:
        bound = bound + _half_ulp16(torch.maximum(y.abs(), got.double().abs()), fmt)
        y32 = y32.to(fmt)
    return _check(what, got, y, bound, y32, scale)


OUT_FORMATS = {"fp32": 0, "bf16": 1, "fp16": 2}


@pytest.mark.parametrize("kind", ["plain", "eps", "cancel", "const"])
@pytest.mark.parametrize("out", sorted(OUT_FORMATS))
def test_layernorm(out, kind):
    """Every output format at 1, 7 (one partial block of 8 warps), 8 and 3 * 257 rows, and 3 * 257 rows read from a column
    slice (ld_in = 1088 > 1024)."""
    import torch
    from facet_b200 import ops
    fmt = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[out]
    g, b = _ln_params()
    for rows in (1, 7, 8, 3 * TOKENS):
        x = _ln_rows(kind, rows, rows)
        _check_layernorm(x, ops.vit_layernorm(x, g, b, out_bf16=OUT_FORMATS[out]), fmt, f"layernorm {out} {kind} {rows} rows")
    big = torch.full((3 * TOKENS, WIDTH + 64), float("nan"), device="cuda")
    big[:, 32:32 + WIDTH] = _ln_rows(kind, 3 * TOKENS, 5)
    x = big[:, 32:32 + WIDTH]
    assert x.stride(0) == WIDTH + 64
    _check_layernorm(x, ops.vit_layernorm(x, g, b, out_bf16=OUT_FORMATS[out]), fmt, f"layernorm {out} {kind} strided")


def test_layernorm_assembly():
    """Assembly mode (ln_pre): row t of image b is (t == 0 ? class_emb : patch row b * 256 + t - 1) + pos[t].  The kernel
    adds in fp32, as PyTorch does (both round to nearest), so the assembled rows are its exact inputs."""
    import torch
    from facet_b200 import ops
    gen = torch.Generator(device="cuda").manual_seed(8)
    pe = torch.randn(3 * 256, WIDTH, device="cuda", generator=gen)
    cls, pos = torch.randn(WIDTH, device="cuda", generator=gen), torch.randn(TOKENS, WIDTH, device="cuda", generator=gen)
    g, b = _ln_params()
    tok = (torch.cat([cls.expand(3, 1, WIDTH), pe.reshape(3, 256, WIDTH)], 1) + pos).reshape(-1, WIDTH)
    got = ops.vit_layernorm(pe, g, b, out_bf16=False, class_emb=cls, pos_emb=pos, rows=3 * TOKENS)
    _check_layernorm(pe, got, torch.float32, "layernorm assembly batch 3", tok=tok)


# ------------------------------------------------------------------------------------------------------------------
# im2col_patch14_kernel


def _pixels(batch, t16, seed=5):
    """Random pixels; every 5th lies exactly halfway between two neighbouring 16-bit values, so round-to-nearest-even is
    pinned, not only round-to-nearest."""
    import torch
    x = torch.randn(batch, 3, 224, 224, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed)) * 2
    a = x.view(-1)[::5].to(t16)
    nxt = (a.view(torch.int16) + 1).view(t16)
    x.view(-1)[::5] = ((a.double() + nxt.double()) / 2).float()
    return x


def _unfold16(x, t16):
    import torch.nn.functional as F
    return F.unfold(x, 14, stride=14).transpose(1, 2).reshape(-1, 588).to(t16)


# the grid is capped at sm_count * 32 blocks of 256 threads, 14.8 images per sweep on 148 SMs: 37 images take 2.5 sweeps
@pytest.mark.parametrize("batch", [1, 37])
def test_im2col_bit_exact(batch):
    """fb_vit_im2col (bf16, the format its C entry writes) equals F.unfold(x, 14, stride=14) rounded to bf16 bit for
    bit; columns 588..639 are +0 and nothing past the batch * 256 rows is written."""
    import torch
    from facet_b200 import _lib
    x = _pixels(batch, torch.bfloat16)
    buf = torch.full((batch * 256 + 4, 640), -7.25, dtype=torch.bfloat16, device="cuda")
    lib = _lib.load()
    _lib.check(lib.fb_vit_im2col(C.c_void_p(x.data_ptr()), batch, C.c_void_p(buf.data_ptr()), _lib.stream_ptr()), "fb_vit_im2col")
    torch.cuda.synchronize()
    out = buf[: batch * 256].view(torch.int16)
    assert torch.equal(out[:, :588], _unfold16(x, torch.bfloat16).view(torch.int16))
    assert bool((out[:, 588:] == 0).all())
    assert bool((buf[batch * 256:] == -7.25).all())


def test_im2col_fp16_through_tower():
    """The fp16 instantiation runs only inside fb_vit_forward.  conv1 = [I_588; 0] makes the patch GEMM copy the im2col
    rows exactly (one non-zero exact product per output) and quiet blocks keep the ln_pre output as the final residual
    stream, so every row read back is the fp32 LayerNorm of (rounded pixels, 436 zeros) + pos.  A pixel rounded the
    wrong way moves its row's output by an fp16 ulp x rstd, ~1e3 x the LayerNorm bound."""
    import torch
    from facet_b200.models.clip_vit import ClipVitL14
    sd = _quiet_blocks(_state_dict(1))
    sd["conv1.weight"] = torch.eye(WIDTH, 588).reshape(WIDTH, 3, 14, 14)
    batch = 37
    x = _pixels(batch, torch.float16)
    model = ClipVitL14(sd, dtype="fp16", fold_layernorm=False)
    model.encode(x)
    m = batch * TOKENS
    got = model._ws[: m * WIDTH * 4].view(torch.float32).view(m, WIDTH)
    pe = torch.zeros(batch * 256, WIDTH, device="cuda")
    pe[:, :588] = _unfold16(x, torch.float16).float()
    cls, pos = sd["class_embedding"].cuda(), sd["positional_embedding"].cuda()
    tok = (torch.cat([cls.expand(batch, 1, WIDTH), pe.view(batch, 256, WIDTH)], 1) + pos).reshape(-1, WIDTH)
    g, b = sd["ln_pre.weight"].cuda(), sd["ln_pre.bias"].cuda()
    y, bound, scale = _layernorm_truth(tok.double(), g.double(), b.double(), N_LN)
    _check("im2col fp16 -> ln_pre, batch 37", got, y, bound, torch.nn.functional.layer_norm(tok, (WIDTH,), g, b, EPS), scale)
