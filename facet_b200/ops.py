"""Thin host wrappers over the C ABI: torch tensors in, torch tensors out.

torch is used for device memory and streams only; every kernel is in libfacet_b200.so.
All functions run on the current CUDA stream of the current device and raise RuntimeError on
failure.  Nothing here falls back to the CPU.
"""
from __future__ import annotations

import ctypes as C
from typing import Sequence

import numpy as np

from . import _lib
from .analyzers._closed_form import TechStats

HS_BINS = 180 * 256
# Largest pair list a single call materialises (2^28 pairs = 2 GiB of int32 pairs).  A degenerate library (many
# identical hashes / embeddings) has O(n^2) pairs; the reference merely runs slowly there, this raises a clear
# error instead of an opaque allocation failure.
MAX_PAIRS = 1 << 28


def _grown_cap(needed: int, what: str) -> int:
    if needed > MAX_PAIRS:
        raise RuntimeError(f"{what}: {needed} pairs exceed the {MAX_PAIRS}-pair limit of one call "
                           "(degenerate input: deduplicate identical hashes first or split the row range)")
    return int(needed)


def _ptr(t) -> C.c_void_p:
    return C.c_void_p(t.data_ptr())


def to_device_u8(images, device=None):
    """numpy [H,W,3] / [n,H,W,3] uint8 or a CUDA tensor -> contiguous CUDA uint8 [n,H,W,3]."""
    torch = _lib.require_cuda()
    if isinstance(images, np.ndarray):
        arr = np.ascontiguousarray(images)
        if arr.dtype != np.uint8:
            raise TypeError("images must be uint8")
        t = torch.from_numpy(arr).to(device or "cuda", non_blocking=False)
    elif isinstance(images, torch.Tensor):
        if images.dtype != torch.uint8:
            raise TypeError("images must be uint8")
        t = images if images.is_cuda else images.to(device or "cuda")
        t = t.contiguous()
    else:
        raise TypeError(f"unsupported image container {type(images)!r}")
    if t.dim() == 3:
        t = t.unsqueeze(0)
    if t.dim() != 4 or t.shape[-1] != 3:
        raise ValueError(f"expected [n,H,W,3] uint8, got {tuple(t.shape)}")
    return t


def box4_multipliers(h: int, w: int) -> np.ndarray:
    """Pillow's ImagingReduce multipliers of the (full, right-edge, bottom-edge, corner) boxes of a (4, 4) reduction."""
    from .utils import thumbnail as th
    return np.array([th.reduce_multiplier(max(1, a * b)) for a, b in
                     ((4, 4), (w % 4 or 4, 4), (4, h % 4 or 4), (w % 4 or 4, h % 4 or 4))], dtype=np.uint32)


def tech_stats_raw(images, rgb_order: bool = False, force_generic: bool = False, luma_out=None, box_out=None):
    """Run the technical pass.  Returns CUDA tensors (hist256 u32->int32 view [n,256],
    hs_hist int32 [n,180,256], sums int64 [n,4], derived float64 [n,4]).  luma_out: optional CUDA uint8
    [n,H,W] tensor that receives Pillow's luma plane in the same pass (input of `phash(..., luma=...)`); box_out:
    optional CUDA uint8 [n,ceil(H/4),ceil(W/4),3] tensor that receives Pillow's (4, 4) box reduction of the frames
    (input of `thumbnails(..., reduced=...)`)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    t = to_device_u8(images)
    n, h, w, _ = t.shape
    if h < 2 or w < 2:
        raise ValueError("images must be at least 2x2 (reflect-101 borders)")
    dev = t.device
    with torch.cuda.device(dev):
        hist = torch.empty((n, 256), dtype=torch.int32, device=dev)
        hs = torch.empty((n, 180, 256), dtype=torch.int32, device=dev)
        sums = torch.empty((n, 4), dtype=torch.int64, device=dev)
        derived = torch.empty((n, 4), dtype=torch.float64, device=dev)
        st = _lib.stream_ptr()
        if box_out is not None:
            if tuple(box_out.shape) != (n, (h + 3) // 4, (w + 3) // 4, 3) or not box_out.is_contiguous():
                raise ValueError("box_out must be a contiguous [n, ceil(H/4), ceil(W/4), 3] uint8 tensor")
            mult = box4_multipliers(h, w)
            _lib.check(lib.fb_tech_stats_fused(_ptr(t), n, h, w, h * w * 3, int(bool(rgb_order)), _ptr(hist), _ptr(hs),
                                               _ptr(sums), _ptr(luma_out) if luma_out is not None else None, _ptr(box_out),
                                               mult.ctypes.data, st), "fb_tech_stats_fused")
        elif luma_out is not None:
            _lib.check(lib.fb_tech_stats_luma(_ptr(t), n, h, w, h * w * 3, int(bool(rgb_order)), _ptr(hist), _ptr(hs),
                                              _ptr(sums), int(bool(force_generic)), _ptr(luma_out), st), "fb_tech_stats_luma")
        else:
            _lib.check(lib.fb_tech_stats(_ptr(t), n, h, w, h * w * 3, int(bool(rgb_order)), _ptr(hist), _ptr(hs),
                                         _ptr(sums), int(bool(force_generic)), st), "fb_tech_stats")
        _lib.check(lib.fb_tech_derive(_ptr(hs), n, _ptr(derived), st), "fb_tech_derive")
    return hist, hs, sums, derived


def tech_stats(images, rgb_order: bool = False, want_hs: bool = False, force_generic: bool = False) -> list[TechStats]:
    """Technical pass + copy of the small per-image results to the host."""
    t = to_device_u8(images)
    n, h, w, _ = t.shape
    hist, hs, sums, derived = tech_stats_raw(t, rgb_order, force_generic)
    hist_h = hist.cpu().numpy().view(np.uint32).astype(np.int64)
    sums_h = sums.cpu().numpy()
    der_h = derived.cpu().numpy()
    hs_h = hs.cpu().numpy().view(np.uint32) if want_hs else None
    out = []
    for i in range(n):
        out.append(TechStats(height=h, width=w, hist256=hist_h[i], sum_lap=int(sums_h[i, 0]),
                             sum_lap_sq=int(sums_h[i, 1]), sum_abs_noise=int(sums_h[i, 2]),
                             hs_entropy=float(der_h[i, 0]), sum_saturation=float(der_h[i, 1]),
                             hs_hist=hs_h[i] if want_hs else None))
    return out


def tech_stats_host(images: np.ndarray, rgb_order: bool = False, want_hs: bool = False) -> list[TechStats]:
    """Same pass through fb_tech_stats_host: host numpy in, host numpy out, copies inside the call.
    This is the entry point a non-torch caller (the reference's analyzers) binds."""
    lib = _lib.load()
    arr = np.ascontiguousarray(images)
    if arr.ndim == 3:
        arr = arr[None]
    n, h, w, _ = arr.shape
    hist = np.empty((n, 256), np.uint32)
    sums = np.empty((n, 4), np.int64)
    der = np.empty((n, 4), np.float64)
    hs = np.empty((n, 180, 256), np.uint32) if want_hs else None
    _lib.check(lib.fb_tech_stats_host(arr.ctypes.data, n, h, w, int(bool(rgb_order)), hist.ctypes.data,
                                      sums.ctypes.data, der.ctypes.data, hs.ctypes.data if want_hs else None),
               "fb_tech_stats_host")
    return [TechStats(height=h, width=w, hist256=hist[i].astype(np.int64), sum_lap=int(sums[i, 0]),
                      sum_lap_sq=int(sums[i, 1]), sum_abs_noise=int(sums[i, 2]), hs_entropy=float(der[i, 0]),
                      sum_saturation=float(der[i, 1]), hs_hist=hs[i] if want_hs else None) for i in range(n)]


def gray_hsv_planes(image, rgb_order: bool = False):
    """(gray uint8 [H,W], hsv uint8 [H,W,3]) numpy arrays of one image (image_cache.py:30-31)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    t = to_device_u8(image)
    if t.shape[0] != 1:
        raise ValueError("gray_hsv_planes takes a single image")
    _, h, w, _ = t.shape
    gray = torch.empty((h, w), dtype=torch.uint8, device=t.device)
    hsv = torch.empty((h, w, 3), dtype=torch.uint8, device=t.device)
    with torch.cuda.device(t.device):
        _lib.check(lib.fb_gray_hsv(_ptr(t), h, w, int(bool(rgb_order)), _ptr(gray), _ptr(hsv), _lib.stream_ptr()),
                   "fb_gray_hsv")
    return gray.cpu().numpy(), hsv.cpu().numpy()


def gray_plane(image, rgb_order: bool = False, want_hist: bool = False):
    """CUDA uint8 [H,W] gray plane of one frame (cv2.cvtColor BGR2GRAY, composition.py:30,210) and, when
    want_hist, its 256-bin histogram as a CUDA int32 tensor."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    t = to_device_u8(image)
    if t.shape[0] != 1:
        raise ValueError("gray_plane takes a single image")
    _, h, w, _ = t.shape
    with torch.cuda.device(t.device):
        gray = torch.empty((h, w), dtype=torch.uint8, device=t.device)
        hist = torch.empty(256, dtype=torch.int32, device=t.device) if want_hist else None
        _lib.check(lib.fb_gray_plane(_ptr(t), h, w, int(bool(rgb_order)), _ptr(gray), _ptr(hist) if want_hist else None,
                                     _lib.stream_ptr()), "fb_gray_plane")
    return (gray, hist) if want_hist else gray


def canny_edges(gray, low: int, high: int, blur: bool = False, want_count: bool = False):
    """cv2.Canny(gray, low, high) of a uint8 [H,W] plane (numpy or CUDA tensor), after cv2.GaussianBlur(gray, (5, 5), 0)
    when `blur` (composition.py:215-218, :36).  Returns the CUDA uint8 [H,W] edge map (0 / 255), bit-exact with OpenCV."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    if isinstance(gray, np.ndarray):
        if gray.dtype != np.uint8 or gray.ndim != 2:
            raise TypeError("gray must be a uint8 [H,W] plane")
        g = torch.from_numpy(np.ascontiguousarray(gray)).cuda()
    else:
        if gray.dtype != torch.uint8 or gray.dim() != 2:
            raise TypeError("gray must be a uint8 [H,W] plane")
        g = (gray if gray.is_cuda else gray.cuda()).contiguous()
    h, w = g.shape
    with torch.cuda.device(g.device):
        nbytes = int(lib.fb_canny_workspace_bytes(h, w))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=g.device)
        edges = torch.empty((h, w), dtype=torch.uint8, device=g.device)
        count = torch.zeros(1, dtype=torch.int64, device=g.device) if want_count else None
        _lib.check(lib.fb_canny(_ptr(g), h, w, int(bool(blur)), int(low), int(high), _ptr(ws), nbytes, _ptr(edges),
                                _ptr(count) if want_count else None, _lib.stream_ptr()), "fb_canny")
    return (edges, count) if want_count else edges


def roi_laplacian(image, boxes: Sequence[Sequence[int]], rgb_order: bool = False) -> np.ndarray:
    """[k,3] int64 (pixel count, sum L, sum L^2) for crops x1,y1,x2,y2 of one image."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    t = to_device_u8(image)
    if t.shape[0] != 1:
        raise ValueError("roi_laplacian takes a single image")
    _, h, w, _ = t.shape
    b = torch.as_tensor(np.asarray(boxes, dtype=np.int32).reshape(-1, 4), device=t.device)
    out = torch.empty((b.shape[0], 3), dtype=torch.int64, device=t.device)
    if b.shape[0] == 0:
        return out.cpu().numpy()
    with torch.cuda.device(t.device):
        _lib.check(lib.fb_roi_laplacian(_ptr(t), h, w, int(bool(rgb_order)), _ptr(b), b.shape[0], _ptr(out),
                                        _lib.stream_ptr()), "fb_roi_laplacian")
    return out.cpu().numpy()


def hamming_pairs(hashes, max_distance: int, part: int = 0, nparts: int = 1, cap: int | None = None):
    """All (i<j) pairs of this part with popcount(h_i ^ h_j) <= max_distance, as a CUDA int32 [m,2]."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    if isinstance(hashes, np.ndarray):
        h = torch.from_numpy(np.ascontiguousarray(hashes.astype(np.uint64)).view(np.int64)).cuda()
    else:
        h = hashes.contiguous()
        if h.dtype not in (torch.int64, torch.uint64):
            raise TypeError("hashes must be 64-bit integers")
    n = h.numel()
    cap = int(cap if cap is not None else max(1 << 16, 4 * n))
    with torch.cuda.device(h.device):
        count = torch.zeros(1, dtype=torch.int64, device=h.device)
        while True:
            pairs = torch.empty((cap, 2), dtype=torch.int32, device=h.device)
            _lib.check(lib.fb_hamming_pairs(_ptr(h), n, int(max_distance), int(part), int(nparts), _ptr(pairs), cap,
                                            _ptr(count), _lib.stream_ptr()), "fb_hamming_pairs")
            m = int(count.item())
            if m <= cap:
                return pairs[:m]
            cap = _grown_cap(m, 'hamming_pairs')   # truncated: retry once with the exact size


def burst_links(hashes: np.ndarray, time_s: np.ndarray, flags: np.ndarray, lo: np.ndarray, thr: int,
                window_s: int, rapid_s: float):
    """(last_slow int32[n], rapid_pairs int32[m,2]) — see fb_burst_links."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    n = int(len(hashes))
    dev = torch.device("cuda", torch.cuda.current_device())
    h = torch.from_numpy(np.ascontiguousarray(hashes.astype(np.uint64)).view(np.int64)).to(dev)
    t = torch.from_numpy(np.ascontiguousarray(time_s.astype(np.int64))).to(dev)
    f = torch.from_numpy(np.ascontiguousarray(flags.astype(np.uint8))).to(dev)
    l = torch.from_numpy(np.ascontiguousarray(lo.astype(np.int32))).to(dev)
    last = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    count = torch.zeros(1, dtype=torch.int64, device=dev)
    cap = max(1 << 14, 4 * n)
    while True:
        rp = torch.empty((cap, 2), dtype=torch.int32, device=dev)
        _lib.check(lib.fb_burst_links(_ptr(h), _ptr(t), _ptr(f), _ptr(l), n, int(thr), int(window_s), float(rapid_s),
                                      _ptr(last), _ptr(rp), cap, _ptr(count), _lib.stream_ptr()), "fb_burst_links")
        m = int(count.item())
        if m <= cap:
            return last[:n].cpu().numpy(), rp[:m].cpu().numpy()
        cap = _grown_cap(m, 'burst_links')


_PLAN_CACHE: dict = {}


def _device_plan(height: int, width: int, out: int, device):
    torch = _lib.require_cuda()
    from .utils import resample as rs
    key = (height, width, out, str(device))
    if key not in _PLAN_CACHE:
        p = rs.plan(height, width, out)
        dev = {name: torch.from_numpy(getattr(p, name)).to(device) for name in ("hp0", "hcpad", "vbounds", "vcoef")}
        dev["tc_coef"] = torch.from_numpy(p.tc_coef).to(device) if p.tc_coef is not None else None
        dev["tc_kb0"] = torch.from_numpy(p.tc_kb0).to(device) if p.tc_kb0 is not None else None
        _PLAN_CACHE[key] = (p, dev)
    return _PLAN_CACHE[key]


def clip_preprocess(images, out_size: int = 224, mean=(0.5, 0.5, 0.5), std=(0.5, 0.5, 0.5), rgb_order: bool = False,
                    tensor_cores: bool = True):
    """Resize(out, bicubic, antialias) + CenterCrop + ToTensor + Normalize on the GPU.

    images: [n,H,W,3] uint8 (numpy or CUDA tensor; BGR unless rgb_order).  Returns a CUDA float32
    tensor [n,3,out,out] with planes R,G,B — what `scorer.preprocess` returns per image, stacked.
    """
    torch = _lib.require_cuda()
    lib = _lib.load()
    t = to_device_u8(images)
    n, h, w, _ = t.shape
    p, dev = _device_plan(h, w, out_size, t.device)
    tmp = torch.empty((n, p.rows, out_size, 3), dtype=torch.uint8, device=t.device)
    out = torch.empty((n, 3, out_size, out_size), dtype=torch.float32, device=t.device)
    use_tc = bool(tensor_cores) and dev["tc_coef"] is not None
    m = (C.c_float * 3)(*[float(v) for v in mean])
    s = (C.c_float * 3)(*[float(v) for v in std])
    with torch.cuda.device(t.device):
        _lib.check(lib.fb_clip_preprocess(_ptr(t), n, h, w, h * w * 3, int(bool(rgb_order)), out_size,
                                          _ptr(dev["hp0"]), _ptr(dev["hcpad"]), p.hgroups, p.h_px_lo, p.h_span_px,
                                          _ptr(dev["vbounds"]), _ptr(dev["vcoef"]), p.vk, p.row0, p.rows,
                                          C.cast(m, C.c_void_p), C.cast(s, C.c_void_p), _ptr(tmp), _ptr(out),
                                          _ptr(dev["tc_coef"]) if use_tc else None, p.tc_kw if use_tc else 0,
                                          p.tc_limbs if use_tc else 0, _ptr(dev["tc_kb0"]) if use_tc else None,
                                          _lib.stream_ptr()), "fb_clip_preprocess")
    return out


GEMM_BIAS_BF16, GEMM_BIAS_GELU_BF16, GEMM_BIAS_RESIDUAL_F32, GEMM_F32 = 0, 1, 2, 3


def gemm_bf16(a, b, mode: int = GEMM_F32, bias=None, residual=None, out=None):
    """C[M,N] = A[M,K] @ B[N,K]^T with the tcgen05 kernel.  a, b: CUDA bf16, row-major (last dim
    contiguous).  Returns bf16 (modes 0/1) or float32 (modes 2/3)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    if a.dtype != b.dtype or a.dtype not in (torch.bfloat16, torch.float16):
        raise TypeError("gemm_bf16 takes two bf16 or two fp16 operands")
    f16 = a.dtype == torch.float16
    if a.stride(-1) != 1 or b.stride(-1) != 1:
        raise ValueError("operands must be K-contiguous")
    m, k = a.shape
    n, kb = b.shape
    if k != kb:
        raise ValueError("K mismatch")
    odt = a.dtype if mode in (GEMM_BIAS_BF16, GEMM_BIAS_GELU_BF16) else torch.float32
    if out is None:
        out = torch.empty((m, n), dtype=odt, device=a.device)
    with torch.cuda.device(a.device):
        _lib.check(lib.fb_gemm_bf16(_ptr(a), a.stride(0), _ptr(b), b.stride(0), m, n, k, int(mode) | (16 if f16 else 0),
                                    _ptr(bias) if bias is not None else None, _ptr(out), out.stride(0),
                                    _ptr(residual) if residual is not None else None,
                                    residual.stride(0) if residual is not None else 0, _lib.stream_ptr()), "fb_gemm_bf16")
    return out


def vit_layernorm(x, gamma, beta, out_bf16=True, class_emb=None, pos_emb=None, rows=None):
    """out_bf16: False / 0 -> fp32, True / 1 -> bf16, 2 -> fp16."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    rows = int(rows if rows is not None else x.shape[0])
    out_bf16 = int(out_bf16)
    odt = {0: torch.float32, 1: torch.bfloat16, 2: torch.float16}[out_bf16]
    out = torch.empty((rows, 1024), dtype=odt, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.fb_vit_layernorm(_ptr(x), x.stride(0), rows, _ptr(gamma), _ptr(beta),
                                        _ptr(class_emb) if class_emb is not None else None,
                                        _ptr(pos_emb) if pos_emb is not None else None, _ptr(out), 1024,
                                        out_bf16, _lib.stream_ptr()), "fb_vit_layernorm")
    return out


def vit_attention(qkv, batch: int):
    """qkv: CUDA bf16 / fp16 [batch*257, 3072] -> same dtype [batch*257, 1024] (tcgen05 kernel)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    out = torch.empty((batch * 257, 1024), dtype=qkv.dtype, device=qkv.device)
    fn = lib.fb_vit_attention_f16 if qkv.dtype == torch.float16 else lib.fb_vit_attention
    with torch.cuda.device(qkv.device):
        _lib.check(fn(_ptr(qkv), batch, _ptr(out), _lib.stream_ptr()), "fb_vit_attention")
    return out


def embedding_heads(vectors, head=None, tag_embeddings=None):
    """Heads on stored embeddings (fb_embedding_heads): vectors CUDA float32 [n,768]; head = (w1 [256,768], b1 [256],
    w2 [256], b2 [1]) CUDA float32 tensors or None; tag_embeddings CUDA float32 [t,768] or None.
    Returns (raw [n] or None, sims [n,t] or None) as CUDA tensors."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    v = vectors.contiguous()
    n = int(v.shape[0])
    raw = torch.empty((n,), dtype=torch.float32, device=v.device) if head is not None else None
    nt = int(tag_embeddings.shape[0]) if tag_embeddings is not None else 0
    sims = torch.empty((n, nt), dtype=torch.float32, device=v.device) if nt else None
    w1, b1, w2, b2 = head if head is not None else (None, None, None, None)
    with torch.cuda.device(v.device):
        _lib.check(lib.fb_embedding_heads(_ptr(v), n, _ptr(w1) if head is not None else None, _ptr(b1) if head is not None else None,
                                          _ptr(w2) if head is not None else None, _ptr(b2) if head is not None else None,
                                          _ptr(tag_embeddings) if nt else None, nt, _ptr(raw) if raw is not None else None,
                                          _ptr(sims) if nt else None, _lib.stream_ptr()), "fb_embedding_heads")
    return raw, sims


def balanced_row_blocks(n: int, parts: int):
    """Row boundaries that give every part the same number of upper-triangle (i<j) pairs."""
    bounds = [int(round(n * (1.0 - (1.0 - k / parts) ** 0.5))) for k in range(parts + 1)]
    bounds[0], bounds[-1] = 0, n
    return bounds


def cosine_pairs(emb_f32, tau: float, part: int = 0, nparts: int = 1, band: float = 0.01, cap: int | None = None):
    """All (i<j) pairs of this part's row block with float32 <e_i,e_j> >= tau.
    emb_f32: CUDA float32 [n,d] (L2-normalised, d % 64 == 0).  Returns (pairs int32 [m,2], sims float32 [m])."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    e = emb_f32.contiguous()
    n, d = e.shape
    bounds = balanced_row_blocks(n, nparts)
    r0, r1 = bounds[part], bounds[part + 1]
    with torch.cuda.device(e.device):
        eb = torch.empty((n, d), dtype=torch.bfloat16, device=e.device)
        _lib.check(lib.fb_f32_to_bf16(_ptr(e), _ptr(eb), n * d, _lib.stream_ptr()), "fb_f32_to_bf16")
        cap = int(cap if cap is not None else max(1 << 20, 8 * n))      # 1 M candidates (12 MB): small, dense sets need no second pass
        counts = torch.zeros(2, dtype=torch.int64, device=e.device)
        while True:
            cand = torch.empty((cap, 2), dtype=torch.int32, device=e.device)
            cand_s = torch.empty((cap,), dtype=torch.float32, device=e.device)
            pairs = torch.empty((cap, 2), dtype=torch.int32, device=e.device)
            sims = torch.empty((cap,), dtype=torch.float32, device=e.device)
            _lib.check(lib.fb_cosine_pairs(_ptr(e), _ptr(eb), n, d, float(tau), float(band), r0, r1 - r0, _ptr(cand),
                                           _ptr(cand_s), cap, C.c_void_p(counts.data_ptr()), _ptr(pairs), _ptr(sims), cap,
                                           C.c_void_p(counts.data_ptr() + 8), _lib.stream_ptr()), "fb_cosine_pairs")
            nc, m = (int(x) for x in counts.tolist())
            if nc <= cap and m <= cap:
                return pairs[:m], sims[:m]
            cap = _grown_cap(max(nc, m), 'cosine_pairs')


def to_bf16(emb_f32):
    """float32 CUDA tensor -> bf16 copy with the library's conversion kernel (round to nearest even)."""
    torch = _lib.require_cuda()
    e = emb_f32.contiguous()
    out = torch.empty(e.shape, dtype=torch.bfloat16, device=e.device)
    with torch.cuda.device(e.device):
        _lib.check(_lib.load().fb_f32_to_bf16(_ptr(e), _ptr(out), e.numel(), _lib.stream_ptr()), "fb_f32_to_bf16")
    return out


def cosine_blocks(blocks, get_emb_f32, dim: int, tau: float, band: float = 0.01, cap: int | None = None, before_block=None):
    """Cosine pairs of a list of shard-against-shard blocks (the multi-GPU scan).  blocks: [(a_bf16 [m,dim], a_offset, b_bf16
    [n,dim], b_offset, triangle)] with GLOBAL row offsets; `before_block(k)` is called before block k is launched (the sharded
    flow waits there for the all-gather the block needs); `get_emb_f32()` returns the gathered float32 matrix for the recheck.
    Returns (pairs int32 [p,2] with i < j, sims float32 [p]) — the same pairs the single-matrix scan finds for these blocks."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    dev = blocks[0][0].device
    rows = sum(int(b[0].shape[0]) for b in blocks)
    e32 = None
    with torch.cuda.device(dev):
        cap = int(cap if cap is not None else max(1 << 20, 8 * rows))   # 1 M candidates (12 MB): small, dense sets need no second pass
        counts = torch.zeros(2, dtype=torch.int64, device=dev)
        while True:
            counts.zero_()
            cand = torch.empty((cap, 2), dtype=torch.int32, device=dev)
            cand_s = torch.empty((cap,), dtype=torch.float32, device=dev)
            for k, (a, a_off, b, b_off, tri) in enumerate(blocks):
                if before_block is not None:
                    before_block(k)
                if a.shape[0] == 0 or b.shape[0] == 0:
                    continue
                _lib.check(lib.fb_cosine_block(_ptr(a), int(a.shape[0]), int(a_off), _ptr(b), int(b.shape[0]), int(b_off), int(dim),
                                               float(tau) - float(band), int(bool(tri)), _ptr(cand), _ptr(cand_s), cap,
                                               C.c_void_p(counts.data_ptr()), _lib.stream_ptr()), "fb_cosine_block")
            if e32 is None:
                e32 = get_emb_f32().contiguous()
            pairs = torch.empty((cap, 2), dtype=torch.int32, device=dev)
            sims = torch.empty((cap,), dtype=torch.float32, device=dev)
            _lib.check(lib.fb_cosine_recheck(_ptr(e32), int(dim), _ptr(cand), C.c_void_p(counts.data_ptr()), cap, float(tau), _ptr(pairs),
                                             _ptr(sims), cap, C.c_void_p(counts.data_ptr() + 8), _lib.stream_ptr()), "fb_cosine_recheck")
            nc, m = (int(x) for x in counts.tolist())
            if nc <= cap and m <= cap:
                pairs = pairs[:m]
                lo = torch.minimum(pairs[:, 0], pairs[:, 1])
                hi = torch.maximum(pairs[:, 0], pairs[:, 1])
                return torch.stack([lo, hi], dim=1), sims[:m]
            cap = _grown_cap(max(nc, m), 'cosine_blocks')
            before_block = None          # everything has arrived by now


def orient(images, exif_orientation: int = 1, swap_rb: bool = False):
    """`ImageOps.exif_transpose` of a same-shaped batch for the given EXIF orientation code (1..8), then an
    optional channel swap (`cv2.cvtColor(RGB2BGR)`): the pixel work of utils/image_loading.py:101-106.
    images: uint8 [n,H,W,3] or [H,W,3].  Returns a new CUDA uint8 tensor ([n,W,H,3] for orientations 5..8)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    t = to_device_u8(images)
    n, h, w, _ = t.shape
    code = int(exif_orientation)
    if not 1 <= code <= 8:
        raise ValueError(f"EXIF orientation {exif_orientation} outside 1..8")
    oh, ow = (w, h) if code >= 5 else (h, w)
    with torch.cuda.device(t.device):
        out = torch.empty((n, oh, ow, 3), dtype=torch.uint8, device=t.device)
        _lib.check(lib.fb_orient(_ptr(t), n, h, w, h * w * 3, code, int(bool(swap_rb)), _ptr(out), oh * ow * 3,
                                 _lib.stream_ptr()), "fb_orient")
    return out


_THUMB_PLANS: dict = {}


def thumbnail_reduces_by_4(h: int, w: int, size: int = 640) -> bool:
    """True when Pillow's thumbnail of an h x w frame starts with the (4, 4) box reduction `tech_stats_raw(box_out=)` emits."""
    from .utils import thumbnail as th
    p = th.plan(h, w, size)
    return p is not None and p.fx == 4 and p.fy == 4


def thumbnails(images, size: int = 640, rgb_order: bool = False, to_rgb: bool = True, reduced=None):
    """Pillow `Image.thumbnail((size, size), LANCZOS)` of a same-shaped batch, bit-exact (the pixel work of
    utils/image_transforms.py:32-50).  images: uint8 [n,H,W,3] (BGR unless rgb_order).  Returns a CUDA uint8
    tensor [n,h,w,3] in RGB order when to_rgb (what PIL would hold), else in the input's channel order.
    reduced: the (4, 4) box reduction of the frames from `tech_stats_raw(box_out=)` when `thumbnail_reduces_by_4`
    (the frames are then not read at all)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    from .utils import thumbnail as th
    t = to_device_u8(images)
    n, h, w, _ = t.shape
    swap = bool(to_rgb) and not rgb_order
    p = th.plan(h, w, size)
    if reduced is not None and not (p is not None and p.fx == 4 and p.fy == 4 and tuple(reduced.shape) == (n, p.red_h, p.red_w, 3)):
        raise ValueError("reduced does not match the thumbnail plan of these frames")
    if p is None:                                   # Pillow leaves images that already fit unchanged
        return t.flip(-1).contiguous() if swap else t.clone()
    key = (h, w, size, str(t.device))
    if key not in _THUMB_PLANS:
        mult = np.array([th.reduce_multiplier(max(1, a * b)) for a, b in
                         ((p.fx, p.fy), (w % p.fx or p.fx, p.fy), (p.fx, h % p.fy or p.fy), (w % p.fx or p.fx, h % p.fy or p.fy))],
                        dtype=np.uint32)
        _THUMB_PLANS[key] = (mult,) + tuple(torch.from_numpy(np.ascontiguousarray(a)).to(t.device)
                                            for a in (p.hbounds, p.hcoef, p.vbounds, p.vcoef))
    mult, hb, hc, vb, vc = _THUMB_PLANS[key]
    with torch.cuda.device(t.device):
        tmp = torch.empty((n, p.red_h, p.out_w, 3), dtype=torch.uint8, device=t.device)
        out = torch.empty((n, p.out_h, p.out_w, 3), dtype=torch.uint8, device=t.device)
        if reduced is not None:
            _lib.check(lib.fb_thumbnail_from_reduced(_ptr(reduced), n, h, w, p.fx, p.fy, p.red_h, p.red_w, _ptr(hb), _ptr(hc), p.hk,
                                                     _ptr(vb), _ptr(vc), p.vk, p.out_h, p.out_w, int(swap), _ptr(tmp), _ptr(out),
                                                     _lib.stream_ptr()), "fb_thumbnail_from_reduced")
            return out
        reduced = torch.empty((n, p.red_h, p.red_w, 3), dtype=torch.uint8, device=t.device) if (p.fx > 1 or p.fy > 1) else None
        _lib.check(lib.fb_thumbnail(_ptr(t), n, h, w, h * w * 3, p.fx, p.fy, p.red_h, p.red_w, mult.ctypes.data,
                                    _ptr(hb), _ptr(hc), p.hk, _ptr(vb), _ptr(vc), p.vk, p.out_h, p.out_w, int(swap),
                                    _ptr(reduced) if reduced is not None else None, _ptr(tmp), _ptr(out), _lib.stream_ptr()),
                   "fb_thumbnail")
    return out


_JPEG_ENC_DEV: dict = {}


def jpeg_encode(images_rgb, quality: int = 80, as_device: bool = False):
    """JPEG streams of a same-shaped batch of RGB images (CUDA uint8 [n,H,W,3] or numpy), byte-exact with
    `PIL.Image.fromarray(img).save(buf, format='JPEG', quality=quality)` — the encoder call of utils/image_transforms.py:47.
    Returns a list of `bytes`, or with as_device the (streams uint8 [n, stride], lengths int32 [n]) CUDA tensors."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    from .utils import jpeg as fj
    t = to_device_u8(images_rgb)
    n, h, w, _ = t.shape
    header, packed = fj.encoder_tables(h, w, quality)
    key = (h, w, int(quality), str(t.device))
    if key not in _JPEG_ENC_DEV:
        _JPEG_ENC_DEV[key] = (torch.from_numpy(np.frombuffer(header, np.uint8).copy()).to(t.device),
                              torch.from_numpy(np.frombuffer(packed, np.uint8).copy()).to(t.device))
    d_header, d_tables = _JPEG_ENC_DEV[key]
    with torch.cuda.device(t.device):
        ws_bytes = int(lib.fb_jpeg_encode_workspace_bytes(n, h, w))
        stride = int(lib.fb_jpeg_encode_out_stride(h, w, len(header)))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=t.device)
        out = torch.empty((n, stride), dtype=torch.uint8, device=t.device)
        lengths = torch.empty(n, dtype=torch.int32, device=t.device)
        _lib.check(lib.fb_jpeg_encode(_ptr(t), n, h, w, h * w * 3, _ptr(d_tables), _ptr(d_header), len(header), _ptr(ws), ws_bytes,
                                      _ptr(out), stride, _ptr(lengths), _lib.stream_ptr()), "fb_jpeg_encode")
    if as_device:
        return out, lengths
    lens = lengths.cpu().numpy()
    host = out[:, :int(lens.max())].cpu().numpy()
    return [host[i, :lens[i]].tobytes() for i in range(n)]


_PHASH_PLANS: dict = {}


def phash_uses_luma_plane(h: int, w: int) -> bool:
    """True when phash() takes the tensor-core route and can consume a luma plane from tech_stats_raw."""
    from .utils import resample as rs
    return w % 16 == 0 and rs.phash_tc_tables(h, w)[0] is not None


def phash(images, rgb_order: bool = False, debug: bool = False, tensor_cores: bool = True, device_only: bool = False,
          luma=None):
    """64-bit perceptual hashes (imagehash.phash) of a same-shaped batch.  Returns a uint64 numpy array
    (and, with debug=True, the 32x32 uint8 luma thumbnails and the 8x8 float64 DCT blocks); with
    device_only=True the CUDA int64 tensor is returned without synchronising."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    from .utils import resample as rs
    t = to_device_u8(images)
    n, h, w, _ = t.shape
    key = (h, w, str(t.device))
    if key not in _PHASH_PLANS:
        hb, hc, hk, vb, vc, vk = rs.phash_plan(h, w)
        tcc, tkb0, tkw, tlimbs = rs.phash_tc_tables(h, w)
        tc_dev = (torch.from_numpy(tcc).to(t.device), torch.from_numpy(tkb0).to(t.device), tkw, tlimbs) if tcc is not None else None
        _PHASH_PLANS[key] = tuple(torch.from_numpy(a).to(t.device) for a in (hb, hc, vb, vc)) + (hk, vk, tc_dev)
    hb, hc, vb, vc, hk, vk, tc_dev = _PHASH_PLANS[key]
    use_tc = bool(tensor_cores) and tc_dev is not None and w % 16 == 0
    luma_ready = luma is not None
    if luma_ready and not use_tc:
        raise ValueError("a precomputed luma plane needs the tensor-core route (width % 16 == 0)")
    if use_tc and luma is None:
        luma = torch.empty((n, h, w), dtype=torch.uint8, device=t.device)
    tmp = torch.empty((n, h, 32), dtype=torch.uint8, device=t.device)
    hashes = torch.empty((n,), dtype=torch.int64, device=t.device)
    small = torch.empty((n, 32, 32), dtype=torch.uint8, device=t.device) if debug else None
    dct = torch.empty((n, 64), dtype=torch.float64, device=t.device) if debug else None
    with torch.cuda.device(t.device):
        _lib.check(lib.fb_phash(_ptr(t), n, h, w, h * w * 3, int(bool(rgb_order)), _ptr(hb), _ptr(hc), hk, _ptr(vb), _ptr(vc), vk,
                                _ptr(tmp), _ptr(hashes), _ptr(small) if debug else None, _ptr(dct) if debug else None,
                                _ptr(luma) if use_tc else None, int(luma_ready), _ptr(tc_dev[0]) if use_tc else None,
                                tc_dev[2] if use_tc else 0, tc_dev[3] if use_tc else 0, _ptr(tc_dev[1]) if use_tc else None,
                                _lib.stream_ptr()), "fb_phash")
    if device_only:
        return hashes
    out = hashes.cpu().numpy().view(np.uint64)
    if debug:
        return out, small.cpu().numpy(), dct.cpu().numpy().reshape(n, 8, 8)
    return out


def phash_hex(images, rgb_order: bool = False):
    """str(imagehash.phash(img)) for each frame: 16 lowercase hex digits."""
    return ["%016x" % int(v) for v in phash(images, rgb_order=rgb_order)]


# ---- JPEG decoding (csrc/jpeg_decode.cu) -------------------------------------------------------------------------------
def jpeg_decode_device(dev_bytes, slot_bytes: int, infos, bgr: bool = True, out=None):
    """Decode n same-geometry JPEG streams whose file bytes already sit in `dev_bytes` (CUDA uint8, stream i at offset
    i * slot_bytes).  infos: the `utils.jpeg.parse` results.  Returns (frames CUDA uint8 [n,H,W,3], status CUDA int32 [n]);
    nothing is synchronised.  EXIF orientation is NOT applied (ops.orient does that)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    from .utils import jpeg as fj
    n = len(infos)
    i0 = infos[0]
    key = i0.geometry_key()
    if any(i.geometry_key() != key for i in infos[1:]):
        raise ValueError("jpeg_decode_device takes streams of one geometry (size, components, sampling, restart interval)")
    dev = dev_bytes.device
    slots, blobs = {}, []
    table_slot = np.empty(n, np.int32)
    for k, inf in enumerate(infos):
        blob = inf.packed_tables
        s = slots.get(id(blob))
        if s is None:
            s = slots[id(blob)] = len(blobs)
            blobs.append(blob)
        table_slot[k] = s
    scan_off = np.array([k * slot_bytes + inf.scan_offset for k, inf in enumerate(infos)], np.int64)
    scan_len = np.array([inf.scan_end - inf.scan_offset for inf in infos], np.int64)
    if int((scan_off + scan_len).max()) > dev_bytes.numel() or int(scan_len.min()) < 0:
        raise ValueError("jpeg_decode_device: a stream does not fit its slot")
    meta = torch.from_numpy(np.concatenate([scan_off, scan_len])).to(dev, non_blocking=True)
    tslot = torch.from_numpy(table_slot).to(dev, non_blocking=True)
    tables = torch.from_numpy(np.frombuffer(b"".join(blobs), np.uint8).copy()).to(dev, non_blocking=True)
    hmax, vmax = i0.hs[0], i0.vs[0]
    max_scan = int(scan_len.max())
    ws_bytes = int(lib.fb_jpeg_workspace_bytes(n, i0.width, i0.height, i0.ncomp, hmax, vmax, i0.restart_interval, max_scan))
    arr3 = lambda v, fill: (C.c_int32 * 3)(*((list(v) + [fill] * 3)[:3]))
    with torch.cuda.device(dev):
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        frames = out if out is not None else torch.empty((n, i0.height, i0.width, 3), dtype=torch.uint8, device=dev)
        status = torch.empty((n,), dtype=torch.int32, device=dev)
        _lib.check(lib.fb_jpeg_decode(_ptr(dev_bytes), C.c_void_p(meta.data_ptr()), C.c_void_p(meta.data_ptr() + 8 * n), _ptr(tslot),
                                      _ptr(tables), n, i0.width, i0.height, i0.ncomp, C.cast(arr3(i0.hs, 1), C.c_void_p),
                                      C.cast(arr3(i0.vs, 1), C.c_void_p), C.cast(arr3(i0.tq, 0), C.c_void_p),
                                      C.cast(arr3(i0.td, 0), C.c_void_p), C.cast(arr3(i0.ta, 0), C.c_void_p), i0.restart_interval,
                                      max_scan, int(bool(bgr)), _ptr(ws), ws_bytes, _ptr(frames), i0.height * i0.width * 3,
                                      _ptr(status), _lib.stream_ptr()), "fb_jpeg_decode")
    return frames, status


def jpeg_decode(streams, bgr: bool = True, apply_orientation: bool = True):
    """Decode JPEG file contents on the GPU: the pixel work of `load_image_from_path` (utils/image_loading.py:90-106) —
    byte-exact with `np.asarray(ImageOps.exif_transpose(Image.open(f)).convert('RGB'))` (reversed to BGR when `bgr`).
    streams: list of bytes / 1-D uint8 arrays of ONE geometry.  Returns a CUDA uint8 tensor [n,H,W,3] ([n,W,H,3] after
    a transposing EXIF orientation).  Raises utils.jpeg.UnsupportedJpeg for streams the device decoder does not take
    and RuntimeError for corrupt entropy data."""
    torch = _lib.require_cuda()
    from .utils import jpeg as fj
    infos = [fj.parse(s) for s in streams]
    slot = (max(len(s) for s in streams) + 255) & ~255
    dev = torch.device("cuda", torch.cuda.current_device())
    buf = torch.empty(len(streams) * slot + 256, dtype=torch.uint8, device=dev)      # the bit reader reads up to 15 bytes past a stream
    for k, s in enumerate(streams):
        a = np.frombuffer(s, np.uint8) if isinstance(s, (bytes, bytearray, memoryview)) else np.ascontiguousarray(s, dtype=np.uint8).reshape(-1)
        buf[k * slot:k * slot + a.size].copy_(torch.from_numpy(a.copy() if not a.flags.writeable else a), non_blocking=True)
    frames, status = jpeg_decode_device(buf, slot, infos, bgr=bgr)
    st = status.cpu().numpy()
    if st.any():
        bad = int(np.flatnonzero(st)[0])
        raise RuntimeError(f"JPEG stream {bad}: " + ("restart markers do not match the DRI header" if st[bad] & 1 else
                                                     "self-synchronisation did not settle" if st[bad] & 4 else "invalid Huffman data"))
    if apply_orientation:
        codes = {i.orientation for i in infos}
        if codes != {1}:
            if len(codes) != 1:
                raise ValueError("jpeg_decode: streams of one call must share their EXIF orientation")
            frames = orient(frames, codes.pop())
    return frames
