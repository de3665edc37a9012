"""Torch-tensor front end of the vdb200 C ABI (include/vdb200.h).

torch is used here for device memory, streams and allocation only; every arithmetic op on the hot
path is a kernel of libvdb200.so.  All functions enqueue on torch's current CUDA stream and are
CUDA-graph capturable (no host syncs, scratch comes from the caller or torch's caching allocator).
"""
import ctypes
import math
import os

import torch

from ._lib import lib, check

ACT_NONE, ACT_SILU, ACT_GELU, ACT_QUICK_GELU, ACT_GEGLU, ACT_GELU_TANH, ACT_TANH = 0, 1, 2, 3, 4, 5, 6
BF16 = torch.bfloat16


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _need(t, dtype, name, rows_ok=False):
    if t is None:
        return
    if not t.is_cuda:
        raise ValueError(f"{name}: vdb200 kernels need CUDA tensors (no CPU fallback)")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    if rows_ok and t.dim() == 2 and t.stride(1) == 1:
        return  # row-strided 2-D view: the kernels take a leading dimension
    if not t.is_contiguous():
        raise ValueError(f"{name}: must be contiguous")


_workspace = {}
WORKSPACE_BYTES = 160 << 20   # covers 16-way split-K of any MN grid that fits in half the SMs (74 tiles x 128 x 256 fp32)


def _scratch_key(device):
    """(device, stream) key of the split-K workspace / GroupNorm scratch.  The C ABI promises reuse of a scratch buffer on ONE
    stream only (the GroupNorm arrival counters and the split-K partials are not re-entrant), so every eager stream gets its
    own buffers: two threads sampling on two streams of one GPU no longer share counters.  Launches issued while a CUDA graph
    is being captured (torch captures on a side stream) use the buffers of the device's FIRST stream — the one the eager
    warm-up step ran on — so the addresses baked into the graph are the ones that were sized and zeroed before capture.
    Graphs captured from different streams therefore still share one scratch set and must not be replayed concurrently."""
    dev = device.index if device.index is not None else torch.cuda.current_device()
    sid = torch.cuda.current_stream(dev).cuda_stream
    owner = _scratch_owner.setdefault(dev, sid)
    if torch.cuda.is_current_stream_capturing():
        sid = owner
    return (dev, sid)


_scratch_owner = {}


def workspace(device):
    """Fixed-size fp32 split-K scratch per (device, stream). Never reallocated: its address is baked into captured CUDA graphs."""
    key = _scratch_key(device)
    w = _workspace.get(key)
    if w is None:
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("split-K workspace must exist before CUDA-graph capture (run one eager step first)")
        w = torch.empty(WORKSPACE_BYTES // 4, dtype=torch.float32, device=device)
        _workspace[key] = w
    return w


# ------------------------------------------------------------------------------------------------
# optional per-family device timing (bench.py roofline leg): CUDA events on the launching stream
# ------------------------------------------------------------------------------------------------
_PROFILE = None


class _Span(object):
    __slots__ = ("name", "flops", "nbytes", "e0", "e1")

    def __init__(self, name, flops, nbytes):
        self.name, self.flops, self.nbytes = name, flops, nbytes

    def __enter__(self):
        if _PROFILE is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if _PROFILE is not None:
            self.e1.record()
            _PROFILE.append(self)
        return False


def profile_start():
    global _PROFILE
    _PROFILE = []


def profile_stop():
    """-> {family: {"ms": total, "launches": n, "flops": total, "bytes": total}}"""
    global _PROFILE
    spans, _PROFILE = _PROFILE, None
    torch.cuda.synchronize()
    out = {}
    for sp in spans or []:
        d = out.setdefault(sp.name, {"ms": 0.0, "launches": 0, "flops": 0.0, "bytes": 0.0})
        d["ms"] += sp.e0.elapsed_time(sp.e1)
        d["launches"] += 1
        d["flops"] += sp.flops
        d["bytes"] += sp.nbytes
    return out


# ------------------------------------------------------------------------------------------------
# optional recording of the tensor-core GEMM / conv launches (bench.py: replay of exactly these launches inside a CUDA
# graph, so the roofline leg can time the kernel without the host launch path).  Each record keeps its tensors alive.
# ------------------------------------------------------------------------------------------------
_RECORD = None


def record_start():
    global _RECORD
    _RECORD = []


def record_stop():
    """-> [(C function, arguments without the stream, tensors kept alive, algorithmic FLOPs)]"""
    global _RECORD
    rec, _RECORD = _RECORD, None
    return rec or []


def replay(records):
    """Re-issue recorded launches on the current stream (capturable)."""
    for fn, cargs, _keep, _flops in records:
        check(fn(*cargs, _stream()), "replay")


_gn_scratch_buf = {}


def _gn_scratch(device, nfloats):
    """Persistent zero-initialised GroupNorm scratch per (device, stream) (the kernels restore its counters to zero)."""
    key = _scratch_key(device)
    buf = _gn_scratch_buf.get(key)
    if buf is None or buf.numel() < nfloats:
        if buf is not None and torch.cuda.is_current_stream_capturing():
            raise RuntimeError("GroupNorm scratch must be sized before CUDA-graph capture (run one eager step first)")
        buf = torch.zeros(max(int(nfloats), 1 << 20), dtype=torch.float32, device=device)
        _gn_scratch_buf[key] = buf
    return buf


def launch_count():
    return int(lib.vdb_launch_count())


def reset_launch_count():
    lib.vdb_reset_launch_count()


# ------------------------------------------------------------------------------------------------
def ddim_cfg_step(e_uncond, e_cond, x, coef, scale, x_prev=None, pred_x0=None, noise=None,
                  temperature=1.0, step_idx=None, x_prev_dup=None):
    """K4 (ddim.py:144-171). e_*/x/noise fp32 same shape; coef fp32 [.,4] device tensor."""
    for n, t in (("e_uncond", e_uncond), ("e_cond", e_cond), ("x", x), ("noise", noise), ("coef", coef)):
        _need(t, torch.float32, n)
    if x_prev is None:
        x_prev = torch.empty_like(x)
    if step_idx is not None:
        _need(step_idx, torch.int32, "step_idx")
    check(lib.vdb_ddim_cfg_step(_ptr(e_uncond), _ptr(e_cond), _ptr(x), _ptr(noise), _ptr(coef), _ptr(step_idx),
                                float(scale), float(temperature), _ptr(x_prev), _ptr(x_prev_dup), _ptr(pred_x0), x.numel(),
                                _stream()),
          "ddim_cfg_step")
    return x_prev, pred_x0


def axpby(x, z, a, b, out=None):
    _need(x, torch.float32, "x"); _need(z, torch.float32, "z")
    if out is None:
        out = torch.empty_like(x)
    check(lib.vdb_axpby_f32(_ptr(x), _ptr(z), float(a), float(b), _ptr(out), x.numel(), _stream()), "axpby")
    return out


def lincomb4(xs, cs, out=None):
    """sum_i cs[i] * xs[i] for 1..4 fp32 tensors of one shape."""
    assert 1 <= len(xs) <= 4 and len(xs) == len(cs)
    for t in xs:
        _need(t, torch.float32, "x")
    if out is None:
        out = torch.empty_like(xs[0])
    ptrs = [_ptr(t) for t in xs] + [0] * (4 - len(xs))
    coef = [float(c) for c in cs] + [0.0] * (4 - len(cs))
    check(lib.vdb_lincomb4_f32(ptrs[0], ptrs[1], ptrs[2], ptrs[3], coef[0], coef[1], coef[2], coef[3], _ptr(out),
                               xs[0].numel(), _stream()), "lincomb4")
    return out


def add_int(t, delta):
    _need(t, torch.int32, "counter")
    check(lib.vdb_add_int(_ptr(t), int(delta), _stream()), "add_int")


def _skinny_rows():
    """largest small operand (rows) that ops.gemm sends to vdb_gemm_skinny_bf16 instead of the tensor-core kernel
    (VDB_SKINNY=<rows>; default 0 = never: on the full-size 0-D diffuser the CUDA-core kernel streams weights at 1.1-1.3 TB/s
    against 2.7-3.5 TB/s for split-K tensor-core tiles — i2t step 4.43 ms (<= 16 rows) / 7.3 ms (<= 64) vs 3.38 ms,
    profiles/r02_visit_x_skinny_gemm.log)"""
    return int(os.environ.get("VDB_SKINNY", "0"))


def gemm(a, w, bias=None, resid=None, out=None, act=ACT_NONE, a2=None, out_dtype=BF16, alpha=1.0,
         bias_bstride=0, rows_per_batch=1, bn=0, ksplit=0):
    """out[M,N'] = act(alpha*[a|a2] @ w^T + bias) + resid ; a [M,K] bf16, w [N,K(+K2)] bf16."""
    _need(a, BF16, "a", True); _need(w, BF16, "w", True); _need(a2, BF16, "a2", True); _need(bias, torch.float32, "bias")
    _need(resid, BF16, "resid", True)
    M, K = a.shape
    N = w.shape[0]
    K2 = a2.shape[1] if a2 is not None else 0
    assert w.shape[1] == K + K2, (w.shape, K, K2)
    n_out = N // 2 if act == ACT_GEGLU else N
    if out is None:
        out = torch.empty((M, n_out), dtype=out_dtype, device=a.device)
    _need(out, out_dtype, "out", True)
    smax = _skinny_rows()
    if act == ACT_NONE and alpha == 1.0 and out_dtype == BF16 and bn == 0 and ksplit == 0 and smax > 0:
        # a small operand of <= 64 rows: weight-streaming CUDA-core kernel instead of the tensor-core latency chain
        if M <= smax and (bias_bstride == 0 or rows_per_batch == 1) and lib.vdb_gemm_skinny_fits(M, K + K2):
            check(lib.vdb_gemm_skinny_bf16(_ptr(a), M, K, a.stride(0), _ptr(a2), K2, a2.stride(0) if a2 is not None else 0,
                                           _ptr(w), N, w.stride(0), _ptr(bias), int(bias_bstride), _ptr(resid),
                                           resid.stride(0) if resid is not None else 0, _ptr(out), out.stride(0), 0, _stream()),
                  "gemm_skinny_bf16")
            return out
        if N <= smax and M > N and a2 is None and bias is None and resid is None and lib.vdb_gemm_skinny_fits(N, K):
            check(lib.vdb_gemm_skinny_bf16(_ptr(w), N, K, w.stride(0), None, 0, 0, _ptr(a), M, a.stride(0), None, 0, None, 0,
                                           _ptr(out), out.stride(0), 1, _stream()), "gemm_skinny_bf16")
            return out
    ws, ws_bytes = None, 0
    if ksplit != 1 and M <= 8192:   # split-K only ever triggers for small MN grids
        ws, ws_bytes = workspace(a.device), WORKSPACE_BYTES
    cargs = (_ptr(a), M, K, a.stride(0), _ptr(a2), K2, a2.stride(0) if a2 is not None else 0,
             _ptr(w), N, w.stride(0), _ptr(bias), int(bias_bstride), int(rows_per_batch),
             _ptr(resid), resid.stride(0) if resid is not None else 0, _ptr(out), out.stride(0),
             1 if out_dtype == torch.float32 else 0, int(act), float(alpha), int(bn), int(ksplit),
             _ptr(ws), ws_bytes)
    with _Span("gemm", 2.0 * M * N * (K + K2), 2.0 * (M * (K + K2) + N * (K + K2) + M * n_out)):
        check(lib.vdb_gemm_bf16(*cargs, _stream()), "gemm_bf16")
    if _RECORD is not None:
        _RECORD.append((lib.vdb_gemm_bf16, cargs, (a, a2, w, bias, resid, out, ws), 2.0 * M * N * (K + K2)))
    return out


class LnFold(object):
    """What a GEMM needs to consume a LayerNorm it never sees (vdb_gemm_ln_bf16): the producer's partial sums `stats`
    [>= parts, rows, 2] fp32 (`parts` of them valid), the LayerNorm's width and epsilon; the weights' column sums ride with the
    packed weights."""

    def __init__(self, stats, parts, dim, eps):
        self.stats, self.parts, self.dim, self.eps = stats, int(parts), int(dim), float(eps)


def ln_stats_buffer(rows, width, device):
    """statistics table a producer GEMM with N = width columns fills for its `rows` output rows (worst case: 64-column tiles)"""
    assert width % 32 == 0
    return torch.empty((2 * ((width + 63) // 64), rows, 2), dtype=torch.float32, device=device)


def gemm_ln(a, w, bias=None, resid=None, out=None, act=ACT_NONE, ln=None, colsum=None, on_cols=False, rowbias=None,
            stats_out=None, bn=0):
    """vdb_gemm_ln_bf16: consumer (ln = LnFold, colsum) or producer (stats_out; returns (out, parts)) of folded-LayerNorm
    statistics."""
    _need(a, BF16, "a", True); _need(w, BF16, "w", True); _need(bias, torch.float32, "bias"); _need(resid, BF16, "resid", True)
    _need(colsum, torch.float32, "colsum"); _need(rowbias, torch.float32, "rowbias"); _need(stats_out, torch.float32, "stats_out")
    M, K = a.shape
    N = w.shape[0]
    assert w.shape[1] == K, (w.shape, K)
    n_out = N // 2 if act == ACT_GEGLU else N
    if out is None:
        out = torch.empty((M, n_out), dtype=BF16, device=a.device)
    _need(out, BF16, "out", True)
    st = None
    if ln is not None:
        st = ln.stats
        _need(st, torch.float32, "ln.stats")
        assert st.dim() == 3 and st.shape[0] >= ln.parts and st.shape[2] == 2, (tuple(st.shape), ln.parts)
    parts = ctypes.c_int(0)
    if stats_out is not None:
        assert stats_out.dim() == 3 and stats_out.shape[0] >= 2 * ((N + 63) // 64) and stats_out.shape[1] == M and stats_out.shape[2] == 2, \
            (tuple(stats_out.shape), N, M)
    cargs = (_ptr(a), M, K, a.stride(0), _ptr(w), N, w.stride(0), _ptr(bias), _ptr(resid),
             resid.stride(0) if resid is not None else 0, _ptr(out), out.stride(0), int(act),
             _ptr(st), st.shape[1] if st is not None else 0, ln.parts if ln is not None else 0, ln.dim if ln is not None else 0,
             ln.eps if ln is not None else 0.0, _ptr(colsum), 1 if on_cols else 0, _ptr(rowbias), _ptr(stats_out),
             ctypes.addressof(parts) if stats_out is not None else None, int(bn))
    with _Span("gemm", 2.0 * M * N * K, 2.0 * (M * K + N * K + M * n_out)):
        check(lib.vdb_gemm_ln_bf16(*cargs, _stream()), "gemm_ln_bf16")
    if _RECORD is not None:
        _RECORD.append((lib.vdb_gemm_ln_bf16, cargs, (a, w, bias, resid, out, st, colsum, rowbias, stats_out, parts), 2.0 * M * N * K))
    return (out, parts.value) if stats_out is not None else out


def conv3x3(x, w, bias=None, resid=None, out=None, mode=0, skip1=None, skip2=None, act=ACT_NONE,
            out_dtype=BF16, bias_bstride=0, bn=0, ksplit=0):
    """3x3 conv on NHWC bf16 x [B,H,W,C]; w [N, 9*C + Cs1 + Cs2] packed (ky,kx,c | skip)."""
    _need(x, BF16, "x"); _need(w, BF16, "w"); _need(bias, torch.float32, "bias")
    _need(resid, BF16, "resid"); _need(skip1, BF16, "skip1"); _need(skip2, BF16, "skip2")
    B, H, W, Cc = x.shape
    N = w.shape[0]
    Ho, Wo = (H // 2, W // 2) if mode in (1, 2) else (H, W)
    cs1 = skip1.shape[-1] if skip1 is not None else 0
    cs2 = skip2.shape[-1] if skip2 is not None else 0
    ntaps = 4 if mode >= 3 else 9          # modes 3..6 (7..10: stored interleaved into `out` [B,2H,2W,N]): folded nearest-2x upsample
    assert w.shape[1] == ntaps * Cc + cs1 + cs2, (w.shape, Cc, cs1, cs2, mode)
    if out is None:
        out = torch.empty((B, Ho, Wo, N), dtype=out_dtype, device=x.device)
    M = B * Ho * Wo
    ws, ws_bytes = None, 0
    if ksplit != 1 and M <= 8192:
        ws, ws_bytes = workspace(x.device), WORKSPACE_BYTES
    ktot = ntaps * Cc + cs1 + cs2
    cargs = (_ptr(x), B, H, W, Cc, int(mode), _ptr(w), N, w.stride(0), _ptr(skip1), cs1,
             _ptr(skip2), cs2, _ptr(bias), int(bias_bstride), _ptr(resid),
             resid.shape[-1] if resid is not None else 0, _ptr(out), out.shape[-1],
             1 if out_dtype == torch.float32 else 0, int(act), int(bn), int(ksplit), _ptr(ws), ws_bytes)
    with _Span("conv3x3", 2.0 * M * N * ktot, 2.0 * (B * H * W * Cc + M * (cs1 + cs2) + N * ktot + M * N)):
        check(lib.vdb_conv3x3_bf16(*cargs, _stream()), "conv3x3_bf16")
    if _RECORD is not None:
        _RECORD.append((lib.vdb_conv3x3_bf16, cargs, (x, w, skip1, skip2, bias, resid, out, ws), 2.0 * M * N * ktot))
    return out


def attention_pads(d_head):
    dk, dv = lib.vdb_attention_dk_pad(d_head), lib.vdb_attention_dv_pad(d_head)
    if dk < 0 or dv < 0:
        raise ValueError(f"d_head {d_head} unsupported by the attention kernel")
    return dk, dv


def attention(q, k, vt, out, B, H, Nq, Nk, d_head, scale=None, q_col0=0, k_col0=0, causal=False,
              q_bstride=0, kv_bstride=0, kv_len=None):
    """Flash attention. q [B*q_bstride, ldq], k [B*kv_bstride, ldk], vt [H*DVP, B*kv_bstride], out [B*q_bstride, H*d_head].
    kv_bstride (default Nk) must be a multiple of 8: pad ragged contexts per batch item.
    kv_len: int32 device tensor [B] -> batch item b attends to its first kv_len[b] keys only (vdb_attention_keylen_bf16)."""
    _need(q, BF16, "q", True); _need(k, BF16, "k", True); _need(vt, BF16, "vt", True); _need(out, BF16, "out", True)
    _need(kv_len, torch.int32, "kv_len")
    if kv_len is not None and kv_len.numel() < B:
        raise ValueError(f"kv_len: need one key count per batch item ({B}), got {kv_len.numel()}")
    if scale is None:
        scale = d_head ** -0.5
    args = (_ptr(q), q.stride(0), int(q_col0), _ptr(k), k.stride(0), int(k_col0), _ptr(vt), vt.stride(0), _ptr(out),
            out.stride(0), B, H, Nq, Nk, int(q_bstride), int(kv_bstride), d_head, float(scale), 1 if causal else 0)
    with _Span("attention", 4.0 * B * H * Nq * Nk * d_head, 2.0 * B * H * d_head * (2 * Nq + 2 * Nk)):
        if kv_len is None:
            check(lib.vdb_attention_bf16(*args, _stream()), "attention_bf16")
        else:
            check(lib.vdb_attention_keylen_bf16(*args, _ptr(kv_len), _stream()), "attention_keylen_bf16")
    return out


def groupnorm(x1, gamma, beta, eps, act=ACT_NONE, x2=None, out=None, groups=32):
    """GN32(+SiLU) over NHWC bf16 [B,H,W,C1] (+ concat x2 [B,H,W,C2]) -> [B,H,W,C1+C2]."""
    _need(x1, BF16, "x1"); _need(x2, BF16, "x2"); _need(gamma, torch.float32, "gamma"); _need(beta, torch.float32, "beta")
    B = x1.shape[0]
    C1 = x1.shape[-1]
    C2 = x2.shape[-1] if x2 is not None else 0
    HW = x1.numel() // (B * C1)
    if out is None:
        out = torch.empty(x1.shape[:-1] + (C1 + C2,), dtype=BF16, device=x1.device)
    partial = _gn_scratch(x1.device, lib.vdb_groupnorm_scratch_floats(B, HW))
    with _Span("groupnorm", 0.0, 2.0 * 3 * B * HW * (C1 + C2)):
        check(lib.vdb_groupnorm_nhwc(_ptr(x1), C1, _ptr(x2), C2, B, HW, groups, _ptr(gamma), _ptr(beta), float(eps),
                                     int(act), _ptr(partial), _ptr(out), _stream()), "groupnorm_nhwc")
    return out


def layernorm(x, gamma, beta, eps=1e-5, out=None):
    _need(x, BF16, "x"); _need(gamma, torch.float32, "gamma"); _need(beta, torch.float32, "beta")
    C = x.shape[-1]
    rows = x.numel() // C
    if out is None:
        out = torch.empty_like(x)
    with _Span("layernorm", 0.0, 2.0 * 2 * rows * C):
        check(lib.vdb_layernorm(_ptr(x), rows, C, _ptr(gamma), _ptr(beta), float(eps), _ptr(out), _stream()), "layernorm")
    return out


def affine_silu_rows(x, gamma, beta, act=ACT_SILU, out=None):
    """y[r, i] = act(x[r, i] * gamma[i] + beta[i]); x bf16 [rows, n], gamma / beta fp32 [n] (FCBlock's per-position GroupNorm affine)."""
    _need(x, BF16, "x"); _need(gamma, torch.float32, "gamma"); _need(beta, torch.float32, "beta")
    rows, n = x.shape
    if out is None:
        out = torch.empty_like(x)
    check(lib.vdb_affine_act_rows(_ptr(x), rows, n, _ptr(gamma), _ptr(beta), int(act), _ptr(out), _stream()), "affine_act_rows")
    return out


def pack_conv_weight(w, out=None, col0=0):
    """Conv2d weight fp32 [Cout, Cin, kh, kw] -> bf16 [Cout, ldo] with column col0 + (ky*kw + kx)*Cin + ci (C ABI repack)."""
    _need(w, torch.float32, "w")
    Cout, Cin, kh, kw = w.shape
    if out is None:
        out = torch.empty((Cout, col0 + kh * kw * Cin), dtype=BF16, device=w.device)
    check(lib.vdb_pack_conv_weight(_ptr(w), Cout, Cin, kh, kw, _ptr(out), out.stride(0), col0, _stream()), "pack_conv_weight")
    return out


def pack_geglu(w, b=None):
    """GEGLU.proj weight fp32 [2*n2, K] (+ bias) -> (bf16 rows interleaved per 256-row tile, fp32 bias in the same order)."""
    _need(w, torch.float32, "w")
    n2, K = w.shape[0] // 2, w.shape[1]
    wo = torch.empty((2 * n2, K), dtype=BF16, device=w.device)
    bo = torch.empty(2 * n2, dtype=torch.float32, device=w.device) if b is not None else None
    if b is not None:
        _need(b, torch.float32, "b")
    check(lib.vdb_pack_geglu(_ptr(w), _ptr(b) if b is not None else None, n2, K, _ptr(wo), _ptr(bo) if bo is not None else None,
                             _stream()), "pack_geglu")
    return wo, bo


def pad_heads(w, H, d, dpad):
    """attention projection fp32 [H*d, K] -> bf16 [H*dpad, K], zero rows after each head's d rows."""
    _need(w, torch.float32, "w")
    out = torch.empty((H * dpad, w.shape[1]), dtype=BF16, device=w.device)
    check(lib.vdb_pad_heads(_ptr(w), H, d, dpad, w.shape[1], _ptr(out), _stream()), "pad_heads")
    return out


def upsample2x(x, out=None):
    _need(x, BF16, "x")
    B, H, W, C = x.shape
    if out is None:
        out = torch.empty((B, 2 * H, 2 * W, C), dtype=BF16, device=x.device)
    check(lib.vdb_upsample2x_nhwc(_ptr(x), B, H, W, C, _ptr(out), _stream()), "upsample2x")
    return out


def interleave2x2(src, out=None):
    """src bf16 [4, B, H, W, C] (parity py*2+px major) -> [B, 2H, 2W, C]."""
    _need(src, BF16, "src")
    _, B, H, W, C = src.shape
    if out is None:
        out = torch.empty((B, 2 * H, 2 * W, C), dtype=BF16, device=src.device)
    check(lib.vdb_interleave2x2_nhwc(_ptr(src), B, H, W, C, _ptr(out), _stream()), "interleave2x2")
    return out


def upsample2x_conv3x3_folded(x, wf, bias=None):
    """nearest-2x upsample + 3x3 conv (pad 1) without materialising the upsampled image: four 2x2-tap convs on the source
    (one per output parity, weights folded by diffusion_utils.fold_upsample_conv3x3) + one interleave pass.
    x bf16 [B,H,W,C]; wf bf16 [4, N, 4*C]; -> [B,2H,2W,N]."""
    B, H, W, _ = x.shape
    N = wf.shape[1]
    if N % 32 == 0 and os.environ.get("VDB_UPFOLD_DIRECT", "1") != "0" and os.environ.get("VDB_EPI_TMA", "1") != "0" \
            and os.environ.get("VDB_IGEMM_SPEC", "1") != "0":
        # modes 7..10: every parity conv stores straight into its pixels of the [B,2H,2W,N] result (output tensor map with
        # doubled strides): no interleave pass, no parity temporaries
        out = torch.empty((B, 2 * H, 2 * W, N), dtype=BF16, device=x.device)
        for par in range(4):
            conv3x3(x, wf[par], bias=bias, out=out, mode=7 + par, ksplit=1)
        return out
    parts = torch.empty((4, B, H, W, N), dtype=BF16, device=x.device)
    for par in range(4):
        conv3x3(x, wf[par], bias=bias, out=parts[par], mode=3 + par, ksplit=1)
    return interleave2x2(parts)


def im2col3x3_small(x, kpad=64, in_scale=1.0, in_shift=0.0, out=None):
    """x fp32 NHWC [B,H,W,Cin<=7] -> bf16 [B*H*W, kpad]."""
    _need(x, torch.float32, "x")
    B, H, W, Cin = x.shape
    if out is None:
        out = torch.empty((B * H * W, kpad), dtype=BF16, device=x.device)
    check(lib.vdb_im2col3x3_small(_ptr(x), B, H, W, Cin, kpad, float(in_scale), float(in_shift), _ptr(out), _stream()),
          "im2col3x3_small")
    return out


def nchw_to_nhwc(x, mul=1.0, add=0.0, out=None):
    _need(x, torch.float32, "x")
    B, C = x.shape[:2]
    HW = x.numel() // (B * C)
    if out is None:
        out = torch.empty((B,) + tuple(x.shape[2:]) + (C,), dtype=torch.float32, device=x.device)
    check(lib.vdb_permute_f32(_ptr(x), B, C, HW, 1, float(mul), float(add), 0, _ptr(out), _stream()), "permute")
    return out


def nhwc_to_nchw(x, mul=1.0, add=0.0, clamp01=False, out=None):
    _need(x, torch.float32, "x")
    B, C = x.shape[0], x.shape[-1]
    HW = x.numel() // (B * C)
    if out is None:
        out = torch.empty((B, C) + tuple(x.shape[1:-1]), dtype=torch.float32, device=x.device)
    check(lib.vdb_permute_f32(_ptr(x), B, C, HW, 0, float(mul), float(add), 1 if clamp01 else 0, _ptr(out), _stream()),
          "permute")
    return out


def to_bf16(x, out=None):
    _need(x, torch.float32, "x")
    if out is None:
        out = torch.empty(x.shape, dtype=BF16, device=x.device)
    check(lib.vdb_cast_f32_bf16(_ptr(x), _ptr(out), x.numel(), _stream()), "cast")
    return out


def to_f32(x, out=None):
    _need(x, BF16, "x")
    if out is None:
        out = torch.empty(x.shape, dtype=torch.float32, device=x.device)
    check(lib.vdb_cast_bf16_f32(_ptr(x), _ptr(out), x.numel(), _stream()), "cast")
    return out


def pointwise_small(x, w, bias=None, pre_mul=1.0, out=None):
    """x fp32 [..., Cin<=8] NHWC, w fp32 [Cout, Cin] -> fp32 [..., Cout]."""
    _need(x, torch.float32, "x"); _need(w, torch.float32, "w"); _need(bias, torch.float32, "bias")
    cout, cin = w.shape
    npix = x.numel() // cin
    if out is None:
        out = torch.empty(x.shape[:-1] + (cout,), dtype=torch.float32, device=x.device)
    check(lib.vdb_pointwise_small(_ptr(x), npix, cin, cout, _ptr(w), _ptr(bias), float(pre_mul), _ptr(out), _stream()),
          "pointwise_small")
    return out


def gaussian_sample(moments, noise=None, post_mul=1.0, out=None):
    """moments fp32 NHWC [..., 2C]; noise fp32 NHWC [..., C] or None (posterior mean)."""
    _need(moments, torch.float32, "moments"); _need(noise, torch.float32, "noise")
    C = moments.shape[-1] // 2
    npix = moments.numel() // (2 * C)
    if out is None:
        out = torch.empty(moments.shape[:-1] + (C,), dtype=torch.float32, device=moments.device)
    check(lib.vdb_gaussian_sample(_ptr(moments), _ptr(noise), C, npix, float(post_mul), _ptr(out), _stream()),
          "gaussian_sample")
    return out


def timestep_embedding(ts, dim, max_period=10000, step_idx=None, batch=None, out=None):
    """ts int64 device tensor [B] (or a table + step_idx int32 device scalar, broadcast to `batch` rows)."""
    _need(ts, torch.int64, "timesteps")
    B = batch if step_idx is not None else ts.shape[0]
    if out is None:
        out = torch.empty((B, dim), dtype=torch.float32, device=ts.device)
    nlp = torch.tensor(-math.log(max_period), dtype=torch.float32).item()
    check(lib.vdb_timestep_embedding(_ptr(ts), _ptr(step_idx), B, dim, nlp, _ptr(out), _stream()), "timestep_embedding")
    return out


def linear_small(x, w, bias=None, act_in=ACT_NONE, act_out=ACT_NONE, out=None):
    """x fp32 [M<=16,K], w bf16 [N,K] -> fp32 [M,N]."""
    _need(x, torch.float32, "x"); _need(w, BF16, "w"); _need(bias, torch.float32, "bias")
    M, K = x.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=x.device)
    check(lib.vdb_linear_small(_ptr(x), M, K, _ptr(w), N, _ptr(bias), int(act_in), int(act_out), _ptr(out), _stream()),
          "linear_small")
    return out


def softmax_rows(x, scale=1.0, out=None):
    _need(x, BF16, "x")
    n = x.shape[-1]
    rows = x.numel() // n
    if out is None:
        out = torch.empty_like(x)
    check(lib.vdb_softmax_rows(_ptr(x), rows, n, x.stride(-2) if x.dim() > 1 else n, float(scale), _ptr(out), _stream()),
          "softmax_rows")
    return out


def to_uint8_hwc(images):
    """fp32 CUDA [n,3,H,W] in [0,1] -> uint8 [n,H,W,3] with torchvision.ToPILImage semantics (x * 255 truncated)."""
    _need(images, torch.float32, "images")
    n, ch, H, W = images.shape
    assert ch == 3
    out = torch.empty((n, H, W, 3), dtype=torch.uint8, device=images.device)
    check(lib.vdb_clip_to_u8_hwc(_ptr(images), n, H, W, _ptr(out), _stream()), "clip_to_u8_hwc")
    return out


def clip_preprocess_device(images, tables, size, mean, std):
    """images fp32 CUDA [n,3,H,W] in [0,1] -> fp32 [n,3,size,size], bit-exact with ToPILImage + Pillow bicubic resize of the
    shortest side + centre crop + rescale + normalise (reference clip.py:88-94 runs this on the host through PIL).
    tables = {"nw","nh","h": (bounds, kk) or None, "v": (bounds, kk) or None} with int32 CUDA tensors (clip.pil_bicubic_coeffs)."""
    import ctypes
    _need(images, torch.float32, "images")
    n, _, H, W = images.shape
    nw, nh = tables["nw"], tables["nh"]
    u8 = torch.empty((n, H, W, 3), dtype=torch.uint8, device=images.device)
    check(lib.vdb_clip_to_u8_hwc(_ptr(images), n, H, W, _ptr(u8), _stream()), "clip_to_u8_hwc")
    if tables["h"] is not None:
        hb, hk = tables["h"]
        mid = torch.empty((n, H, nw, 3), dtype=torch.uint8, device=images.device)
        check(lib.vdb_resample_h_u8(_ptr(u8), n, H, W, nw, _ptr(hb), _ptr(hk), hk.shape[1], _ptr(mid), _stream()), "resample_h_u8")
    else:
        mid = u8
    out = torch.empty((n, 3, size, size), dtype=torch.float32, device=images.device)
    vb, vk = tables["v"] if tables["v"] is not None else (None, None)
    m3, s3 = (ctypes.c_float * 3)(*mean), (ctypes.c_float * 3)(*std)
    check(lib.vdb_resample_v_crop_norm(_ptr(mid), n, H, nw, _ptr(vb), _ptr(vk), 0 if vk is None else vk.shape[1],
                                       (nh - size) // 2, (nw - size) // 2, size, m3, s3, _ptr(out), _stream()),
          "resample_v_crop_norm")
    return out


# ------------------------------------------------------------------------------------------------ CLIP ends
def clip_text_embed(tokens, tok_emb, pos_emb, Lp):
    _need(tokens, torch.int64, "tokens"); _need(tok_emb, torch.float32, "tok_emb"); _need(pos_emb, torch.float32, "pos_emb")
    B, L = tokens.shape
    C = tok_emb.shape[1]
    x = torch.empty((B, Lp, C), dtype=BF16, device=tokens.device)
    check(lib.vdb_clip_text_embed(_ptr(tokens), _ptr(tok_emb), _ptr(pos_emb), B, L, Lp, C, _ptr(x), _stream()), "clip_text_embed")
    return x


def patchify(pixels, patch, kpad):
    _need(pixels, torch.float32, "pixels")
    B, Cin, H, W = pixels.shape
    assert H == W
    g = H // patch
    y = torch.empty((B * g * g, kpad), dtype=BF16, device=pixels.device)
    check(lib.vdb_patchify(_ptr(pixels), B, Cin, H, patch, kpad, _ptr(y), _stream()), "patchify")
    return y


def vit_assemble(patches, cls, pos, B, L, Lp, tok_scale=None):
    _need(patches, BF16, "patches"); _need(cls, torch.float32, "cls"); _need(pos, torch.float32, "pos")
    _need(tok_scale, torch.float32, "tok_scale")
    C = patches.shape[1]
    x = torch.empty((B, Lp, C), dtype=BF16, device=patches.device)
    check(lib.vdb_vit_assemble(_ptr(patches), _ptr(cls), _ptr(pos), _ptr(tok_scale), B, L, Lp, C, _ptr(x), _stream()), "vit_assemble")
    return x


def scale_by_row_norm(z, L, idx=None, row_scale=None):
    """z bf16 [B, Lp, C] -> fp32 [B, L, C] divided by the norm of row idx[b] (token 0 when idx is None)."""
    _need(z, BF16, "z"); _need(idx, torch.int32, "idx"); _need(row_scale, torch.float32, "row_scale")
    B, Lp, C = z.shape
    out = torch.empty((B, L, C), dtype=torch.float32, device=z.device)
    check(lib.vdb_scale_by_row_norm(_ptr(z), _ptr(idx), _ptr(row_scale), B, L, Lp, C, _ptr(out), _stream()), "scale_by_row_norm")
    return out


# ------------------------------------------------------------------------------------------------
# Optimus GPT-2 text decode (optimus.py:662-688): KV-cache attention, on-device sampling, <BOS> embedding
# ------------------------------------------------------------------------------------------------
def kv_decode_attention(qkv, mem, kcache, vcache, step, H, out, scale=0.125):
    """qkv [n, >=3*H*64] bf16 (row-strided ok), mem [n, >=H*64] bf16 view of this layer's memory slot, caches bf16
    [n, H, 32, 64], step int32 [1] device counter; writes out [n, H*64] bf16."""
    _need(qkv, BF16, "qkv", True); _need(mem, BF16, "mem", True); _need(kcache, BF16, "kcache"); _need(vcache, BF16, "vcache")
    _need(step, torch.int32, "step"); _need(out, BF16, "out", True)
    n = qkv.shape[0]
    assert kcache.numel() >= n * H * 32 * 64 and vcache.numel() >= n * H * 32 * 64
    check(lib.vdb_kv_decode_attention(_ptr(qkv), qkv.stride(0), _ptr(mem), mem.stride(0), _ptr(kcache), _ptr(vcache),
                                      _ptr(step), n, int(H), float(scale), _ptr(out), out.stride(0), _stream()),
          "kv_decode_attention")
    return out


def sample_tokens(logits, vocab, step, tokens, eos, temperature=None, seed=None, uniforms=None, forced=None, max_len=30,
                  wte=None, wpe=None, emb_add=None, x_next=None):
    """Draws tokens[:, t+1] from softmax(logits[:, :vocab] / temperature) (t = *step) and, with x_next, embeds it for the
    next step.  logits fp32 [n, >=vocab]; temperature fp32 [1] and seed int64 [1] device tensors; uniforms fp32 [n, >=29]
    replaces Philox; forced int32 [n, ldt] replaces sampling."""
    _need(tokens, torch.int32, "tokens"); _need(step, torch.int32, "step"); _need(logits, torch.float32, "logits", True)
    _need(temperature, torch.float32, "temperature"); _need(seed, torch.int64, "seed"); _need(uniforms, torch.float32, "uniforms")
    _need(forced, torch.int32, "forced"); _need(wte, BF16, "wte"); _need(wpe, torch.float32, "wpe")
    _need(emb_add, torch.float32, "emb_add", True); _need(x_next, BF16, "x_next", True)
    n, ldt = tokens.shape
    if forced is not None:
        assert forced.shape == tokens.shape
    C = wte.shape[1] if wte is not None else 0
    check(lib.vdb_sample_tokens(_ptr(logits), logits.stride(0) if logits is not None else 0, int(vocab), n, _ptr(temperature),
                                _ptr(step), _ptr(seed), _ptr(uniforms), uniforms.stride(0) if uniforms is not None else 0,
                                _ptr(forced), int(eos), int(max_len), _ptr(tokens), ldt, _ptr(wte), _ptr(wpe), _ptr(emb_add),
                                emb_add.stride(0) if emb_add is not None else 0, C, _ptr(x_next),
                                x_next.stride(0) if x_next is not None else 0, _stream()), "sample_tokens")
    return tokens


def token_embed(tokens, wte, wpe, emb_add, out, step=None, pos_offset=1):
    """out[r] = bf16(wte[tokens[r, t]] + wpe[t + pos_offset] + emb_add[r]), t = *step (0 without a counter)."""
    _need(tokens, torch.int32, "tokens"); _need(wte, BF16, "wte"); _need(wpe, torch.float32, "wpe")
    _need(emb_add, torch.float32, "emb_add", True); _need(out, BF16, "out", True); _need(step, torch.int32, "step")
    n, ldt = tokens.shape
    check(lib.vdb_token_embed(_ptr(tokens), ldt, _ptr(step), int(pos_offset), _ptr(wte), _ptr(wpe), _ptr(emb_add),
                              emb_add.stride(0), n, wte.shape[1], _ptr(out), out.stride(0), _stream()), "token_embed")
    return out


# ------------------------------------------------------------------------------------------------
# Optimus BERT text encode (optimus.py:729-743): the embedding layer; the encoder layers use gemm / attention(kv_len) / layernorm
# ------------------------------------------------------------------------------------------------
def bert_embed_ln(ids, word_emb, pos_emb, type_emb, gamma, beta, eps=1e-12, out=None):
    """ids int32 [n, L] -> bf16 [n*L, C] = LayerNorm(word_emb[ids] + pos_emb[:L] + type_emb[0]) (fp32 tables read in place)."""
    _need(ids, torch.int32, "ids"); _need(word_emb, torch.float32, "word_emb"); _need(pos_emb, torch.float32, "pos_emb")
    _need(type_emb, torch.float32, "type_emb"); _need(gamma, torch.float32, "gamma"); _need(beta, torch.float32, "beta")
    n, L = ids.shape
    C = word_emb.shape[1]
    if pos_emb.shape[1] != C or type_emb.shape[-1] != C or gamma.numel() != C or beta.numel() != C:
        raise ValueError(f"bert_embed_ln: tables of width {C}, {pos_emb.shape[1]}, {type_emb.shape[-1]}, gamma {gamma.numel()}, "
                         f"beta {beta.numel()} disagree")
    if out is None:
        out = torch.empty((n * L, C), dtype=BF16, device=ids.device)
    _need(out, BF16, "out")
    assert out.shape == (n * L, C), (tuple(out.shape), n * L, C)
    check(lib.vdb_bert_embed_ln(_ptr(ids), n, L, _ptr(word_emb), word_emb.shape[0], _ptr(pos_emb), pos_emb.shape[0],
                                _ptr(type_emb), _ptr(gamma), _ptr(beta), float(eps), C, _ptr(out), _stream()), "bert_embed_ln")
    return out
