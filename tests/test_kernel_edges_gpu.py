"""The shared tensor-core entry points (vdb_gemm_bf16, vdb_conv3x3_bf16, vdb_attention_bf16 / _keylen_bf16) and the small
elementwise kernels at the shapes, layouts and kernel-selection boundaries where kernels go wrong, against an fp64 restatement
of the same operation on the same bf16-rounded operands, with a bound per element.

Error model (u = 2^-24, the fp32 unit roundoff).
  GEMM / conv.  P = alpha * (A W^T + bias), ref = act(P) + resid, S = |alpha| * (|A| |W|^T), all in fp64:
      |out - ref| <= u_out |ref| + u_mid |act(P)| [resid] + 1.2 K_tot u S + 4 u |act(P)|
    - u_out = 2^-8 for bf16 output (round to nearest is 2^-9; the rest absorbs the fp32 error in front of the rounding) and
      2^-23 for fp32 output (two fp32 roundings: the bias add and the alpha product);
    - u_mid = 2^-8 for an epilogue that rounds act(P) to bf16 before the residual add (none here does, so it is 0);
    - K_tot u S bounds any fp32 accumulation order of the K_tot products (tensor-core partial sums, the split-K reduction);
      1.2 bounds the slope of every activation of the VDB_ACT_* enum, which carries that error through the epilogue;
    - 4 u |act(P)| covers the epilogue's own fp32 roundings (bias, alpha, activation).
  Attention.  With V1[i, c] = sum_j p_ij |v_jc| in fp64:
      |out - ref| <= 2^-8 |ref| + 2^-7 V1 + (scale d 2^-23 max_j sum_c |q_ic| |k_jc|) V1
    - 2^-8 |ref| covers the bf16 output rounding and a row sum taken over the unrounded probabilities;
    - 2^-7 V1 covers the bf16 rounding of P fed to the PV product and the degree-3 polynomial exp2 of the two-tile kernel
      (7.7e-5 relative);
    - the last term carries the fp32 QK^T accumulation error through the exponential.
  A cosine check against the reference stays as a secondary sanity check.

Guard bands.  Every output, and the split-K workspace, lives inside a larger allocation filled with a NaN bit pattern no kernel
produces (bf16 0x7FA5, fp32 0x7FA5A5A5): column slices with ldo > N and rows above and below, the pad rows [Nq, q_bstride) of
attention outputs, a trailing band behind fp32 outputs with ldo = N.  After each call every element outside the view must still
hold the pattern bit for bit.  Base pointers stay 16-byte aligned and leading dimensions multiples of 8.

Path record.  vdb_debug_igemm_last / vdb_debug_attention_last (debug aids, not in include/vdb200.h) report the epilogue mode, BN,
ksplit and CTA pairing of the last GEMM / conv launch and the attention kernel family of the last attention launch; every case
of the three tables asserts the path it exists for, and test_path_tables_cover_every_kernel_path checks that the tables cover
every path.  The path assertions (not the numerics) are skipped when a VDB_* kernel switch is set, as the variant runs do.
"""
import ctypes
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda"
U = 2.0 ** -24
SENT16 = 0x7FA5
SENT32 = 0x7FA5A5A5

# kernel switches read by libvdb200 (getenv in csrc/): any of them set changes which kernel serves a shape
_SWITCHES = ("VDB_ATT_BKV", "VDB_ATT_FA", "VDB_ATT_ONES", "VDB_ATT_SW", "VDB_BN_MODEL", "VDB_CHUNKED", "VDB_EPI_ALT", "VDB_EPI_TMA",
             "VDB_IGEMM_SPEC", "VDB_NFAST", "VDB_PAIR", "VDB_PDL")
CHECK_PATHS = not any(k in os.environ for k in _SWITCHES)

# epilogue modes of igemm_kernel after the TMA-store promotion: 0 generic, 1 / 3 plain bf16 (3 = TMA store), 2 / 4 GEGLU
MODES = {"generic": {0}, "fast": {1, 3}, "geglu": {2, 4}}
# vdb_debug_attention_last ids (csrc/attention.cu)
ATT_TWO_TILE, ATT_COLS64_DBUF, ATT_COLS64, ATT_COLS128, ATT_D80, ATT_D160, ATT_KEYLEN64, ATT_KEYLEN128 = 1, 2, 3, 4, 5, 6, 7, 8


def _lib():
    from vdb200._lib import lib
    if not getattr(lib, "_edges_bound", False):
        lib.vdb_debug_igemm_last.argtypes = [ctypes.c_void_p]
        lib.vdb_debug_igemm_last.restype = None
        lib.vdb_debug_attention_last.argtypes = []
        lib.vdb_debug_attention_last.restype = ctypes.c_int
        lib._edges_bound = True
    return lib


def _check(status, what):
    from vdb200._lib import check
    check(status, what)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def igemm_last():
    r = (ctypes.c_int * 4)()
    _lib().vdb_debug_igemm_last(ctypes.addressof(r))
    return {"mode": r[0], "bn": r[1], "ksplit": r[2], "pair": r[3]}


def assert_igemm_path(want, what):
    """want: {"mode": "generic" | "fast" | "geglu", "bn": int, "split": True | False | int}"""
    if not CHECK_PATHS:
        return
    got = igemm_last()
    if "mode" in want:
        assert got["mode"] in MODES[want["mode"]], f"{what}: epilogue mode {got['mode']}, want {want['mode']}"
    if "bn" in want:
        assert got["bn"] == want["bn"], f"{what}: BN {got['bn']}, want {want['bn']}"
    if "split" in want:
        s = want["split"]
        ok = (got["ksplit"] > 1) if s is True else (got["ksplit"] == 1 if s is False else got["ksplit"] == s)
        assert ok, f"{what}: ksplit {got['ksplit']}, want {s}"


def assert_attention_path(want, what):
    if CHECK_PATHS:
        got = _lib().vdb_debug_attention_last()
        assert got == want, f"{what}: attention kernel {got}, want {want}"


# ---------------------------------------------------------------------------------------------------------------------------
# operands, guarded outputs, bounds
# ---------------------------------------------------------------------------------------------------------------------------
def rnd(*shape, scale=1.0, seed=0, dtype=torch.bfloat16):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(dtype).to(DEV)


def _r8(n):
    return (n + 7) // 8 * 8


class Guarded(object):
    """A [rows, cols] view at (top, col0) of a [top + rows + bottom, ld] sentinel-filled allocation (flat=True: a dense
    [rows, cols] block at element offset `top` of a 1-D allocation with `bottom` trailing elements)."""

    def __init__(self, rows, cols, dtype, top=3, bottom=5, col0=0, ld=None, flat=False):
        self.dtype = dtype
        if flat:
            self.buf = torch.empty(top + rows * cols + bottom, dtype=dtype, device=DEV)
            self.view = self.buf[top:top + rows * cols].view(rows, cols)
            self.inside = torch.zeros(self.buf.shape, dtype=torch.bool, device=DEV)
            self.inside[top:top + rows * cols] = True
        else:
            ld = ld if ld is not None else col0 + _r8(cols) + 8
            self.buf = torch.empty(top + rows + bottom, ld, dtype=dtype, device=DEV)
            self.view = self.buf[top:top + rows, col0:col0 + cols]
            self.inside = torch.zeros(self.buf.shape, dtype=torch.bool, device=DEV)
            self.inside[top:top + rows, col0:col0 + cols] = True
        self._bits().fill_(SENT16 if dtype == torch.bfloat16 else SENT32)
        assert self.view.data_ptr() % 16 == 0

    def _bits(self):
        return self.buf.view(torch.int16 if self.dtype == torch.bfloat16 else torch.int32)

    def exclude(self, mask_inside):
        """narrow the written region (e.g. the pad rows of an attention output inside the view)"""
        self.inside &= mask_inside

    def check(self, what):
        bits = self._bits()[~self.inside]
        sent = SENT16 if self.dtype == torch.bfloat16 else SENT32
        bad = (bits != sent).sum().item()
        assert bad == 0, f"{what}: {bad} elements outside the output view were written"


def _act64(t, act):
    if act == 0:
        return t
    if act == 1:
        return F.silu(t)
    if act == 2:
        return F.gelu(t)
    if act == 3:
        return t * torch.sigmoid(1.702 * t)
    raise ValueError(act)


def assert_within(out, ref, bound, what, cos_min=0.999):
    """per-element |out - ref| <= bound (fp64), then the cosine sanity check"""
    o = out.double()
    assert torch.isfinite(o).all(), f"{what}: non-finite output"
    err = (o - ref).abs()
    over = err > bound
    if over.any():
        idx = torch.nonzero(over)[0].tolist()
        ratio = (err / bound.clamp_min(1e-300)).max().item()
        raise AssertionError(f"{what}: {over.sum().item()} of {err.numel()} elements exceed the bound (worst err/bound {ratio:.3g}); "
                             f"first at {idx}: out {o[tuple(idx)].item():.6g} ref {ref[tuple(idx)].item():.6g} "
                             f"bound {bound[tuple(idx)].item():.3g}")
    cos = F.cosine_similarity(o.flatten(), ref.flatten(), dim=0).item()
    assert cos >= cos_min or ref.abs().max().item() == 0, f"{what}: cosine {cos:.6f}"


def gemm_ref_bound(a64, w64, bias_rows, alpha, act, resid64, f32_out):
    """fp64 reference and per-element bound of the error model (module docstring); a64 [M, K_tot], w64 [N, K_tot]"""
    acc = a64 @ w64.t()
    if bias_rows is not None:
        acc = acc + bias_rows
    p = alpha * acc
    ap = _act64(p, act)
    ref = ap + resid64 if resid64 is not None else ap
    s = abs(alpha) * (a64.abs() @ w64.abs().t())
    u_out = 2.0 ** -23 if f32_out else 2.0 ** -8
    bound = u_out * ref.abs() + 1.2 * a64.shape[1] * U * s + 4 * U * ap.abs()
    return ref, bound


# ---------------------------------------------------------------------------------------------------------------------------
# GEMM
# ---------------------------------------------------------------------------------------------------------------------------
def G(why, M, N, K, *, K2=0, bias=None, rpb=1, resid=False, act=0, alpha=1.0, bn=0, ksplit=0, f32=False, layout="dense",
      path=None):
    return pytest.param(dict(M=M, N=N, K=K, K2=K2, bias=bias, rpb=rpb, resid=resid, act=act, alpha=alpha, bn=bn, ksplit=ksplit,
                             f32=f32, layout=layout, path=path or {}), id=why)


GEMM_CASES = [
    # alpha != 1 (the context mix ratio, attention.py:326, and Optimus' pre_scale): the generic epilogue
    G("alpha_bias_resid", 300, 320, 320, bias="vec", resid=True, alpha=0.37, ksplit=1, path={"mode": "generic", "split": False}),
    # alpha applied in the split-K reduction, fp32 output
    G("alpha_f32_splitk", 256, 320, 1280, bias="vec", alpha=0.37, ksplit=4, f32=True, path={"mode": "generic", "split": 4}),
    # per-batch bias rows whose batch items straddle a 128-row tile (mode-0 per-row bias path)
    G("straddle_rpb77", 308, 320, 320, bias="batch", rpb=77, ksplit=1, path={"mode": "generic", "split": False}),
    G("straddle_rpb100_resid", 400, 256, 192, bias="batch", rpb=100, resid=True, ksplit=1, path={"mode": "generic", "split": False}),
    # ... and through the split-K reduction's m / rows_per_batch
    G("straddle_rpb77_splitk", 231, 640, 2560, bias="batch", rpb=77, ksplit=4, path={"split": 4}),
    G("straddle_rpb100_splitk", 300, 320, 1280, bias="batch", rpb=100, resid=True, ksplit=3, path={"split": 3}),
    # the 0-D diffuser's per-row bias (rows_per_batch = 1, openaimodel.py:603): small M, automatic split-K
    G("row_bias_m8_autosplit", 8, 1280, 1280, bias="batch", rpb=1, path={"split": True}),
    # split-K reduction x output type / activation
    G("splitk_f32_resid_auto", 128, 512, 2048, bias="vec", resid=True, f32=True, path={"mode": "generic", "split": True}),
    G("splitk_silu_resid", 256, 640, 1536, bias="vec", resid=True, act=1, ksplit=6, path={"split": 6}),
    G("splitk_gelu_resid", 192, 384, 1024, bias="vec", resid=True, act=2, ksplit=4, path={"split": 4}),
    G("splitk_quickgelu", 154, 768, 768, bias="vec", act=3, ksplit=3, path={"split": 3}),
    # forced tile widths with a partial last N tile: N % 32 != 0 (generic epilogue) and N % 32 == 0 (fast / TMA-store epilogue)
    G("bn64_generic", 256, 200, 256, bias="vec", bn=64, ksplit=1, path={"mode": "generic", "bn": 64, "split": False}),
    G("bn64_fast", 256, 224, 256, bias="vec", resid=True, bn=64, ksplit=1, path={"mode": "fast", "bn": 64, "split": False}),
    G("bn128_generic", 300, 200, 320, bias="vec", resid=True, bn=128, ksplit=1, path={"mode": "generic", "bn": 128, "split": False}),
    G("bn128_fast", 300, 352, 320, bias="vec", bn=128, ksplit=1, path={"mode": "fast", "bn": 128, "split": False}),
    G("bn160_generic", 256, 200, 192, bias="vec", bn=160, ksplit=1, path={"mode": "generic", "bn": 160, "split": False}),
    G("bn160_fast", 384, 416, 192, resid=True, bn=160, ksplit=1, path={"mode": "fast", "bn": 160, "split": False}),
    G("bn256_generic", 256, 300, 256, bias="vec", bn=256, ksplit=1, path={"mode": "generic", "bn": 256, "split": False}),
    G("bn256_fast", 256, 288, 256, bias="vec", resid=True, bn=256, ksplit=1, path={"mode": "fast", "bn": 256, "split": False}),
    # M at the 128-row tile edges
    G("m1", 1, 320, 320, bias="vec", path={"split": False}),
    G("m127", 127, 256, 512, resid=True, ksplit=1, path={"mode": "fast", "split": False}),
    G("m129", 129, 320, 640, bias="vec", resid=True, ksplit=1, path={"mode": "fast", "split": False}),
    # K tails: the ABI only asks K % 8 == 0 (TMA zero-fills the last 64-wide K block)
    G("k8", 256, 128, 8, bias="vec", path={"split": False}),
    G("k72", 200, 192, 72, bias="vec", resid=True, path={"split": False}),
    G("k200", 300, 96, 200, act=2, path={"mode": "generic", "split": False}),
    G("k1000", 160, 320, 1000, bias="vec", ksplit=1, path={"mode": "fast", "split": False}),
    # two-source A with a K2 tail (torch.cat([h, skip]) folded into one GEMM)
    G("two_source_k2_72", 256, 320, 128, K2=72, bias="vec", ksplit=1, path={"mode": "fast", "split": False}),
    # narrow fp32 outputs with ldo = N (the UNet / VAE conv_out widths)
    G("n3_f32", 1000, 3, 128, bias="vec", f32=True, path={"mode": "generic", "split": False}),
    G("n4_f32", 1000, 4, 320, bias="vec", f32=True, path={"mode": "generic", "split": False}),
    G("n8_f32", 600, 8, 512, bias="vec", f32=True, ksplit=1, path={"mode": "generic", "split": False}),
    # row-strided, pointer-offset operands: the VAE AttnBlock's qk[rows, :C] @ qk[rows, C:]^T (autokl_modules.py:137-140)
    G("vae_qk_rows", 256, 256, 512, layout="vae_qk", ksplit=1, path={"mode": "fast", "split": False}),
    G("strided_a_w_bias", 200, 320, 256, bias="vec", resid=True, layout="strided", ksplit=1, path={"mode": "fast", "split": False}),
    G("strided_a_w_splitk", 96, 320, 1024, bias="vec", layout="strided", ksplit=4, path={"split": 4}),
    # GEGLU into a guarded column slice
    G("geglu_slice", 256, 2560, 320, bias="vec", act=4, path={"mode": "geglu", "bn": 256, "split": False}),
]

WS_FLOATS = 16 * 1000 * 1280      # split-K workspace of these tests (at least what any split below needs)


def guarded_workspace():
    return Guarded(1, WS_FLOATS, torch.float32, top=4, bottom=4096, flat=True)


def run_gemm(a, w, out, *, a2=None, bias=None, bias_bstride=0, rpb=1, resid=None, act=0, alpha=1.0, bn=0, ksplit=0, ws=None):
    M, K = a.shape
    N = w.shape[0]
    K2 = a2.shape[1] if a2 is not None else 0
    wsp, wsb = (ws.view.data_ptr(), ws.view.numel() * 4) if ws is not None else (None, 0)
    _check(_lib().vdb_gemm_bf16(a.data_ptr(), M, K, a.stride(0), a2.data_ptr() if a2 is not None else None, K2,
                                a2.stride(0) if a2 is not None else 0, w.data_ptr(), N, w.stride(0),
                                bias.data_ptr() if bias is not None else None, bias_bstride, rpb,
                                resid.data_ptr() if resid is not None else None, resid.stride(0) if resid is not None else 0,
                                out.data_ptr(), out.stride(0), 1 if out.dtype == torch.float32 else 0, act, alpha, bn, ksplit,
                                wsp, wsb, _stream()), "gemm_bf16")


def pack_geglu(w, b, bn=256):
    """rows [0, n2) value, [n2, 2 n2) gate -> per 256-row tile: 128 value rows then their 128 gate rows"""
    n2 = w.shape[0] // 2
    half = bn // 2
    idx = []
    for t in range(n2 // half):
        idx += list(range(t * half, (t + 1) * half)) + list(range(n2 + t * half, n2 + (t + 1) * half))
    idx = torch.tensor(idx, device=w.device)
    return w[idx].contiguous(), b[idx].contiguous()


@pytest.mark.parametrize("c", GEMM_CASES)
def test_gemm_edges(c):
    M, N, K, K2 = c["M"], c["N"], c["K"], c["K2"]
    what = f"gemm {M}x{N}x{K}+{K2}"
    a2 = None
    if c["layout"] == "vae_qk":
        # one [rows, 2C] buffer: A = qk[r0:r0+M, :C], W = qk[r0:r0+M, C:] (N == M, K == C)
        qk = rnd(M + 40, 2 * K, seed=1)
        a, w = qk[16:16 + M, :K], qk[16:16 + N, K:]
    elif c["layout"] == "strided":
        # A and W as column windows of wider buffers, starting some rows in (pointer offsets, lda / ldw > K)
        abuf = rnd(M + 7, K + 136, seed=1)
        wbuf = rnd(N + 3, K + 72, seed=2, scale=K ** -0.5)
        a, w = abuf[5:5 + M, 64:64 + K], wbuf[3:3 + N, 8:8 + K]
    else:
        a = rnd(M, K, seed=1)
        w = rnd(N, K + K2, seed=2, scale=(K + K2) ** -0.5)
        if K2:
            a2 = rnd(M, K2, seed=5)
    bias, bias_rows, bstride = None, None, 0
    if c["bias"] == "vec":
        bias = rnd(N, seed=3, dtype=torch.float32)
        bias_rows = bias.double()
    elif c["bias"] == "batch":
        nb = (M + c["rpb"] - 1) // c["rpb"]
        bias = rnd(nb, N, seed=3, dtype=torch.float32) * 4.0     # large per-batch offsets: a wrong row is obvious
        bstride = N
        bias_rows = bias.double().repeat_interleave(c["rpb"], 0)[:M]
    act = c["act"]
    n_out = N // 2 if act == 4 else N
    if act == 4:
        w, bias = pack_geglu(w, bias)
    r = None
    if c["resid"]:
        rg = Guarded(M, n_out, torch.bfloat16, col0=8)
        rg.view.copy_(rnd(M, n_out, seed=4))
        r = rg.view
    dt = torch.float32 if c["f32"] else torch.bfloat16
    if c["f32"] and N <= 8:
        og = Guarded(M, n_out, dt, top=4, bottom=37, flat=True)       # ldo = N, trailing band
    else:
        og = Guarded(M, n_out, dt, top=3, bottom=5, col0=16 if dt == torch.bfloat16 else 8)
    ws = guarded_workspace()
    run_gemm(a, w, og.view, a2=a2, bias=bias, bias_bstride=bstride, rpb=c["rpb"], resid=r, act=act, alpha=c["alpha"], bn=c["bn"],
             ksplit=c["ksplit"], ws=ws)
    torch.cuda.synchronize()
    assert_igemm_path(c["path"], what)
    og.check(what)
    ks = igemm_last()["ksplit"]
    ws.exclude(torch.arange(ws.buf.numel(), device=DEV) < 4 + (ks * M * N if ks > 1 else 0))
    ws.check(what + " workspace")
    a64 = torch.cat([a, a2], 1).double() if a2 is not None else a.double()
    w64 = w.double()
    if act == 4:
        # value / gate rows of each 256-row tile -> GELU(gate) * value
        h = a64 @ w64.t() + bias.double()
        hv = h.view(M, N // 256, 2, 128)
        val, gate = hv[:, :, 0].reshape(M, n_out), hv[:, :, 1].reshape(M, n_out)
        ref = val * F.gelu(gate)
        s = (a64.abs() @ w64.abs().t()).view(M, N // 256, 2, 128)
        sv, sg = s[:, :, 0].reshape(M, n_out), s[:, :, 1].reshape(M, n_out)
        # product of two fp32-accumulated values: each carries K u S of its own, scaled by the other factor's magnitude.  The
        # GEGLU epilogue evaluates GELU in tanh form through tanh.approx (gelu_fast_f): Phi off by < 3e-4 against the erf form
        # plus the MUFU tanh's absolute error (< 2^-10.9) times 0.5, both times |gate| |value|
        bound = (2.0 ** -8 * ref.abs() + 1.2 * K * U * (sv * F.gelu(gate).abs() + 1.2 * sg * val.abs()) + 4 * U * ref.abs()
                 + (3e-4 + 0.5 * 2.0 ** -10.9) * gate.abs() * val.abs())
    else:
        ref, bound = gemm_ref_bound(a64, w64, bias_rows, c["alpha"], act, r.double() if r is not None else None, c["f32"])
    assert_within(og.view, ref, bound, what)


def test_gemm_workspace_reuse_leaves_no_stale_partials():
    """a large split-K GEMM, then immediately a small one on the same stream and workspace: the small one's reduction must read
    only its own partials"""
    ws = guarded_workspace()
    big_a, big_w = rnd(1000, 2560, seed=1), rnd(1280, 2560, seed=2, scale=2560 ** -0.5)
    big = Guarded(1000, 1280, torch.bfloat16, col0=8)
    run_gemm(big_a, big_w, big.view, ksplit=4, ws=ws)
    assert_igemm_path({"split": 4}, "big split-K")
    sa, sw = rnd(64, 1024, seed=3), rnd(320, 1024, seed=4, scale=1024 ** -0.5)
    sb = rnd(320, seed=5, dtype=torch.float32)
    small = Guarded(64, 320, torch.float32, col0=8)
    run_gemm(sa, sw, small.view, bias=sb, ksplit=2, ws=ws)
    assert_igemm_path({"split": 2}, "small split-K")
    torch.cuda.synchronize()
    big.check("big split-K")
    small.check("small split-K")
    ref, bound = gemm_ref_bound(big_a.double(), big_w.double(), None, 1.0, 0, None, False)
    assert_within(big.view, ref, bound, "big split-K")
    ref, bound = gemm_ref_bound(sa.double(), sw.double(), sb.double(), 1.0, 0, None, True)
    assert_within(small.view, ref, bound, "small split-K after a large one")


# ---------------------------------------------------------------------------------------------------------------------------
# 3x3 conv (implicit GEMM): the reference is the same GEMM on an fp64 im2col matrix with the packed (ky, kx, c) column order
# ---------------------------------------------------------------------------------------------------------------------------
def im2col(x, mode):
    """x [B, H, W, C] -> [B*Ho*Wo, 9*C] in (ky, kx, c) order, fp64"""
    x = x.double()
    B, H, W, C = x.shape
    if mode == 0:
        xp, st, Ho, Wo = F.pad(x, (0, 0, 1, 1, 1, 1)), 1, H, W
    elif mode == 1:
        xp, st, Ho, Wo = F.pad(x, (0, 0, 1, 1, 1, 1)), 2, H // 2, W // 2
    else:
        xp, st, Ho, Wo = F.pad(x, (0, 0, 0, 1, 0, 1)), 2, H // 2, W // 2
    taps = [xp[:, ky:ky + st * (Ho - 1) + 1:st, kx:kx + st * (Wo - 1) + 1:st, :] for ky in range(3) for kx in range(3)]
    return torch.stack(taps, 3).reshape(B * Ho * Wo, 9 * C)


def C_(why, B, H, W, C, N, *, mode=0, bias="vec", skips=(), resid=False, f32=False, ksplit=0, path=None):
    return pytest.param(dict(B=B, H=H, W=W, C=C, N=N, mode=mode, bias=bias, skips=skips, resid=resid, f32=f32, ksplit=ksplit,
                             path=path or {}), id=why)


CONV_EDGE_CASES = [
    # the (TW, TH, TB) pixel box runs past the image edge (non-power-of-two latents)
    C_("m0_24x40", 2, 24, 40, 64, 128, resid=True, ksplit=1, path={"mode": "fast", "split": False}),
    C_("m0_7x9", 3, 7, 9, 128, 64, ksplit=1, path={"mode": "fast", "split": False}),
    # several images per tile (5x5 images in an 8x8x2 box)
    C_("m0_5x5_multi_image", 6, 5, 5, 64, 96, resid=True, ksplit=1, path={"mode": "fast", "split": False}),
    C_("m1_12x20", 2, 12, 20, 128, 128, mode=1, ksplit=1, path={"split": False}),
    C_("m2_24x40", 1, 24, 40, 64, 64, mode=2, ksplit=1, path={"split": False}),
    # per-batch bias (ResBlock conv1 + timestep bias, openaimodel.py:166) at 8x8: two images per 128-pixel tile
    C_("batch_bias_8x8_b3_320", 3, 8, 8, 320, 320, bias="batch", ksplit=1, path={"mode": "generic", "split": False}),
    C_("batch_bias_8x8_b8_320", 8, 8, 8, 320, 320, bias="batch", ksplit=1, path={"mode": "generic", "split": False}),
    C_("batch_bias_8x8_b3_1280_splitk", 3, 8, 8, 1280, 1280, bias="batch", path={"split": True}),
    C_("batch_bias_8x8_b8_1280_splitk", 8, 8, 8, 1280, 1280, bias="batch", path={"split": True}),
    # ResBlock tail (conv2 + 1x1 skip over cat(h, skip) + residual) at 8x8 with per-batch bias, with and without split-K
    C_("resblock_tail_8x8", 4, 8, 8, 320, 320, bias="batch", skips=(320, 320), resid=True, ksplit=1,
       path={"mode": "generic", "split": False}),
    C_("resblock_tail_8x8_splitk", 4, 8, 8, 320, 320, bias="batch", skips=(320, 320), resid=True, path={"split": True}),
    # fp32 conv_outs with ldo = N: UNet out (N 4), VAE decoder (N 3), VAE encoder (N 8)
    C_("f32_n4_c320", 2, 32, 32, 320, 4, f32=True, path={"mode": "generic"}),
    C_("f32_n3_c128", 1, 48, 40, 128, 3, f32=True, path={"mode": "generic", "split": False}),
    C_("f32_n8_c512", 2, 16, 16, 512, 8, f32=True, path={"mode": "generic"}),
]


@pytest.mark.parametrize("c", CONV_EDGE_CASES)
def test_conv3x3_edges(c):
    B, H, W, C, N, mode = c["B"], c["H"], c["W"], c["C"], c["N"], c["mode"]
    Ho, Wo = (H // 2, W // 2) if mode else (H, W)
    M = B * Ho * Wo
    what = f"conv {B}x{H}x{W}x{C}->{N} mode {mode}"
    x = rnd(B, H, W, C, seed=1)
    cs = list(c["skips"])
    skips = [rnd(B, Ho, Wo, s, seed=10 + i) for i, s in enumerate(cs)]
    ktot = 9 * C + sum(cs)
    wt = rnd(N, ktot, seed=2, scale=ktot ** -0.5)       # packed [N, (ky, kx, c) | skip columns]
    bias, bias_rows, bstride = None, None, 0
    if c["bias"] == "vec":
        bias = rnd(N, seed=3, dtype=torch.float32)
        bias_rows = bias.double()
    elif c["bias"] == "batch":
        bias = rnd(B, N, seed=3, dtype=torch.float32) * 4.0
        bstride = N
        bias_rows = bias.double().repeat_interleave(Ho * Wo, 0)
    r = rnd(B, Ho, Wo, N, seed=4) if c["resid"] else None     # dense (ldr = N)
    dt = torch.float32 if c["f32"] else torch.bfloat16
    if c["f32"] and N <= 8:
        og = Guarded(M, N, dt, top=4, bottom=61, flat=True)           # ldo = N, trailing band
    else:
        og = Guarded(M, N, dt, top=2, bottom=3, col0=8)
    ws = guarded_workspace()
    s1 = skips[0] if len(skips) > 0 else None
    s2 = skips[1] if len(skips) > 1 else None
    _check(_lib().vdb_conv3x3_bf16(x.data_ptr(), B, H, W, C, mode, wt.data_ptr(), N, wt.stride(0),
                                   s1.data_ptr() if s1 is not None else None, cs[0] if s1 is not None else 0,
                                   s2.data_ptr() if s2 is not None else None, cs[1] if s2 is not None else 0,
                                   bias.data_ptr() if bias is not None else None, bstride, r.data_ptr() if r is not None else None,
                                   N if r is not None else 0, og.view.data_ptr(), og.view.stride(0), 1 if c["f32"] else 0, 0, 0,
                                   c["ksplit"], ws.view.data_ptr(), ws.view.numel() * 4, _stream()), "conv3x3_bf16")
    torch.cuda.synchronize()
    assert_igemm_path(c["path"], what)
    og.check(what)
    ks = igemm_last()["ksplit"]
    ws.exclude(torch.arange(ws.buf.numel(), device=DEV) < 4 + (ks * M * N if ks > 1 else 0))
    ws.check(what + " workspace")
    cols = im2col(x, mode)
    if skips:
        cols = torch.cat([cols] + [s.double().reshape(M, -1) for s in skips], 1)
    ref, bound = gemm_ref_bound(cols, wt.double(), bias_rows, 1.0, 0, r.double().reshape(M, N) if r is not None else None,
                                c["f32"])
    assert_within(og.view, ref, bound, what)


# ---------------------------------------------------------------------------------------------------------------------------
# attention
# ---------------------------------------------------------------------------------------------------------------------------
def A_(why, B, H, Nq, Nk, d, *, causal=False, scale=None, fused=False, q_bs=0, kv_bs=0, kv_len=None, path=None):
    return pytest.param(dict(B=B, H=H, Nq=Nq, Nk=Nk, d=d, causal=causal, scale=scale, fused=fused, q_bs=q_bs, kv_bs=kv_bs,
                             kv_len=kv_len, path=path), id=why)


def _att_family(Nq, Nk, d, causal=False):
    """the default kernel choice of attention_entry (csrc/attention.cu)"""
    if d > 80:
        return ATT_D160
    if d > 64:
        return ATT_D80
    if not causal and Nk >= 512 and Nq >= 256 and Nq % 256 == 0:
        return ATT_TWO_TILE
    return ATT_COLS64 if 64 < Nk <= 512 else ATT_COLS128


ATT_CASES = [
    # fused q|k projections (one [rows, 2 H DK] buffer, q_col0 = 0, k_col0 = H DK; attention.py:203,232)
    A_("fused_d40_n1024", 1, 2, 1024, 1024, 40, fused=True, path=ATT_TWO_TILE),
    A_("fused_d80_n256", 2, 3, 256, 256, 80, fused=True, path=ATT_D80),
    A_("fused_d160_n64", 2, 2, 64, 64, 160, fused=True, path=ATT_D160),
    # CLIP text: causal 77 tokens stored 80 per batch item (clip.py:121), garbage in the pad rows, guarded output pad rows
    A_("clip_causal_77_in_80", 2, 4, 77, 77, 64, causal=True, fused=True, q_bs=80, kv_bs=80, path=ATT_COLS64),
    # q_bstride > Nq without the fused layout
    A_("q_bstride_gt_nq", 2, 2, 100, 264, 40, q_bs=136, kv_bs=264, path=ATT_COLS64),
]
# key counts around the kernel-selection boundaries (<= 64: 128-column kernel, 65..512: three-CTA, >= 512 with Nq % 256 == 0:
# two-tile kernel) at d_head 40 (DVP 48) and 64
ATT_CASES += [A_(f"nk{nk}_d{d}", 2, 2, 256, nk, d, path=_att_family(256, nk, d))
              for d in (40, 64) for nk in (1, 8, 63, 64, 65, 511, 512, 513)]
# query counts around the two-tile kernel's Nq % 256 condition
ATT_CASES += [A_(f"nq{nq}_nk640", 2, 2, nq, 640, 64, path=_att_family(nq, 640, 64)) for nq in (1, 255, 256, 257)]
# a non-default softmax scale on every kernel family
ATT_CASES += [A_(f"scale{s}_{name}", 2, 2, nq, nk, d, scale=s, path=_att_family(nq, nk, d))
              for s in (0.3, 1.0)
              for name, nq, nk, d in (("two_tile", 256, 640, 40), ("cols64", 200, 300, 64), ("cols128", 200, 700, 40),
                                      ("d80", 200, 300, 80), ("d160", 130, 200, 160))]
ATT_CASES += [A_(f"scale{s}_keylen", 3, 2, 100, 80, 64, scale=s, kv_len=(80, 37, 1), path=ATT_KEYLEN64) for s in (0.3, 1.0)]
# d_head sweep (88..128 run on the (192, 160) kernel)
ATT_CASES += [A_(f"dhead{d}", 2, 3, 200, 300, d, path=_att_family(200, 300, d)) for d in range(8, 161, 8)]
# per-batch key counts, 0 and Nk + 7 included (clamped to [1, Nk])
ATT_CASES += [A_("keylen_nk80", 5, 2, 80, 80, 64, kv_len=(0, 1, 37, 80, 87), path=ATT_KEYLEN64),
              A_("keylen_nk600", 5, 2, 96, 600, 64, kv_len=(0, 1, 37, 600, 607), path=ATT_KEYLEN128)]


@pytest.mark.parametrize("c", ATT_CASES)
def test_attention_edges(c):
    from vdb200 import ops
    B, H, Nq, Nk, d = c["B"], c["H"], c["Nq"], c["Nk"], c["d"]
    DK, DVP = ops.attention_pads(d)
    fused = c["fused"]
    q_bs = c["q_bs"] or Nq
    kv_bs = c["kv_bs"] or _r8(Nk)
    if fused:
        assert Nq == Nk and q_bs == kv_bs
    what = f"attention B{B} H{H} {Nq}x{Nk} d{d}" + (" causal" if c["causal"] else "") + (" fused" if fused else "")
    g = torch.Generator().manual_seed(1000 * d + Nk + Nq)
    q = (torch.randn(B, H, Nq, d, generator=g) * 2.0).to(torch.bfloat16)    # peaky enough to exercise the rescale path
    k = torch.randn(B, H, Nk, d, generator=g).to(torch.bfloat16)
    v = torch.randn(B, H, Nk, d, generator=g).to(torch.bfloat16)
    garbage = lambda *s: (torch.randn(*s, generator=g) * 8.0).to(torch.bfloat16)     # noqa: E731
    # Q / K buffers: real rows hold the heads' d channels and zero head padding; rows past Nq / Nk hold garbage
    if fused:
        QK = garbage(B, q_bs, 2, H, DK)
        QK[:, :Nq] = 0
        QK[:, :Nq, 0, :, :d] = q.permute(0, 2, 1, 3)
        QK[:, :Nk, 1, :, :d] = k.permute(0, 2, 1, 3)
        QK = QK.reshape(B * q_bs, 2 * H * DK).to(DEV)
        Q, K, q_col0, k_col0 = QK, QK, 0, H * DK
    else:
        Qh = garbage(B, q_bs, H, DK)
        Qh[:, :Nq] = 0
        Qh[:, :Nq, :, :d] = q.permute(0, 2, 1, 3)
        Kh = garbage(B, kv_bs, H, DK)
        Kh[:, :Nk] = 0
        Kh[:, :Nk, :, :d] = k.permute(0, 2, 1, 3)
        Q, K, q_col0, k_col0 = Qh.reshape(B * q_bs, H * DK).to(DEV), Kh.reshape(B * kv_bs, H * DK).to(DEV), 0, 0
    Vt = torch.zeros(H, DVP, B, kv_bs, dtype=torch.bfloat16)
    Vt[:, :d, :, :Nk] = v.permute(1, 3, 0, 2)
    Vt[:, :d, :, Nk:] = 1000.0                      # pad keys: masked by Nk, never read as zeros
    Vt = Vt.reshape(H * DVP, B * kv_bs).to(DEV)
    # output: a column slice of a wider buffer, rows above / below, the pad rows [Nq, q_bs) of every batch item guarded too
    og = Guarded(B * q_bs, H * d, torch.bfloat16, top=2, bottom=3, col0=8)
    rows_ok = torch.zeros(og.buf.shape[0], dtype=torch.bool, device=DEV)
    rows_ok[2:2 + B * q_bs] = (torch.arange(B * q_bs, device=DEV) % q_bs) < Nq
    og.exclude(rows_ok[:, None])
    scale = c["scale"] if c["scale"] is not None else d ** -0.5
    kv_len = torch.tensor(c["kv_len"], dtype=torch.int32, device=DEV) if c["kv_len"] is not None else None
    ops.attention(Q, K, Vt, og.view, B, H, Nq, Nk, d, scale=scale, q_col0=q_col0, k_col0=k_col0, causal=c["causal"],
                  q_bstride=q_bs, kv_bstride=kv_bs, kv_len=kv_len)
    torch.cuda.synchronize()
    assert_attention_path(c["path"], what)
    og.check(what)
    # fp64 reference with the scale the kernel sees (fp32)
    sc = float(torch.tensor(scale, dtype=torch.float32))
    q64, k64, v64 = (t.double().to(DEV) for t in (q, k, v))
    sim = torch.einsum("bhid,bhjd->bhij", q64, k64) * sc
    valid = torch.ones(B, 1, Nq, Nk, dtype=torch.bool, device=DEV)
    if c["kv_len"] is not None:
        nk_b = torch.tensor([min(max(n, 1), Nk) for n in c["kv_len"]], device=DEV)
        valid &= (torch.arange(Nk, device=DEV)[None, :] < nk_b[:, None])[:, None, None, :]
    if c["causal"]:
        valid &= torch.ones(Nq, Nk, dtype=torch.bool, device=DEV).tril()[None, None]
    p = sim.masked_fill(~valid, float("-inf")).softmax(-1)
    ref = torch.einsum("bhij,bhjd->bhid", p, v64)
    v1 = torch.einsum("bhij,bhjd->bhid", p, v64.abs())
    qk_abs = torch.einsum("bhid,bhjd->bhij", q64.abs(), k64.abs()).masked_fill(~valid, 0).amax(-1, keepdim=True)
    bound = 2.0 ** -8 * ref.abs() + 2.0 ** -7 * v1 + sc * d * 2.0 ** -23 * qk_abs * v1
    out = og.view.view(B, q_bs, H, d)[:, :Nq].permute(0, 2, 1, 3)
    assert_within(out, ref, bound, what)


# ---------------------------------------------------------------------------------------------------------------------------
# the path tables cover every kernel path
# ---------------------------------------------------------------------------------------------------------------------------
def test_path_tables_cover_every_kernel_path():
    """Every case above asserts the path it names (when no kernel switch is set), so the paths the tables name are the paths
    the suite reaches: GEMM / conv epilogue modes {generic, fast} x BN {64, 128, 160, 256} plus GEGLU (BN 256 only: its
    value / gate packing is per 256-column tile), a split-K launch per output type, and every default attention kernel."""
    seen = set()
    split_out = set()
    for p in GEMM_CASES + CONV_EDGE_CASES:
        c = p.values[0]
        path = c["path"]
        if "mode" in path and "bn" in path:
            seen.add((path["mode"], path["bn"]))
        if path.get("split", False) is True or (type(path.get("split")) is int and path["split"] > 1):
            split_out.add("f32" if c["f32"] else "bf16")
    want = {(m, bn) for m in ("generic", "fast") for bn in (64, 128, 160, 256)} | {("geglu", 256)}
    assert want <= seen, sorted(want - seen)
    assert split_out == {"f32", "bf16"}, split_out
    att = {p.values[0]["path"] for p in ATT_CASES}
    assert att >= {ATT_TWO_TILE, ATT_COLS64, ATT_COLS128, ATT_D80, ATT_D160, ATT_KEYLEN64, ATT_KEYLEN128}, sorted(att)


# ---------------------------------------------------------------------------------------------------------------------------
# small kernels: sizes off the block / vector width, more than one grid-stride pass (the grids are capped at 16 CTAs of 256
# threads per SM: > 606208 elements on 148 SMs)
# ---------------------------------------------------------------------------------------------------------------------------
N_BIG = 1_000_003


def _bits_equal(a, b, what):
    assert a.dtype == b.dtype and a.shape == b.shape, (what, a.dtype, b.dtype, a.shape, b.shape)
    ia = a.view(torch.int16 if a.dtype == torch.bfloat16 else torch.int32)
    ib = b.view(torch.int16 if b.dtype == torch.bfloat16 else torch.int32)
    bad = (ia != ib).sum().item()
    assert bad == 0, f"{what}: {bad} of {a.numel()} elements differ"


def test_patchify_bit_exact():
    B, Cin, HW, P, Kpad = 5, 3, 224, 14, 592          # 5 x 256 rows x 592 = 757760 elements
    px = rnd(B, Cin, HW, HW, seed=1, dtype=torch.float32)
    G_ = HW // P
    og = Guarded(B * G_ * G_, Kpad, torch.bfloat16, top=8, bottom=40, flat=True)
    _check(_lib().vdb_patchify(px.data_ptr(), B, Cin, HW, P, Kpad, og.view.data_ptr(), _stream()), "patchify")
    torch.cuda.synchronize()
    og.check("patchify")
    ref = px.view(B, Cin, G_, P, G_, P).permute(0, 2, 4, 1, 3, 5).reshape(B * G_ * G_, Cin * P * P)
    ref = F.pad(ref, (0, Kpad - Cin * P * P)).to(torch.bfloat16)
    _bits_equal(og.view, ref, "patchify")


def test_clip_text_embed_bit_exact():
    B, L, Lp, C, V = 12, 77, 80, 768, 1000            # 737280 elements; pad rows are zeros
    g = torch.Generator().manual_seed(3)
    tokens = torch.randint(0, V, (B, L), generator=g).to(DEV)
    tok, pos = rnd(V, C, seed=1, dtype=torch.float32), rnd(L, C, seed=2, dtype=torch.float32)
    og = Guarded(B * Lp, C, torch.bfloat16, top=8, bottom=24, flat=True)
    _check(_lib().vdb_clip_text_embed(tokens.data_ptr(), tok.data_ptr(), pos.data_ptr(), B, L, Lp, C, og.view.data_ptr(), _stream()),
           "clip_text_embed")
    torch.cuda.synchronize()
    og.check("clip_text_embed")
    ref = torch.zeros(B, Lp, C, dtype=torch.float32, device=DEV)
    ref[:, :L] = tok[tokens] + pos[None]
    _bits_equal(og.view.view(B, Lp, C), ref.to(torch.bfloat16), "clip_text_embed")


@pytest.mark.parametrize("scaled", [False, True])
def test_vit_assemble_bit_exact(scaled):
    B, L, Lp, C = 3, 257, 264, 1024                   # 811008 elements
    patches = rnd(B * (L - 1), C, seed=1)
    cls, pos = rnd(C, seed=2, dtype=torch.float32), rnd(L, C, seed=3, dtype=torch.float32)
    ts = (rnd(B, L, seed=4, dtype=torch.float32).abs() + 0.5) if scaled else None
    og = Guarded(B * Lp, C, torch.bfloat16, top=8, bottom=24, flat=True)
    _check(_lib().vdb_vit_assemble(patches.data_ptr(), cls.data_ptr(), pos.data_ptr(), ts.data_ptr() if scaled else None, B, L, Lp,
                                   C, og.view.data_ptr(), _stream()), "vit_assemble")
    torch.cuda.synchronize()
    og.check("vit_assemble")
    x = torch.cat([cls[None, None].expand(B, 1, C), patches.float().view(B, L - 1, C)], 1) + pos[None]
    if scaled:
        x = x * ts[:, :, None]
    ref = torch.zeros(B, Lp, C, dtype=torch.float32, device=DEV)
    ref[:, :L] = x
    _bits_equal(og.view.view(B, Lp, C), ref.to(torch.bfloat16), f"vit_assemble scaled={scaled}")


def test_token_embed_bit_exact():
    n, ldt, C, V, Pn, t, off = 37, 30, 768, 500, 64, 5, 1
    g = torch.Generator().manual_seed(4)
    tokens = torch.randint(0, V, (n, ldt), generator=g).to(torch.int32).to(DEV)
    step = torch.tensor([t], dtype=torch.int32, device=DEV)
    wte, wpe = rnd(V, C, seed=1), rnd(Pn, C, seed=2, dtype=torch.float32)
    emb = Guarded(n, C, torch.float32, col0=8).view        # row-strided emb_add
    emb.copy_(rnd(n, C, seed=3, dtype=torch.float32))
    og = Guarded(n, C, torch.bfloat16, col0=16)
    _check(_lib().vdb_token_embed(tokens.data_ptr(), ldt, step.data_ptr(), off, wte.data_ptr(), wpe.data_ptr(), emb.data_ptr(),
                                  emb.stride(0), n, C, og.view.data_ptr(), og.view.stride(0), _stream()), "token_embed")
    torch.cuda.synchronize()
    og.check("token_embed")
    ref = (wte[tokens[:, t].long()].float() + wpe[t + off][None]) + emb
    _bits_equal(og.view.contiguous(), ref.to(torch.bfloat16), "token_embed")


def _fp32_terms_bound(terms, roundings):
    """error of an fp32 evaluation of sum(terms) with `roundings` rounding steps: roundings * u * sum |term|"""
    return roundings * U * sum(t.abs() for t in terms)


def test_axpby():
    x, z = rnd(N_BIG, seed=1, dtype=torch.float32), rnd(N_BIG, seed=2, dtype=torch.float32)
    a, b = 0.8123456, -0.5831234
    og = Guarded(1, N_BIG, torch.float32, top=4, bottom=13, flat=True)
    _check(_lib().vdb_axpby_f32(x.data_ptr(), z.data_ptr(), a, b, og.view.data_ptr(), N_BIG, _stream()), "axpby")
    torch.cuda.synchronize()
    og.check("axpby")
    a32, b32 = (float(torch.tensor(v, dtype=torch.float32)) for v in (a, b))
    terms = [a32 * x.double(), b32 * z.double()]
    # at most 2 fp32 ulp of the term magnitudes: two products and one add, or an FMA-contracted product and the add
    assert_within(og.view[0], terms[0] + terms[1], _fp32_terms_bound(terms, 4), "axpby")


@pytest.mark.parametrize("nterms", [1, 2, 3, 4])
def test_lincomb4(nterms):
    xs = [rnd(N_BIG, seed=s, dtype=torch.float32) for s in range(nterms)]
    cs = [55 / 24, -59 / 24, 37 / 24, -9 / 24][:nterms]              # PLMS 4th-order coefficients
    og = Guarded(1, N_BIG, torch.float32, top=4, bottom=13, flat=True)
    ptrs = [t.data_ptr() for t in xs] + [None] * (4 - nterms)
    co = cs + [0.0] * (4 - nterms)
    _check(_lib().vdb_lincomb4_f32(ptrs[0], ptrs[1], ptrs[2], ptrs[3], co[0], co[1], co[2], co[3], og.view.data_ptr(), N_BIG,
                                   _stream()), "lincomb4")
    torch.cuda.synchronize()
    og.check("lincomb4")
    terms = [float(torch.tensor(c, dtype=torch.float32)) * x.double() for c, x in zip(cs, xs)]
    # 2 ulp (4 u) of the term magnitudes: one product, then one FMA-contracted step per further term (<= 4 roundings)
    assert_within(og.view[0], sum(terms), _fp32_terms_bound(terms, 4), f"lincomb4 {nterms} terms")


@pytest.mark.parametrize("cin,cout", [(1, 1), (3, 8), (4, 4), (8, 8), (8, 3)])
def test_pointwise_small(cin, cout):
    npix = 620_011
    x = rnd(npix, cin, seed=1, dtype=torch.float32)
    w = rnd(cout, cin, seed=2, dtype=torch.float32)
    b = rnd(cout, seed=3, dtype=torch.float32)
    pre = 1.0 / 0.18215
    og = Guarded(npix, cout, torch.float32, top=4, bottom=21, flat=True)
    _check(_lib().vdb_pointwise_small(x.data_ptr(), npix, cin, cout, w.data_ptr(), b.data_ptr(), pre, og.view.data_ptr(), _stream()),
           "pointwise_small")
    torch.cuda.synchronize()
    og.check("pointwise_small")
    pre32 = float(torch.tensor(pre, dtype=torch.float32))
    xin = x.double() * pre32
    terms = [b.double()[None, :].expand(npix, cout)] + [w.double()[None, :, c] * xin[:, c:c + 1] for c in range(cin)]
    # cin + 1 roundings reach an element: the x * pre_mul product and one per FMA-contracted accumulation step; for cin <= 3
    # this is the 2-ulp (4 u) bound, the 8-channel chain needs 9 u
    assert_within(og.view, sum(terms), _fp32_terms_bound(terms, max(4, cin + 1)), f"pointwise_small {cin}->{cout}")


@pytest.mark.parametrize("with_noise", [False, True])
def test_gaussian_sample(with_noise):
    npix, C = 160_001, 4                               # 640004 outputs
    mean = rnd(npix, C, seed=1, dtype=torch.float32)
    logvar = (torch.rand(npix, C, generator=torch.Generator().manual_seed(2)) * 70.0 - 40.0).to(DEV)   # [-40, 30]: both clamps
    mom = torch.cat([mean, logvar], 1).contiguous()
    noise = rnd(npix, C, seed=3, dtype=torch.float32) if with_noise else None
    post = 0.18215
    og = Guarded(npix, C, torch.float32, top=4, bottom=9, flat=True)
    _check(_lib().vdb_gaussian_sample(mom.data_ptr(), noise.data_ptr() if with_noise else None, C, npix, post, og.view.data_ptr(),
                                      _stream()), "gaussian_sample")
    torch.cuda.synchronize()
    og.check("gaussian_sample")
    post32 = float(torch.tensor(post, dtype=torch.float32))
    terms = [mean.double()]
    if with_noise:
        terms.append(torch.exp(0.5 * logvar.double().clamp(-30.0, 20.0)) * noise.double())
    ref = sum(terms) * post32
    # 4 ulp (8 u) of the term magnitudes: expf (<= 2 ulp), the noise product, the add and the post_mul product
    assert_within(og.view, ref, 8 * U * sum(t.abs() for t in terms) * post32, f"gaussian_sample noise={with_noise}")


def test_scale_by_row_norm():
    B, L, Lp, C = 5, 77, 80, 768
    z = rnd(B, Lp, C, seed=1)
    idx = torch.tensor([0, 76, 3, 40, 9], dtype=torch.int32, device=DEV)
    rs = rnd(B, L, seed=2, dtype=torch.float32).abs() + 0.25
    og = Guarded(B * L, C, torch.float32, top=4, bottom=9, flat=True)
    _check(_lib().vdb_scale_by_row_norm(z.data_ptr(), idx.data_ptr(), rs.data_ptr(), B, L, Lp, C, og.view.data_ptr(), _stream()),
           "scale_by_row_norm")
    torch.cuda.synchronize()
    og.check("scale_by_row_norm")
    z64 = z.double()
    nrm = z64[torch.arange(B, device=DEV), idx.long()].norm(dim=-1)
    ref = z64[:, :L] / nrm[:, None, None] * rs.double()[:, :, None]
    # 6 ulp (12 u) relative: the fp32 sum of C squares runs through a reduction of depth 16 (3 per thread, 5 shuffle levels,
    # 8 warps in sequence: <= 16 u relative, halved by the square root), then sqrtf, the reciprocal and two products
    assert_within(og.view.view(B, L, C), ref, 12 * U * ref.abs(), "scale_by_row_norm")


@pytest.mark.parametrize("act", [0, 1])
def test_affine_act_rows(act):
    rows, n = 2003, 328                                 # 82123 uint4 items: n / 8 = 41 per row
    x = rnd(rows, n, seed=1)
    gamma = rnd(n, seed=2, dtype=torch.float32) + 1.0
    beta = rnd(n, seed=3, dtype=torch.float32) * 0.5
    og = Guarded(rows, n, torch.bfloat16, top=8, bottom=24, flat=True)
    _check(_lib().vdb_affine_act_rows(x.data_ptr(), rows, n, gamma.data_ptr(), beta.data_ptr(), act, og.view.data_ptr(), _stream()),
           "affine_act_rows")
    torch.cuda.synchronize()
    og.check("affine_act_rows")
    h = x.double() * gamma.double() + beta.double()
    ref = F.silu(h) if act else h
    _, e = torch.frexp(ref)
    ulp = torch.ldexp(torch.ones_like(ref), e - 8)      # one bf16 ulp at |ref| (8 significant bits)
    bound = ulp
    if act:
        # SiLU = 0.5 h (1 + tanh.approx(h / 2)): the MUFU tanh's absolute error (< 2^-10.9) is carried by the 0.5 h factor
        bound = bound + 2.0 ** -10.9 * 0.5 * h.abs()
    assert_within(og.view, ref, bound, f"affine_act_rows act={act}")
