"""Opt-in kernel variants (environment switches read once per process) against the same kernel parity tests, each in its own
process.  Skipped unless VDB_TEST_VARIANTS=1: variants that have not been measured/validated on a B200 yet stay out of the
default GPU suite (the default kernels are covered by test_kernels_gpu.py / test_kernel_edges_gpu.py / test_parity_gpu.py)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

VARIANTS = [
    ({"VDB_ATT_BKV": "64"}, "attention"),          # 64-column kv tiles, double-buffered S / P           (validated, round 1)
    ({"VDB_ATT_BKV": "643"}, "attention"),         # three CTAs per SM                                     (validated, round 1)
    ({"VDB_ATT_BKV": "128"}, "attention"),         # the 128-column kernel for every context length        (validated, round 1)
    ({"VDB_GN_REG": "0"}, "groupnorm"),            # generic two-read single-launch GroupNorm              (validated, round 1)
    ({"VDB_GN_FUSED": "0"}, "groupnorm"),          # statistics + apply kernels                            (validated, round 1)
    ({"VDB_PAIR": "1"}, "gemm or conv3x3"),        # CTA pairs (cta_group::2)                              (validated, round 1)
    ({"VDB_NFAST": "2"}, "gemm or conv3x3"),       # N-fast tile order wherever it is legal                (validated, round 2: no gain)
    ({"VDB_IGEMM_SPEC": "0"}, "gemm or conv3x3"),  # generic epilogue only
    ({"VDB_EPI_TMA": "0"}, "gemm or conv3x3"),     # transposing epilogues instead of the TMA-store ones (round-1 default)
    ({"VDB_GN_BUNDLE": "0"}, "groupnorm"),         # single-launch pixel-range GroupNorm instead of the group-bundle kernel
    ({"VDB_LN_RG": "0"}, "layernorm"),             # warp-per-row LayerNorm instead of the row-group kernel
    ({"VDB_ATT_FA": "0"}, "attention"),            # column-split attention kernel for every shape (round-1 default)
    ({"VDB_ATT_ONES": "0"}, "attention"),          # two-tile kernel with the row sums on the softmax threads
    ({"VDB_CHUNKED": "1"}, "gemm or conv3x3"),     # contiguous tile range per CTA instead of the grid-strided walk (validated, round 2: neutral)
]

RUN = pytest.mark.skipif(os.environ.get("VDB_TEST_VARIANTS") != "1", reason="set VDB_TEST_VARIANTS=1 to run the opt-in kernel variants")


@RUN
@pytest.mark.parametrize("env,select", VARIANTS, ids=lambda v: "_".join(f"{k}={x}" for k, x in v.items()) if isinstance(v, dict) else None)
def test_variant(env, select):
    e = dict(os.environ, **env)
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "--timeout", "120",
                          os.path.join(ROOT, "tests", "test_kernels_gpu.py"), os.path.join(ROOT, "tests", "test_kernel_edges_gpu.py"),
                          "-k", select],
                         capture_output=True, text=True, env=e, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-1000:]


@RUN
def test_folded_upsample_conv_kernel():
    """conv modes 3..6 + interleave2x2 against torch's upsample + conv2d on the bf16-rounded operands."""
    import torch
    import torch.nn.functional as F
    sys.path.insert(0, os.path.join(ROOT, "versatile-diffusion_b200"))
    from lib.model_zoo.diffusion_utils import fold_upsample_conv3x3
    from vdb200 import ops
    for (B, H, W, C, N) in [(2, 16, 16, 64, 64), (8, 32, 32, 640, 640), (1, 24, 40, 128, 192)]:
        g = torch.Generator().manual_seed(H * 7 + C)
        x = torch.randn(B, H, W, C, generator=g).to(torch.bfloat16).cuda()
        w = (torch.randn(N, C, 3, 3, generator=g) * 0.05)
        b = torch.randn(N, generator=g).cuda()
        out = ops.upsample2x_conv3x3_folded(x, fold_upsample_conv3x3(w).cuda(), bias=b)
        ref = F.conv2d(F.interpolate(x.float().permute(0, 3, 1, 2), scale_factor=2, mode="nearest"),
                       w.to(torch.bfloat16).float().cuda(), b, padding=1).permute(0, 2, 3, 1)
        err = (out.float() - ref).abs().max().item()
        assert err <= 3e-2 * ref.abs().max().item(), (B, H, W, C, N, err)


@RUN
def test_folded_upsample_in_the_model_paths():
    """VDB_UPFOLD=2 forces the folded path in every Upsample of the UNet and the VAE: the path-level parity tests must hold."""
    e = dict(os.environ, VDB_UPFOLD="2")
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "--timeout", "300",
                          os.path.join(ROOT, "tests", "test_parity_gpu.py"), "-k", "apply_model or vae_decode or ddim_5"],
                         capture_output=True, text=True, env=e, timeout=1500, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-1000:]
