"""ctypes loader for libvdb200.so; declares every symbol of include/vdb200.h."""
import ctypes as C
import os

# VDB200_LIB: load another build of the same library (debug builds with -DVDB_TIMELINE); default = the in-tree product build
LIB_PATH = os.environ.get("VDB200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libvdb200.so")


class VdbError(RuntimeError):
    pass


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(nvcc, sm_100a). vdb200 has no CPU / library fallback by design.")

lib = C.CDLL(LIB_PATH)

p, i, ll, f, sz = C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_size_t

SIGNATURES = {
    "vdb_version": (C.c_char_p, []),
    "vdb_last_error": (C.c_char_p, []),
    "vdb_launch_count": (ll, []),
    "vdb_reset_launch_count": (None, []),
    "vdb_num_sms": (i, []),
    "vdb_ddim_cfg_step": (i, [p, p, p, p, p, p, f, f, p, p, p, ll, p]),
    "vdb_axpby_f32": (i, [p, p, f, f, p, ll, p]),
    "vdb_add_int": (i, [p, i, p]),
    "vdb_lincomb4_f32": (i, [p, p, p, p, f, f, f, f, p, ll, p]),
    "vdb_gemm_bf16": (i, [p, ll, ll, ll, p, ll, ll, p, ll, ll, p, ll, ll, p, ll, p, ll, i, i, f, i, i, p, sz, p]),
    "vdb_gemm_ln_bf16": (i, [p, ll, ll, ll, p, ll, ll, p, p, ll, p, ll, i, p, ll, i, i, f, p, i, p, p, p, i, p]),
    "vdb_gemm_skinny_fits": (i, [i, ll]),
    "vdb_gemm_skinny_bf16": (i, [p, i, ll, ll, p, ll, ll, p, ll, ll, p, ll, p, ll, p, ll, i, p]),
    "vdb_conv3x3_bf16": (i, [p, i, i, i, i, i, p, i, ll, p, i, p, i, p, ll, p, ll, p, ll, i, i, i, i, p, sz, p]),
    "vdb_attention_dk_pad": (i, [i]),
    "vdb_attention_dv_pad": (i, [i]),
    "vdb_attention_bf16": (i, [p, ll, i, p, ll, i, p, ll, p, ll, i, i, i, i, i, i, i, f, i, p]),
    "vdb_groupnorm_nsplit": (i, [i, i]),
    "vdb_groupnorm_scratch_floats": (ll, [i, i]),
    "vdb_groupnorm_nhwc": (i, [p, i, p, i, i, i, i, p, p, f, i, p, p, p]),
    "vdb_layernorm": (i, [p, ll, i, p, p, f, p, p]),
    "vdb_upsample2x_nhwc": (i, [p, i, i, i, i, p, p]),
    "vdb_interleave2x2_nhwc": (i, [p, i, i, i, i, p, p]),
    "vdb_clip_to_u8_hwc": (i, [p, i, i, i, p, p]),
    "vdb_resample_h_u8": (i, [p, i, i, i, i, p, p, i, p, p]),
    "vdb_resample_v_crop_norm": (i, [p, i, i, i, p, p, i, i, i, i, C.POINTER(f), C.POINTER(f), p, p]),
    "vdb_im2col3x3_small": (i, [p, i, i, i, i, i, f, f, p, p]),
    "vdb_permute_f32": (i, [p, i, i, ll, i, f, f, i, p, p]),
    "vdb_gaussian_sample": (i, [p, p, i, ll, f, p, p]),
    "vdb_cast_f32_bf16": (i, [p, p, ll, p]),
    "vdb_cast_bf16_f32": (i, [p, p, ll, p]),
    "vdb_pointwise_small": (i, [p, ll, i, i, p, p, f, p, p]),
    "vdb_timestep_embedding": (i, [p, p, i, i, f, p, p]),
    "vdb_linear_small": (i, [p, i, i, p, i, p, i, i, p, p]),
    "vdb_softmax_rows": (i, [p, ll, i, ll, f, p, p]),
    "vdb_clip_text_embed": (i, [p, p, p, i, i, i, i, p, p]),
    "vdb_patchify": (i, [p, i, i, i, i, i, p, p]),
    "vdb_vit_assemble": (i, [p, p, p, p, i, i, i, i, p, p]),
    "vdb_scale_by_row_norm": (i, [p, p, p, i, i, i, i, p, p]),
    "vdb_affine_act_rows": (i, [p, ll, i, p, p, i, p, p]),
    "vdb_pack_conv_weight": (i, [p, i, i, i, i, p, ll, ll, p]),
    "vdb_pack_geglu": (i, [p, p, i, i, p, p, p]),
    "vdb_pad_heads": (i, [p, i, i, i, i, p, p]),
    "vdb_kv_decode_attention": (i, [p, ll, p, ll, p, p, p, i, i, f, p, ll, p]),
    "vdb_sample_tokens": (i, [p, ll, i, i, p, p, p, p, i, p, i, i, p, i, p, p, p, ll, i, p, ll, p]),
    "vdb_token_embed": (i, [p, i, p, i, p, p, p, ll, i, i, p, ll, p]),
    "vdb_attention_keylen_bf16": (i, [p, ll, i, p, ll, i, p, ll, p, ll, i, i, i, i, i, i, i, f, i, p, p]),
    "vdb_bert_embed_ln": (i, [p, i, i, p, i, p, i, p, p, p, f, i, p, p]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)  # AttributeError here == header/library mismatch: fail loudly
    _fn.restype = _res
    _fn.argtypes = _args


_TRACE = bool(os.environ.get("VDB_TRACE"))


def check(status: int, what: str = "") -> None:
    if _TRACE:  # debugging aid: name every launch and wait for it, so a hung kernel is identified
        import sys
        import torch
        print(f"[vdb] {what} ...", file=sys.stderr, flush=True)
        torch.cuda.synchronize()
        print(f"[vdb] {what} done", file=sys.stderr, flush=True)
    if status != 0:
        msg = lib.vdb_last_error().decode("utf-8", "replace")
        raise VdbError(f"vdb200 {what} failed with status {status}: {msg}")
