"""model_cfg_bank for the hot-path models (reference lib/cfg_helper.py:102-146 + configs/model/*.yaml).

The reference resolves YAML with `super_cfg` inheritance and MODEL(name) indirection; the values below
are the resolved results for the shipped configs (configs/model/{vd,openai_unet,autokl,clip}.yaml).
By default 'vd_four_flow_v1-0' carries the image VAE, both CLIP context encoders, the 2D diffuser and the 0D diffuser's
context blocks.  VDB_TEXT_FLOWS=1 adds what the text-latent flows (i2t / t2t) need: the 0D diffuser's data blocks and the
Optimus text VAE's decoder (configs/model/optimus.yaml), registered as vae['text']; VDB_TEXT_ENCODER=1 on top of it adds the
text VAE's BERT encoder (vae_encode(x, 'text')).
"""
import copy
import os


class CfgDict(dict):
    """attribute dict (the reference uses easydict.EasyDict)"""

    def __init__(self, d=None, **kw):
        super().__init__()
        d = dict(d or {}); d.update(kw)
        for k, v in d.items():
            self[k] = v

    @staticmethod
    def _wrap(v):
        if isinstance(v, dict) and not isinstance(v, CfgDict):
            return CfgDict(v)
        if isinstance(v, (list, tuple)):
            return type(v)(CfgDict._wrap(x) for x in v)
        return v

    def __setitem__(self, k, v):
        super().__setitem__(k, CfgDict._wrap(v))

    def __setattr__(self, k, v):
        self[k] = v

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k)

    def __delattr__(self, k):
        del self[k]

    def update(self, e=None, **f):
        d = dict(e or {}); d.update(f)
        for k, v in d.items():
            self[k] = v

    def __deepcopy__(self, memo):
        return CfgDict({k: copy.deepcopy(v, memo) for k, v in self.items()})


def _unet2d(parts):
    return dict(type="openai_unet_2d_next", args=dict(
        in_channels=4, out_channels=4, model_channels=320, attention_resolutions=[4, 2, 1],
        num_res_blocks=[2, 2, 2, 2], channel_mult=[1, 2, 4, 4], num_heads=8, context_dim=768,
        use_checkpoint=True, parts=parts))


def _unet0d(parts):
    return dict(type="openai_unet_0d_next", args=dict(
        input_channels=768, model_channels=320, output_channels=768, num_noattn_blocks=[2, 2, 2, 2],
        channel_mult=[1, 2, 4, 4], second_dim=[4, 4, 4, 4], with_attn=[True, True, True, False], num_heads=8,
        context_dim=768, use_checkpoint=True, parts=parts))


_PARTS = {"": ["global", "data", "context"], "_g": ["global"], "_d": ["data"], "_c": ["context"],
          "_gd": ["global", "data"], "_gc": ["global", "context"], "_dc": ["data", "context"]}

_BANK = {
    "autokl_v1": dict(symbol="autokl", find_unused_parameters=False, type="autoencoderkl", args=dict(
        embed_dim=4, lossconfig=None, ddconfig=dict(
            double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128, ch_mult=[1, 2, 4, 4],
            num_res_blocks=2, attn_resolutions=[], dropout=0.0))),
    "clip_text_context_encoder": dict(symbol="clip", type="clip_text_context_encoder", args={}),
    "clip_image_context_encoder": dict(symbol="clip", type="clip_image_context_encoder", args={}),
    "vd_base": dict(symbol="vd", find_unused_parameters=True, type="vd_v2_0", args=dict(
        beta_linear_start=0.00085, beta_linear_end=0.012, timesteps=1000, use_ema=False)),
}
# configs/model/optimus.yaml:7-41, 43-90, 96-102 with MODEL(...) resolved, without the training-only fields (dropouts, summary
# heads, the MLM head's settings); optimus_v1 carries the BERT encoder only with VDB_TEXT_ENCODER=1 (no app.py flow encodes text)
_TEXT_BANK = {
    "optimus_bert_encoder": dict(symbol="optimus", find_unused_parameters=False, type="optimus_bert_connector", args=dict(
        config=dict(hidden_act="gelu", hidden_size=768, initializer_range=0.02, intermediate_size=3072, layer_norm_eps=1e-12,
                    max_position_embeddings=512, num_attention_heads=12, num_hidden_layers=12, type_vocab_size=2,
                    vocab_size=28996),
        latent_size=768)),
    "optimus_bert_tokenizer": dict(symbol="optimus", find_unused_parameters=False, type="optimus_bert_tokenizer", args=dict(
        do_lower_case=False, max_len=512, vocab_file="lib/model_zoo/optimus_models/vocab/bert-base-cased-vocab.txt")),
    "optimus_gpt2_decoder": dict(symbol="optimus", find_unused_parameters=False, type="optimus_gpt2_connector", args=dict(
        config=dict(hidden_size=768, initializer_range=0.02, latent_size=768, layer_norm_epsilon=1e-05,
                    max_position_embeddings=1024, n_ctx=1024, n_embd=768, n_head=12, n_layer=12, n_positions=1024,
                    num_attention_heads=12, num_hidden_layers=12, vocab_size=50260))),
    "optimus_gpt2_tokenizer": dict(symbol="optimus", find_unused_parameters=False, type="optimus_gpt2_tokenizer", args=dict(
        do_lower_case=False, max_len=1024, vocab_file="lib/model_zoo/optimus_models/vocab/gpt2-vocab.json",
        merges_file="lib/model_zoo/optimus_models/vocab/gpt2-merges.txt")),
}
_TEXT_BANK["optimus_v1"] = dict(symbol="optimus", find_unused_parameters=False, type="optimus_vae_next", args=dict(
    decoder=_TEXT_BANK["optimus_gpt2_decoder"], tokenizer_decoder=_TEXT_BANK["optimus_gpt2_tokenizer"],
    args=dict(latent_size=768)))


def _text_flows():
    return os.environ.get("VDB_TEXT_FLOWS") == "1"


def _text_encoder():
    """VDB_TEXT_ENCODER=1 (together with VDB_TEXT_FLOWS=1): vae['text'] also builds the BERT encoder behind
    vae_encode(x, 'text') / ctx_encode(x, 'vae_text') (+108 M parameters the i2t / t2t flows do not use)"""
    return os.environ.get("VDB_TEXT_ENCODER") == "1"


for _sfx, _parts in _PARTS.items():
    _BANK["openai_unet_2d_v1" + _sfx] = _unet2d(_parts)
    _BANK["openai_unet_0d_v1" + _sfx] = _unet0d(_parts)


class model_cfg_bank(object):
    def __call__(self, name):
        if name == "vd_four_flow_v1-0":
            cfg = CfgDict(copy.deepcopy(_BANK["vd_base"]))
            vaes = [["image", self("autokl_v1")]] + ([["text", self("optimus_v1")]] if _text_flows() else [])
            cfg.args.update(dict(
                vae_cfg_list=vaes,
                ctx_cfg_list=[["image", self("clip_image_context_encoder")], ["text", self("clip_text_context_encoder")]],
                # the 0D (text-latent) diffuser contributes only its context blocks to image sampling; VDB_TEXT_FLOWS=1 builds its
                # data blocks too (the reference's 'openai_unet_0d_v1_dc': +1.7 G parameters) for the i2t / t2t diffusion
                diffuser_cfg_list=[["image", self("openai_unet_2d_v1")],
                                   ["text", self("openai_unet_0d_v1_dc" if _text_flows() else "openai_unet_0d_v1_c")]],
                global_layer_ptr="image", latent_scale_factor={"image": 0.18215}))
            return cfg
        if _text_flows() and name in _TEXT_BANK:
            cfg = CfgDict(copy.deepcopy(_TEXT_BANK[name]))
            if name == "optimus_v1" and _text_encoder():
                cfg.args.update(dict(encoder=self("optimus_bert_encoder"), tokenizer_encoder=self("optimus_bert_tokenizer")))
            return cfg
        if name not in _BANK:
            raise KeyError(f"config '{name}' is outside the B200 hot-path build (have: {sorted(_BANK)} + vd_four_flow_v1-0; "
                           "VDB_TEXT_FLOWS=1 adds the Optimus text VAE)")
        return CfgDict(copy.deepcopy(_BANK[name]))
