"""Optimus text encode on the B200: the BERT embedding kernel, attention with per-sentence key counts and the tanh GEMM epilogue
against torch restatements, and the whole encode (mini and full size) against the fp32 oracle of tests/bert_oracle.py and the
reference's own z; then the flows a text VAE user runs on the latent: round trip, interpolation, ctx_encode('vae_text') and the
text-latent DDIM started from an encoded sentence."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import bert_oracle as bo
import optimus_oracle as oo

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _cmp(out, ref, cos_min=0.999, tol=3e-2, what=""):
    out, ref = out.float().cpu().flatten(), ref.float().cpu().flatten()
    assert torch.isfinite(out).all(), what
    cos = F.cosine_similarity(out, ref, dim=0).item()
    err, scale = (out - ref).abs().max().item(), ref.abs().max().item()
    print(f"[bert] {what}: cos {cos:.6f} max|err| {err:.4g} / {scale:.4g}")
    assert cos >= cos_min and err <= tol * scale, (what, cos, err, scale)


def _vae(mini, vocab):
    from lib.model_zoo.optimus import BertForLatentConnector_XX, BertTokenizer
    from lib.model_zoo.optimus import optimus_vae_next, GPT2ForLatentConnector_XX, GPT2Detokenizer
    cfg = bo.encoder_config(mini)
    enc = BertForLatentConnector_XX(cfg, latent_size=768)
    sd = bo.synth_encoder_sd(bo.encoder_shapes(cfg))
    enc.load_state_dict(sd, strict=True)
    vae = optimus_vae_next(encoder=enc, decoder=GPT2ForLatentConnector_XX(oo.decoder_config(True)),
                           tokenizer_encoder=BertTokenizer(vocab_file=vocab), tokenizer_decoder=GPT2Detokenizer())
    vae.eval().to(DEV)
    return vae, sd, cfg


@pytest.fixture(scope="module")
def vocab(tmp_path_factory):
    return bo.write_vocab(tmp_path_factory.mktemp("vocab") / "bert-vocab.txt")


@pytest.fixture(scope="module")
def mini(vocab):
    return _vae(True, vocab)


@pytest.fixture(scope="module")
def gold():
    import os
    return np.load(os.path.join(bo.ROOT, "tests", "golden", "bert_mini.npz"))


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("C", [128, 768])
@pytest.mark.parametrize("L", [2, 79])
def test_bert_embed_ln_vs_torch(C, L):
    from vdb200 import ops
    g = torch.Generator().manual_seed(C + L)
    n, V, P = 3, 1000, 512
    word, pos, typ = torch.randn(V, C, generator=g) * 0.5, torch.randn(P, C, generator=g) * 0.5, torch.randn(2, C, generator=g)
    gamma, beta = 1 + 0.1 * torch.randn(C, generator=g), 0.1 * torch.randn(C, generator=g)
    ids = torch.randint(0, V, (n, L), generator=g, dtype=torch.int32)
    ids[1, L // 2:] = 0                                                   # padding rows are embedded like any token
    out = ops.bert_embed_ln(ids.to(DEV), word.to(DEV), pos.to(DEV), typ[0].to(DEV), gamma.to(DEV), beta.to(DEV), eps=1e-12)
    ref = F.layer_norm(word[ids.long()] + pos[:L][None] + typ[0], (C,), gamma, beta, 1e-12).reshape(n * L, C)
    assert out.shape == (n * L, C) and out.dtype == torch.bfloat16
    assert (out.float().cpu() - ref).abs().max().item() <= 8e-3 * ref.abs().max().item()


def _attention_case(H, lens, Lp, seed):
    g = torch.Generator().manual_seed(seed)
    B, C = len(lens), H * 64
    qk = torch.randn(B * Lp, 2 * C, generator=g).bfloat16()
    vt = torch.randn(C, B * Lp, generator=g).bfloat16()
    return B, C, qk, vt


@pytest.mark.parametrize("H", [2, 12])
@pytest.mark.parametrize("Nk,lens", [(80, (1, 2, 7, 8, 79, 80)), (40, (1, 2, 7, 8, 39, 40))])
def test_attention_keylen_vs_torch_masked_softmax(H, Nk, lens):
    from vdb200 import ops
    Lp = (Nk + 7) // 8 * 8
    B, C, qk, vt = _attention_case(H, lens, Lp, H * 1000 + Nk)
    kv_len = torch.tensor(lens, dtype=torch.int32, device=DEV)
    out = torch.zeros(B * Lp, C, dtype=torch.bfloat16, device=DEV)
    ops.attention(qk.to(DEV), qk.to(DEV), vt.to(DEV), out, B, H, Nk, Nk, 64, q_col0=0, k_col0=C, q_bstride=Lp,
                  kv_bstride=Lp, kv_len=kv_len)
    out = out.float().cpu()
    for b, n in enumerate(lens):
        rows = slice(b * Lp, b * Lp + Nk)
        q = qk[rows, :C].float().reshape(Nk, H, 64).transpose(0, 1)
        k = qk[rows, C:].float().reshape(Nk, H, 64).transpose(0, 1)
        v = vt[:, b * Lp:b * Lp + Nk].float().reshape(H, 64, Nk).transpose(1, 2)
        s = q @ k.transpose(-1, -2) / 8.0
        s[:, :, n:] = -float("inf")
        ref = (torch.softmax(s, dim=-1) @ v).transpose(0, 1).reshape(Nk, C)
        assert (out[rows] - ref).abs().max().item() <= 2e-2 * ref.abs().max().item(), (H, Nk, n)


@pytest.mark.parametrize("H", [2, 12])
@pytest.mark.parametrize("Nk", [40, 80])
def test_attention_keylen_all_full_equals_plain_attention(H, Nk):
    from vdb200 import ops
    Lp = (Nk + 7) // 8 * 8
    B, C, qk, vt = _attention_case(H, (Nk,) * 4, Lp, H + Nk)
    qd, vd = qk.to(DEV), vt.to(DEV)
    a = torch.zeros(B * Lp, C, dtype=torch.bfloat16, device=DEV)
    b = torch.zeros(B * Lp, C, dtype=torch.bfloat16, device=DEV)
    ops.attention(qd, qd, vd, a, B, H, Nk, Nk, 64, q_col0=0, k_col0=C, q_bstride=Lp, kv_bstride=Lp)
    ops.attention(qd, qd, vd, b, B, H, Nk, Nk, 64, q_col0=0, k_col0=C, q_bstride=Lp, kv_bstride=Lp,
                  kv_len=torch.full((B,), Nk, dtype=torch.int32, device=DEV))
    assert torch.equal(a, b)


@pytest.mark.parametrize("M", [4, 64])
@pytest.mark.parametrize("ksplit", [0, 1, 4])
def test_gemm_tanh_epilogue(M, ksplit):
    from vdb200 import ops
    g = torch.Generator().manual_seed(M * 10 + ksplit)
    K, N = 768, 768
    a = torch.randn(M, K, generator=g).bfloat16()
    w = (torch.randn(N, K, generator=g) * K ** -0.5).bfloat16()
    b = torch.randn(N, generator=g) * 0.5
    for out_dtype in (torch.bfloat16, torch.float32):
        out = ops.gemm(a.to(DEV), w.to(DEV), bias=b.to(DEV), act=ops.ACT_TANH, out_dtype=out_dtype, ksplit=ksplit)
        ref = torch.tanh(a.float() @ w.float().t() + b)
        tol = 1e-2 if out_dtype == torch.bfloat16 else 1e-4
        assert (out.float().cpu() - ref).abs().max().item() <= tol, (M, ksplit, out_dtype)


# ------------------------------------------------------------------------------------------------ encode
def test_mini_encode_vs_oracle_and_reference(mini, gold):
    from vdb200 import ops
    vae, sd, cfg = mini
    sents = bo.golden_sentences()
    rows = vae.tokenizer_encoder.encode_sentences(sents)
    ids = bo.pad_ids(rows)
    assert np.array_equal(ids.numpy(), gold["ids"])
    n0 = ops.launch_count()
    z = vae.encode(sents)
    launches = ops.launch_count() - n0
    assert z.is_cuda and z.dtype == torch.float32 and z.shape == (len(sents), 768)
    L = cfg["num_hidden_layers"]
    print(f"[bert] mini encode: {launches} launches")
    assert 8 * L + 3 <= launches <= 13 * L + 5, launches     # 8 per layer + embedding, pooler, mean head; split-K adds reductions
    _cmp(z, bo.bert_encode(sd, ids, cfg)[1], what="mini encode vs oracle")
    _cmp(z, torch.from_numpy(gold["z"]), what="mini encode vs reference z")


def test_full_encode_vs_oracle_and_reference(vocab, gold):
    vae, sd, cfg = _vae(False, vocab)
    sents = bo.full_sentences()
    ids = bo.pad_ids(vae.tokenizer_encoder.encode_sentences(sents))
    assert np.array_equal(ids.numpy(), gold["full_ids"])
    z = vae.encode(sents)
    _cmp(z, bo.bert_encode(sd, ids, cfg)[1], what="full encode vs oracle")
    _cmp(z, torch.from_numpy(gold["full_z"]), what="full encode vs reference z")


def test_padding_does_not_leak(mini):
    """a sentence's z alone equals its z in a batch padded to a longer sentence"""
    vae, sd, cfg = mini
    sents = bo.golden_sentences()
    batch = vae.encode(sents)
    for i, s in enumerate(sents):
        _cmp(vae.encode([s])[0], batch[i], what=f"sentence {i} alone vs in the batch")


# ------------------------------------------------------------------------------------------------ flows on the text latent
@pytest.fixture(scope="module")
def net(vocab, tmp_path_factory):
    mp = pytest.MonkeyPatch()
    mp.setenv("VDB_TEXT_FLOWS", "1")
    mp.setenv("VDB_TEXT_ENCODER", "1")
    mp.setenv("VDB_BERT_VOCAB", vocab)
    mp.setenv("VDB_GPT2_VOCAB", oo.synthetic_vocab(tmp_path_factory.mktemp("gpt2") / "v.json"))
    from lib.cfg_helper import model_cfg_bank
    from lib.model_zoo import get_model
    from oracle import weights
    cfg = model_cfg_bank()("vd_four_flow_v1-0")
    cfg.args.ctx_cfg_list = []
    for _, d in cfg.args.diffuser_cfg_list:
        d.args.update(dict(model_channels=64))
    cfg.args.vae_cfg_list = [v for v in cfg.args.vae_cfg_list if v[0] == "text"]
    cfg.args.vae_cfg_list[0][1].args.decoder.args.config.update(oo.decoder_config(True))
    cfg.args.vae_cfg_list[0][1].args.encoder.args.config.update(bo.encoder_config(True))
    m = get_model()(cfg, verbose=False)
    sd = weights.synth_state_dict(weights.param_shapes(m), seed=2)
    res = m.load_state_dict(sd, strict=False)
    assert not [k for k in res.missing_keys if k.startswith("vae.text.encoder.")], res.missing_keys
    m.eval()
    m.to(DEV)
    yield m, sd
    mp.undo()


def test_ctx_encode_vae_text_equals_vae_encode(net):
    m, _ = net
    sents = ["a man rides a horse on the beach.", "two words"]
    a = m.vae_encode(sents, which="text")
    b = m.ctx_encode(sents, which="vae_text")
    assert a.shape == (2, 768) and torch.equal(a, b)


def test_round_trip_and_interpolation_decode_to_strings(net):
    m, _ = net
    z = m.vae_encode(["a man rides a horse on the beach.", "the quick brown fox jumps over the lazy dog"], which="text")
    torch.manual_seed(3)
    back = m.vae_decode(z, which="text")
    mix = torch.stack([(1 - w) * z[0] + w * z[1] for w in (0.0, 0.25, 0.5, 0.75, 1.0)])
    inter = m.vae_decode(mix, which="text")
    assert len(back) == 2 and len(inter) == 5 and all(isinstance(s, str) for s in back + inter)
    print("[bert] round trip:", back, "interpolation:", inter)


def test_text_x0_start_vs_oracle(net):
    """inference_i2i's start on a text latent: vae_encode -> q_sample at ddim_timesteps[k] -> exactly the first k DDIM steps,
    against the same composition of the oracle's encoder, q_sample and text-latent DDIM step; then decode to strings"""
    from lib.model_zoo.ddim import DDIMSampler
    from oracle import vd_oracle as O
    m, sd = net
    sents = ["a man rides a horse on the beach.", "", "two words"]
    n, steps, k, scale = len(sents), 8, 5, 7.5
    g = torch.Generator().manual_seed(21)
    noise = torch.randn(n, 768, generator=g)
    c, u = torch.randn(n, 257, 768, generator=g) * 0.5, torch.zeros(n, 257, 768)
    z = m.vae_encode(sents, which="text")
    orig = m.q_sample
    m.q_sample = lambda x_start, t, noise_=None: orig(x_start, t, noise=noise.to(x_start.device))   # inject the draw
    try:
        with torch.no_grad():
            x, inter = DDIMSampler(m).sample(
                steps=steps, shape=[n, 768], x_info={"type": "text", "x0": z, "x0_forward_timesteps": k},
                c_info={"type": "image", "conditioning": c.to(DEV), "unconditional_conditioning": u.to(DEV),
                        "unconditional_guidance_scale": scale}, verbose=False, eta=0., log_every_t=1)
    finally:
        m.q_sample = orig
    assert len(inter["pred_x0"]) == k, "the text x0 start walks exactly x0_forward_timesteps steps"
    esd = {kk[len("vae.text.encoder."):]: v for kk, v in sd.items() if kk.startswith("vae.text.encoder.")}
    ecfg = bo.encoder_config(True)
    zr = bo.bert_encode(esd, bo.pad_ids(m.vae["text"].tokenizer_encoder.encode_sentences(sents)), ecfg)[1]
    _cmp(z, zr, what="net.vae_encode(x, 'text') vs oracle")
    sched = O.ddim_schedule(O.ddpm_schedule(1000)["alphas_cumprod"], steps)
    ts = sched["timesteps"]
    xr = O.q_sample(zr, torch.full((n,), int(ts[k]), dtype=torch.long), noise)
    for i, step in enumerate(np.flip(ts[:k])):
        index = k - i - 1
        t = torch.full((n,), int(step), dtype=torch.long)
        e_u, e_c = O.apply_model_text(sd, torch.cat([xr, xr]), torch.cat([t, t]), [torch.cat([u, c])], c_types=("image",),
                                      model_channels=64).chunk(2)
        e = e_u + scale * (e_c - e_u)
        a_t, a_prev = float(sched["alphas"][index]), float(sched["alphas_prev"][index])
        pred_x0 = (xr - float(sched["sqrt_one_minus_alphas"][index]) * e) / a_t ** 0.5
        xr = a_prev ** 0.5 * pred_x0 + (1.0 - a_prev) ** 0.5 * e
    _cmp(x, xr, cos_min=0.995, tol=0.1, what=f"text x0 start, {k} of {steps} DDIM steps vs oracle")
    out = m.vae_decode(x, which="text")
    assert isinstance(out, list) and len(out) == n and all(isinstance(s, str) for s in out)
