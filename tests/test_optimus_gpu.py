"""Optimus text decode on the B200: the KV-cache attention and sampler kernels against torch / numpy restatements, the tanh-GELU
GEMM epilogue, and the whole decode path (teacher-forced logits, greedy-limit sampling, graph == eager, seeding, the
inference_i2t shape) against the fp32 oracle of tests/optimus_oracle.py."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import optimus_oracle as oo

pytestmark = pytest.mark.gpu
DEV = "cuda"
VPAD = 50304


def _cmp(out, ref, cos_min=0.999, tol=3e-2, what=""):
    out, ref = out.float().cpu().flatten(), ref.float().cpu().flatten()
    assert torch.isfinite(out).all(), what
    cos = F.cosine_similarity(out, ref, dim=0).item()
    err, scale = (out - ref).abs().max().item(), ref.abs().max().item()
    print(f"[optimus] {what}: cos {cos:.6f} max|err| {err:.4g} / {scale:.4g}")
    assert cos >= cos_min and err <= tol * scale, (what, cos, err, scale)


def _decoder(mini, seed=oo.WEIGHT_SEED):
    from oracle import weights
    from lib.model_zoo.optimus import GPT2ForLatentConnector_XX
    cfg = oo.decoder_config(mini)
    net = GPT2ForLatentConnector_XX(cfg)
    sd = oo.synth_decoder_sd(weights.param_shapes(net), seed)
    net.load_state_dict(sd, strict=False)
    net.eval().to(DEV)
    return net, sd, cfg


@pytest.fixture(scope="module")
def mini():
    return _decoder(True)


@pytest.fixture(scope="module")
def full():
    return _decoder(False)


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("H", [2, 12])
@pytest.mark.parametrize("n", [1, 4, 16])
def test_kv_decode_attention_vs_torch(H, n):
    from vdb200 import ops
    g = torch.Generator().manual_seed(H * 100 + n)
    C = H * 64
    for t in (0, 1, 5, 17, 28, 29):                 # keys = t + 2: the memory slot and tokens 0..t
        qkv = torch.randn(n, 3 * C, generator=g).bfloat16()
        mem_all = torch.randn(n, 3 * C, generator=g).bfloat16()          # a layer's slot is a strided column range
        kc = torch.randn(n, H, 32, 64, generator=g).bfloat16()
        vc = torch.randn(n, H, 32, 64, generator=g).bfloat16()
        kd, vd, qd, md = kc.to(DEV), vc.to(DEV), qkv.to(DEV), mem_all.to(DEV)
        out = torch.empty(n, C, dtype=torch.bfloat16, device=DEV)
        step = torch.tensor([t], dtype=torch.int32, device=DEV)
        ops.kv_decode_attention(qd, md[:, C:2 * C], kd, vd, step, H, out)
        q, k, v = (x.float().reshape(n, H, 64) for x in qkv.split(C, dim=1))
        mem = mem_all[:, C:2 * C].float().reshape(n, H, 1, 64)
        K = torch.cat([mem, kc[:, :, :t].float(), k[:, :, None]], dim=2)
        V = torch.cat([mem, vc[:, :, :t].float(), v[:, :, None]], dim=2)
        w = torch.softmax((q[:, :, None] @ K.transpose(-1, -2)) / 8.0, dim=-1)
        ref = (w @ V).reshape(n, C)
        assert (out.float().cpu() - ref).abs().max().item() <= 2e-2 * ref.abs().max().item(), (t, H, n)
        assert torch.equal(kd[:, :, t].cpu(), k.bfloat16().reshape(n, H, 64)) and torch.equal(vd[:, :, t].cpu(), v.bfloat16().reshape(n, H, 64))
        assert torch.equal(kd[:, :, :t].cpu(), kc[:, :, :t])                 # earlier slots untouched


def _np_probs(logits_row, T):
    x = logits_row[:oo.VOCAB].astype(np.float32) / np.float32(T)
    e = np.exp(x.astype(np.float64) - x.max())
    return e / e.sum()


def test_sample_tokens_vs_numpy_inverse_cdf():
    """token for token on uniforms placed mid-interval (>= 1e-5 from any CDF boundary): temperature, the padded lm_head
    columns, finished rows, the forced <EOS> at length 30, and the next-step embedding"""
    from vdb200 import ops
    rng = np.random.RandomState(7)
    n, C = 16, 128
    logits = (rng.randn(n, VPAD) * 3).astype(np.float32)
    logits[:, oo.VOCAB:] = 1e4                                            # padding columns must never be read
    wte = torch.randn(VPAD, C).bfloat16()
    wpe = torch.randn(64, C)
    lemb = torch.randn(n, C)
    for T, t in ((1.0, 3), (0.6, 3), (1.3, 28)):
        u = np.zeros((n, 32), np.float32)
        want = []
        for r in range(n):
            p = _np_probs(logits[r], T)
            c = np.cumsum(p)
            cand = np.nonzero(p > 1e-4)[0]                                 # intervals wide enough for a 1e-5 margin
            i = int(cand[(37 * r) % len(cand)])
            u[r, t] = np.float32((c[i] - p[i] + c[i]) / 2)
            want.append(i)
        tokens = torch.full((n, 32), 7, dtype=torch.int32)
        tokens[1, t] = oo.EOS_ID                                           # row 1 already finished
        td = tokens.to(DEV)
        x = torch.empty(n, C, dtype=torch.bfloat16, device=DEV)
        ops.sample_tokens(torch.from_numpy(logits).to(DEV), oo.VOCAB, torch.tensor([t], dtype=torch.int32, device=DEV), td,
                          oo.EOS_ID, temperature=torch.tensor([T], device=DEV), uniforms=torch.from_numpy(u).to(DEV),
                          max_len=oo.MAX_LENGTH, wte=wte.to(DEV), wpe=wpe.to(DEV), emb_add=lemb.to(DEV), x_next=x)
        got = td[:, t + 1].cpu().tolist()
        exp = [oo.EOS_ID if (r == 1 or t + 2 >= oo.MAX_LENGTH) else want[r] for r in range(n)]
        assert got == exp, (T, t)
        ref_x = (wte[torch.tensor(got).long()].float() + wpe[t + 2] + lemb).bfloat16()
        assert torch.equal(x.cpu(), ref_x)


def test_sample_tokens_philox_chi_square():
    """uniform logits over a 64-token slice: the Philox draws fill the 64 bins evenly (chi-square, 63 dof, p = 0.001)"""
    from vdb200 import ops
    n, steps, ldt = 256, 60, 64
    logits = torch.full((n, VPAD), -1e30)
    logits[:, 1000:1064] = 0.5
    ld = logits.to(DEV)
    tokens = torch.zeros(n, ldt, dtype=torch.int32, device=DEV)
    step = torch.zeros(1, dtype=torch.int32, device=DEV)
    temp = torch.ones(1, device=DEV)
    seed = torch.tensor([0x1234_5678_9ABC], dtype=torch.int64, device=DEV)
    for _ in range(steps):
        ops.sample_tokens(ld, oo.VOCAB, step, tokens, oo.EOS_ID, temperature=temp, seed=seed, max_len=ldt)
        ops.add_int(step, 1)
    drawn = tokens[:, 1:steps + 1].cpu().flatten()
    assert int(drawn.min()) >= 1000 and int(drawn.max()) < 1064
    counts = torch.bincount(drawn - 1000, minlength=64).double()
    expect = drawn.numel() / 64
    chi2 = float(((counts - expect) ** 2 / expect).sum())
    print(f"[optimus] philox chi-square {chi2:.1f} (63 dof)")
    assert chi2 < 103.4


@pytest.mark.parametrize("M", [4, 8, 64])
@pytest.mark.parametrize("ksplit", [0, 1, 4])
def test_gemm_gelu_tanh_epilogue(M, ksplit):
    from vdb200 import ops
    g = torch.Generator().manual_seed(M + ksplit)
    K, N = 768, 3072
    a = torch.randn(M, K, generator=g).bfloat16()
    w = (torch.randn(N, K, generator=g) * K ** -0.5).bfloat16()
    b = torch.randn(N, generator=g) * 0.5
    for out_dtype in (torch.bfloat16, torch.float32):
        out = ops.gemm(a.to(DEV), w.to(DEV), bias=b.to(DEV), act=ops.ACT_GELU_TANH, out_dtype=out_dtype, ksplit=ksplit)
        ref = F.gelu(a.float() @ w.float().t() + b, approximate="tanh")
        tol = 1e-2 if out_dtype == torch.bfloat16 else 1e-4
        assert (out.float().cpu() - ref).abs().max().item() <= tol * ref.abs().max().item(), (M, ksplit, out_dtype)


# ------------------------------------------------------------------------------------------------ decode path
@pytest.mark.parametrize("size", ["mini", "full"])
def test_teacher_forced_logits_vs_oracle(size, request):
    net, sd, cfg = request.getfixturevalue(size)
    gi = oo.golden_inputs(size)
    got = net.logits_for(gi["z"].to(DEV), gi["tokens"])
    ref = oo.gpt2_text_logits(sd, gi["z"], gi["tokens"], cfg)
    assert got.shape == ref.shape
    _cmp(got, ref, what=f"{size} teacher-forced logits, 2 rows x 12 positions")


@pytest.mark.parametrize("size", ["mini", "full"])
def test_low_temperature_picks_the_oracle_maximum(size, request):
    net, sd, cfg = request.getfixturevalue(size)
    z = oo.golden_inputs(size)["z"]
    ids = net.sample_token_ids(z.to(DEV), temperature=0.01).cpu().long()
    ref = oo.gpt2_text_logits(sd, z, ids, cfg)
    tol = 0.03 * ref.abs().max().item()
    for r in range(ids.shape[0]):
        for k in range(1, oo.MAX_LENGTH - 1):
            tok = int(ids[r, k])
            assert ref[r, k - 1, tok] >= ref[r, k - 1].max() - tol, (r, k, tok)
            if tok == oo.EOS_ID:
                break


def test_graph_replay_equals_eager(mini):
    net, sd, cfg = mini
    gi = oo.golden_inputs("mini")
    z = torch.cat([gi["z"], gi["z"].flip(1)]).to(DEV)
    u = torch.from_numpy(np.concatenate([gi["uniforms"][:2]] * 2).astype(np.float32)).to(DEV)
    eager = net.sample_token_ids(z, 0.9, uniforms=u, use_graph=False).clone()
    graph = net.sample_token_ids(z, 0.9, uniforms=u, use_graph=True).clone()
    again = net.sample_token_ids(z, 0.9, uniforms=u, use_graph=True).clone()      # replay of the cached graph
    assert torch.equal(eager, graph) and torch.equal(graph, again)


def test_seeded_decode_is_reproducible(mini, tmp_path):
    from lib.model_zoo.optimus import optimus_vae_next, GPT2Detokenizer
    net, sd, cfg = mini
    vae = optimus_vae_next(decoder=net, tokenizer_decoder=GPT2Detokenizer(oo.synthetic_vocab(tmp_path / "v.json")))
    z = oo.golden_inputs("mini")["z"].to(DEV)
    runs = []
    for s in (100, 100, 101):
        torch.manual_seed(s)
        runs.append(vae.decode(z))
    assert runs[0] == runs[1] and runs[0] != runs[2]
    assert len(runs[0]) == 2 and all(isinstance(s, str) and s for s in runs[0])


def test_inference_i2t_shape(monkeypatch, tmp_path):
    """app.py's inference_i2t after the context: DDIMSampler.sample(shape=[4, 768]) on the text diffuser, then
    net.vae_decode(x, 'text') -> 4 sentences"""
    monkeypatch.setenv("VDB_TEXT_FLOWS", "1")
    monkeypatch.setenv("VDB_GPT2_VOCAB", oo.synthetic_vocab(tmp_path / "v.json"))
    from lib.cfg_helper import model_cfg_bank
    from lib.model_zoo import get_model
    from lib.model_zoo.ddim import DDIMSampler
    from oracle import weights
    cfg = model_cfg_bank()("vd_four_flow_v1-0")
    cfg.args.ctx_cfg_list = []
    for _, d in cfg.args.diffuser_cfg_list:
        d.args.update(dict(model_channels=64))
    cfg.args.vae_cfg_list = [v for v in cfg.args.vae_cfg_list if v[0] == "text"]
    cfg.args.vae_cfg_list[0][1].args.decoder.args.config.update(oo.decoder_config(True))
    net = get_model()(cfg, verbose=False)
    sd = weights.synth_state_dict(weights.param_shapes(net), seed=2)
    res = net.load_state_dict(sd, strict=False)
    assert all(k.split(".")[0] not in ("vae", "diffuser") or k.endswith((".attn.bias", "lm_head.weight"))
               for k in res.missing_keys), res.missing_keys
    net.eval()
    net.to(DEV)
    g = torch.Generator().manual_seed(9)
    c, u = torch.randn(4, 257, 768, generator=g) * 0.5, torch.zeros(4, 257, 768)
    torch.manual_seed(30)
    with torch.no_grad():
        x, _ = DDIMSampler(net).sample(
            steps=4, shape=[4, 768], x_info={"type": "text"},
            c_info={"type": "image", "conditioning": c.to(DEV), "unconditional_conditioning": u.to(DEV),
                    "unconditional_guidance_scale": 7.5}, verbose=False, eta=0.)
        sentences = net.vae_decode(x, which='text', temperature=1)
    assert isinstance(sentences, list) and len(sentences) == 4 and all(isinstance(s, str) for s in sentences)
    print("[optimus] i2t sentences:", sentences)
