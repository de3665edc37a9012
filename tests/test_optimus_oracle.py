"""Optimus text decode, CPU side: the fp32 oracle (tests/optimus_oracle.py) against the fixtures made from the unmodified
reference (tools/make_optimus_golden.py) and, where the reference tree exists, against the reference itself; the GPT-2
detokenizer string for string; the config bank switch; the decoder's checkpoint keys."""
import gzip
import json
import os

import numpy as np
import pytest
import torch

import optimus_oracle as oo

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def detok(tmp_path_factory):
    """the reference tokenizer's cases and the vocabulary entries they use, written out as a vocabulary json"""
    with gzip.open(os.path.join(GOLD, "gpt2_detok.json.gz")) as fh:
        doc = json.load(fh)
    path = tmp_path_factory.mktemp("vocab") / "gpt2-vocab.json"
    path.write_text(json.dumps(doc["vocab"]))
    return str(path), doc["cases"]


def _mini_fixture():
    from oracle import weights
    from lib.model_zoo.optimus import GPT2ForLatentConnector_XX
    cfg = oo.decoder_config(True)
    net = GPT2ForLatentConnector_XX(cfg)
    sd = oo.synth_decoder_sd(weights.param_shapes(net))
    return cfg, sd, np.load(os.path.join(GOLD, "optimus_mini.npz")), oo.golden_inputs("mini")


def _seq(row):
    return [int(v) for v in row if v >= 0]


def test_oracle_logits_match_reference_fixture():
    cfg, sd, gold, gi = _mini_fixture()
    logits = oo.gpt2_text_logits(sd, gi["z"], gi["tokens"], cfg)
    got = logits[..., gold["cols"]].numpy()
    ref = gold["logits"]
    assert np.abs(got - ref).max() <= 2e-4 * np.abs(ref).max()
    lse = torch.logsumexp(logits, dim=-1).numpy()
    assert np.abs(lse - gold["lse"]).max() <= 2e-4 * np.abs(gold["lse"]).max()


@pytest.mark.parametrize("temperature", [1.0, 0.7])
def test_oracle_sequences_match_reference_fixture(temperature):
    cfg, sd, gold, gi = _mini_fixture()
    seqs = oo.optimus_sample(sd, gi["z"], gi["uniforms"], temperature, cfg)
    assert seqs == [_seq(r) for r in gold[f"seq_t{temperature}"]]
    assert all(len(s) <= oo.MAX_LENGTH and s[0] == oo.BOS_ID and s[-1] == oo.EOS_ID for s in seqs)


def test_oracle_stops_at_eos_draw():
    cfg, sd, gold, gi = _mini_fixture()
    k = int(gold["eos_step"])
    seq = oo.optimus_sample(sd, gi["z"][:1], gold["eos_uniforms"], 1.0, cfg)[0]
    assert seq == _seq(gold["seq_eos"][0])
    assert len(seq) == k + 2 and seq[-1] == oo.EOS_ID and oo.EOS_ID not in seq[:-1]


def test_top_p_one_filter_changes_no_draw():
    """The GPU sampler draws from the unfiltered softmax; at top_p = 1.0 the reference's filter only drops tokens whose fp32
    cumulative probability rounds above 1, which no golden draw reaches."""
    cfg, sd, gold, gi = _mini_fixture()
    for T in (1.0, 0.7):
        assert oo.optimus_sample(sd, gi["z"], gi["uniforms"], T, cfg, use_filter=False) == \
            oo.optimus_sample(sd, gi["z"], gi["uniforms"], T, cfg, use_filter=True)


def test_oracle_against_live_reference():
    """the reference imports its own `lib` package, so it runs in a child process (tools/make_optimus_golden.py --check)"""
    import subprocess
    import sys
    from oracle import ref_shims
    if not ref_shims.available():
        pytest.skip("reference tree not present")
    tool = os.path.join(os.path.dirname(GOLD), "..", "tools", "make_optimus_golden.py")
    r = subprocess.run([sys.executable, tool, "--check"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "oracle matches the reference" in r.stdout, r.stdout + r.stderr


def test_detokenizer_matches_reference_strings(detok):
    from lib.model_zoo.optimus import GPT2Detokenizer
    vocab_json, cases = detok
    dt = GPT2Detokenizer(vocab_file=vocab_json)
    assert len(cases) >= 200
    for c in cases:
        assert dt.decode(c["ids"]) == c["decoded"], c["ids"]
        assert dt.sentence(c["ids"]) == c["sentence"], c["ids"]
    assert dt.decode([oo.BOS_ID, 15496, 11, 995, 13, oo.EOS_ID]) == " <BOS>Hello, world. <EOS>"


def test_detokenizer_missing_vocab_is_a_clear_error(monkeypatch, tmp_path, detok):
    from lib.model_zoo.optimus import GPT2Detokenizer
    monkeypatch.delenv("VDB_GPT2_VOCAB", raising=False)
    with pytest.raises(RuntimeError, match="VDB_GPT2_VOCAB"):
        GPT2Detokenizer(vocab_file=str(tmp_path / "nope.json")).decode([1])
    monkeypatch.setenv("VDB_GPT2_VOCAB", detok[0])
    assert GPT2Detokenizer(vocab_file=str(tmp_path / "nope.json")).decode([15496]) == "Hello"


def test_text_vae_in_bank_only_with_text_flows(monkeypatch):
    from lib.cfg_helper import model_cfg_bank
    bank = model_cfg_bank()
    monkeypatch.delenv("VDB_TEXT_FLOWS", raising=False)
    with pytest.raises(KeyError):
        bank("optimus_v1")
    assert [n for n, _ in bank("vd_four_flow_v1-0").args.vae_cfg_list] == ["image"]
    monkeypatch.setenv("VDB_TEXT_FLOWS", "1")
    cfg = bank("optimus_v1")
    assert cfg.type == "optimus_vae_next" and cfg.args.decoder.type == "optimus_gpt2_connector"
    c = cfg.args.decoder.args.config
    assert (c.n_embd, c.n_head, c.n_layer, c.vocab_size, c.latent_size, c.layer_norm_epsilon) == (768, 12, 12, 50260, 768, 1e-5)
    assert cfg.args.tokenizer_decoder.args.vocab_file == "lib/model_zoo/optimus_models/vocab/gpt2-vocab.json"
    assert [n for n, _ in bank("vd_four_flow_v1-0").args.vae_cfg_list] == ["image", "text"]


@pytest.mark.parametrize("size", ["mini", "full"])
def test_decoder_keys_match_reference(size):
    from lib.model_zoo.optimus import optimus_vae_next, GPT2ForLatentConnector_XX, GPT2Detokenizer
    vae = optimus_vae_next(decoder=GPT2ForLatentConnector_XX(oo.decoder_config(size == "mini")),
                           tokenizer_decoder=GPT2Detokenizer())
    keys = {k: list(v.shape) for k, v in vae.state_dict().items()}
    assert keys == json.load(open(os.path.join(GOLD, f"keys_optimus_{size}.json")))
    assert vae.decoder.lm_head.weight is vae.decoder.transformer.wte.weight
    with pytest.raises(NotImplementedError, match="not built"):
        vae.encode(["a sentence"])


def test_decoder_builds_through_registry(monkeypatch):
    monkeypatch.setenv("VDB_TEXT_FLOWS", "1")
    from lib.cfg_helper import model_cfg_bank
    from lib.model_zoo.common.get_model import get_model
    cfg = model_cfg_bank()("optimus_v1")
    cfg.args.decoder.args.config.update(oo.decoder_config(True))
    vae = get_model()(cfg, verbose=False)
    assert type(vae).__name__ == "optimus_vae_next"
    assert {k: list(v.shape) for k, v in vae.state_dict().items()} == json.load(open(os.path.join(GOLD, "keys_optimus_mini.json")))
