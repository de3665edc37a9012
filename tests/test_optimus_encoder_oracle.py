"""Optimus text encode, CPU side: the fp32 oracle (tests/bert_oracle.py) against the fixtures made from the unmodified reference
(tools/make_bert_golden.py) and, where the reference tree exists, against the reference itself; the BERT tokenizer id for id;
the VDB_TEXT_ENCODER config switch; the encoder's checkpoint keys; the host-side checks of the new C ABI entries."""
import json
import os

import numpy as np
import pytest
import torch

import bert_oracle as bo
import optimus_oracle as oo

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def tok(tmp_path_factory):
    """the reference tokenizer's cases and a vocabulary file made of the entries the fixtures use"""
    return bo.write_vocab(tmp_path_factory.mktemp("vocab") / "bert-vocab.txt"), bo.tokenizer_cases()["cases"]


def _mini():
    cfg = bo.encoder_config(True)
    sd = bo.synth_encoder_sd(bo.encoder_shapes(cfg))
    return cfg, sd, np.load(os.path.join(GOLD, "bert_mini.npz"))


def test_oracle_matches_reference_fixture():
    cfg, sd, gold = _mini()
    ids = torch.from_numpy(gold["ids"]).long()
    assert ids.shape[1] == 79 and int((ids[1] > 0).sum()) == 2       # the truncated sentence; the empty one is [CLS] [SEP]
    pooled, z = bo.bert_encode(sd, ids, cfg)
    for got, ref in ((pooled, gold["pooled"]), (z, gold["z"])):
        assert np.abs(got.numpy() - ref).max() <= 2e-4 * np.abs(ref).max()


def test_pad_keys_do_not_change_a_sentence():
    """the -10000 mask of the reference: a sentence padded to a longer row gives the z it gives alone"""
    cfg, sd, gold = _mini()
    ids = torch.from_numpy(gold["ids"]).long()
    z = bo.bert_encode(sd, ids, cfg)[1]
    for b in range(ids.shape[0]):
        n = int((ids[b] > 0).sum())
        alone = bo.bert_encode(sd, ids[b:b + 1, :n], cfg)[1]
        assert (alone - z[b]).abs().max() <= 1e-5 * z.abs().max()


def test_oracle_against_live_reference():
    """the reference imports its own `lib` package, so it runs in a child process (tools/make_bert_golden.py --check)"""
    import subprocess
    import sys
    from oracle import ref_shims
    if not ref_shims.available():
        pytest.skip("reference tree not present")
    tool = os.path.join(os.path.dirname(GOLD), "..", "tools", "make_bert_golden.py")
    r = subprocess.run([sys.executable, tool, "--check"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "oracle matches the reference" in r.stdout, r.stdout + r.stderr


def test_tokenizer_matches_reference_ids(tok):
    from lib.model_zoo.optimus import BertTokenizer
    vocab, cases = tok
    tk = BertTokenizer(vocab_file=vocab)
    assert len(cases) >= 200
    kinds = {"ws": 0, "trunc": 0, "long_word": 0}
    for c in cases:
        pieces = tk.tokenize(c["text"].lower())
        if c["whitespace_only"]:
            # the reference's piece is whichever special token Python's set order puts first; here it is always [UNK]
            assert pieces == ["[UNK]"] and len(c["pieces"]) == 1 and c["pieces"][0].startswith("["), c
            kinds["ws"] += 1
            continue
        assert pieces == c["pieces"], repr(c["text"])
        assert tk.encode_sentences([c["text"]])[0] == c["ids"], repr(c["text"])
        kinds["trunc"] += len(c["pieces"]) > 77
        kinds["long_word"] += "[UNK]" in c["pieces"]
    assert all(v > 0 for v in kinds.values()), kinds
    assert tk.tokenize("don't stop\tthe\x00music") == ["don", "'", "t", "stop", "them", "##us", "##ic"]
    assert (tk.cls_token_id, tk.sep_token_id) == (bo.CLS_ID, bo.SEP_ID)


def test_tokenizer_missing_vocab_is_a_clear_error(monkeypatch, tmp_path, tok):
    from lib.model_zoo.optimus import BertTokenizer
    monkeypatch.delenv("VDB_BERT_VOCAB", raising=False)
    with pytest.raises(RuntimeError, match="VDB_BERT_VOCAB"):
        BertTokenizer(vocab_file=str(tmp_path / "nope.txt")).tokenize("hello")
    monkeypatch.setenv("VDB_BERT_VOCAB", tok[0])
    assert BertTokenizer(vocab_file=str(tmp_path / "nope.txt")).encode_sentences(["A."])[0] == [bo.CLS_ID, 170, 119, bo.SEP_ID]


def test_encoder_in_bank_only_with_text_encoder_switch(monkeypatch):
    from lib.cfg_helper import model_cfg_bank
    bank = model_cfg_bank()
    monkeypatch.setenv("VDB_TEXT_FLOWS", "1")
    monkeypatch.delenv("VDB_TEXT_ENCODER", raising=False)
    cfg = bank("optimus_v1")
    assert "encoder" not in cfg.args and "tokenizer_encoder" not in cfg.args      # the decoder-only default stays
    monkeypatch.setenv("VDB_TEXT_ENCODER", "1")
    cfg = bank("optimus_v1")
    assert cfg.args.encoder.type == "optimus_bert_connector" and cfg.args.tokenizer_encoder.type == "optimus_bert_tokenizer"
    c = cfg.args.encoder.args.config
    assert (c.hidden_size, c.num_attention_heads, c.num_hidden_layers, c.intermediate_size, c.vocab_size, c.layer_norm_eps,
            c.max_position_embeddings, cfg.args.encoder.args.latent_size) == (768, 12, 12, 3072, 28996, 1e-12, 512, 768)
    assert cfg.args.tokenizer_encoder.args.vocab_file == "lib/model_zoo/optimus_models/vocab/bert-base-cased-vocab.txt"
    assert cfg.args.decoder.type == "optimus_gpt2_connector"
    monkeypatch.delenv("VDB_TEXT_FLOWS")                                          # the switch needs VDB_TEXT_FLOWS=1
    with pytest.raises(KeyError):
        bank("optimus_v1")
    assert [n for n, _ in bank("vd_four_flow_v1-0").args.vae_cfg_list] == ["image"]


@pytest.mark.parametrize("size", ["mini", "full"])
def test_encoder_keys_match_reference(size):
    from lib.model_zoo.optimus import BertForLatentConnector_XX, BertTokenizer
    from lib.model_zoo.optimus import optimus_vae_next, GPT2ForLatentConnector_XX, GPT2Detokenizer
    enc = BertForLatentConnector_XX(bo.encoder_config(size == "mini"), latent_size=768)
    ref = json.load(open(os.path.join(GOLD, f"keys_optimus_encoder_{size}.json")))
    assert {"encoder." + k: list(v.shape) for k, v in enc.state_dict().items()} == ref
    assert {k: tuple(v) for k, v in ref.items()} == {"encoder." + k: v for k, v in bo.encoder_shapes(bo.encoder_config(size == "mini")).items()}
    vae = optimus_vae_next(encoder=enc, decoder=GPT2ForLatentConnector_XX(oo.decoder_config(size == "mini")),
                           tokenizer_encoder=BertTokenizer(), tokenizer_decoder=GPT2Detokenizer())
    keys = {k: list(v.shape) for k, v in vae.state_dict().items()}
    dec = json.load(open(os.path.join(GOLD, f"keys_optimus_{size}.json")))
    assert keys == {**dec, **ref}


def test_vae_builds_with_encoder_through_registry(monkeypatch):
    monkeypatch.setenv("VDB_TEXT_FLOWS", "1")
    monkeypatch.setenv("VDB_TEXT_ENCODER", "1")
    from lib.cfg_helper import model_cfg_bank
    from lib.model_zoo.common.get_model import get_model
    cfg = model_cfg_bank()("optimus_v1")
    cfg.args.decoder.args.config.update(oo.decoder_config(True))
    cfg.args.encoder.args.config.update(bo.encoder_config(True))
    vae = get_model()(cfg, verbose=False)
    keys = {k: list(v.shape) for k, v in vae.state_dict().items()}
    assert keys == {**json.load(open(os.path.join(GOLD, "keys_optimus_mini.json"))),
                    **json.load(open(os.path.join(GOLD, "keys_optimus_encoder_mini.json")))}
    # a checkpoint's vae.text.encoder.* keys load with nothing missing
    sd = {k: v + 0.5 for k, v in vae.state_dict().items()}
    res = vae.load_state_dict(sd, strict=False)
    assert not [k for k in res.missing_keys if k.startswith("encoder.")] and not res.unexpected_keys
    assert torch.equal(vae.encoder.linear.weight, sd["encoder.linear.weight"])


def test_encode_argument_checks_without_gpu(tok):
    from lib.model_zoo.optimus import BertForLatentConnector_XX, BertTokenizer
    from lib.model_zoo.optimus import optimus_vae_next, GPT2ForLatentConnector_XX, GPT2Detokenizer
    vae = optimus_vae_next(encoder=BertForLatentConnector_XX(bo.encoder_config(True), latent_size=768),
                           decoder=GPT2ForLatentConnector_XX(oo.decoder_config(True)),
                           tokenizer_encoder=BertTokenizer(vocab_file=tok[0]), tokenizer_decoder=GPT2Detokenizer())
    with pytest.raises(ValueError, match="510"):
        vae.encode(["a sentence"], max_length=511)
    with pytest.raises(ValueError, match="no sentences"):
        vae.encode([])
    with pytest.raises(RuntimeError, match="no CPU path"):
        vae.encode(["a sentence"])


def test_new_abi_entries_check_arguments_without_gpu():
    from vdb200._lib import lib
    # attention with key lengths: a null kv_len, then the checks it shares with vdb_attention_bf16
    assert lib.vdb_attention_keylen_bf16(8, 64, 0, 8, 64, 0, 8, 64, 8, 64, 1, 1, 8, 8, 0, 0, 64, 0.125, 0, None, None) == 1
    assert b"kv_len" in lib.vdb_last_error()
    assert lib.vdb_attention_keylen_bf16(None, 64, 0, None, 64, 0, None, 64, None, 64, 1, 1, 8, 8, 0, 0, 64, 0.125, 0, 8, None) == 1
    assert lib.vdb_attention_keylen_bf16(8, 64, 0, 8, 64, 0, 8, 64, 8, 64, 1, 1, 8, 9, 0, 9, 64, 0.125, 0, 8, None) == 1
    assert b"kv_bstride" in lib.vdb_last_error()
    # the embedding: width, position table, alignment
    args = dict(ids=16, n=2, L=8, word=16, vocab=100, pos=16, max_pos=512, typ=16, g=16, b=16, eps=1e-12, C=128, y=16)

    def call(**kw):
        a = dict(args, **kw)
        return lib.vdb_bert_embed_ln(a["ids"], a["n"], a["L"], a["word"], a["vocab"], a["pos"], a["max_pos"], a["typ"], a["g"],
                                     a["b"], a["eps"], a["C"], a["y"], None)
    assert call(ids=None) == 1 and b"null" in lib.vdb_last_error()
    assert call(C=96) == 1 and b"multiple of 128" in lib.vdb_last_error()
    assert call(C=1152) == 1
    assert call(L=513) == 1 and b"position table" in lib.vdb_last_error()
    assert call(y=24) == 1 and b"aligned" in lib.vdb_last_error()


def test_tanh_act_code():
    from vdb200 import ops
    assert ops.ACT_TANH == 6 and ops.ACT_GELU_TANH == 5
