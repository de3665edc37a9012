"""Generates the Optimus text-encode fixtures under tests/golden/ by running the UNMODIFIED reference encoder and tokenizer on
CPU fp32 (through oracle/ref_shims.py, so it needs the reference tree): the reference's own optimus_vae_next.encode on the
synthetic weights of tests/bert_oracle.py.

    python tools/make_bert_golden.py            # (re)writes the fixtures below
    python tools/make_bert_golden.py --check    # oracle vs the live reference on weights and sentences unlike the fixtures'

Writes only these files (every other fixture is left alone):
  keys_optimus_encoder_full.json / keys_optimus_encoder_mini.json   state_dict key -> shape of the encoder ('encoder.*' keys of
                                                                    optimus_vae_next), full size and the reduced test encoder
  bert_mini.npz       reduced encoder: the padded ids, the pooler output and z of golden_sentences(); z of the full-size encoder
                      for full_sentences() (the tests regenerate the full weights from the seed)
  bert_tok.json.gz    >= 200 strings -> the reference tokenizer's pieces of text.lower() and the ids encode() builds from them,
                      plus the vocabulary entries those ids and the sentences of bert_mini.npz use (greedy longest match
                      gives the same pieces on that subset)
"""
import gzip
import json
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import ref_shims  # noqa: E402
import bert_oracle as bo  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
SPECIAL = ("[UNK]", "[SEP]", "[PAD]", "[CLS]", "[MASK]")


def ref_parts(mini):
    ns = ref_shims.load()
    with ref_shims._cwd(ref_shims.REF):
        bank = ns.model_cfg_bank()
        cfg = bank("optimus_bert_encoder")
        if mini:
            cfg.args.config.update({k: v for k, v in bo.encoder_config(True).items()
                                    if k in ("hidden_size", "num_attention_heads", "num_hidden_layers", "intermediate_size")})
        enc = ns.get_model()(cfg, verbose=False)
        tk = ns.get_model()(bank("optimus_bert_tokenizer"), verbose=False)
    enc.eval()
    return enc, tk


def ref_encode(enc, tk, sentences):
    """the reference's optimus_vae_next.encode, unbound, on an object holding just the encoder half"""
    mod = sys.modules["lib.model_zoo.optimus"]
    host = types.SimpleNamespace(encoder=enc, tokenizer_encoder=tk, get_device=lambda: torch.device("cpu"))
    return mod.optimus_vae_next.encode(host, sentences)


def ref_ids(tk, text, max_length=77):
    """the id row optimus.py:731-737 builds for one sentence"""
    pieces = tk.tokenize(text.lower())
    return pieces, tk.add_special_tokens_single_sentence([tk._convert_token_to_id(p) for p in pieces[:max_length]])


def tok_strings():
    rng = np.random.RandomState(2025)
    words = ["the", "cat", "sat", "on", "mat", "running", "unbelievable", "tokenization", "Paris", "NASA", "x", "I", "hello",
             "world", "don't", "it's", "we'll", "they're", "o'clock", "rock'n'roll", "e-mail", "U.S.A.", "3.14", "2024",
             "1,000,000", "#hashtag", "@user", "a+b=c", "50%", "$9.99", "(parens)", "[brackets]", "{braces}", "<tag>",
             "café", "naïve", "façade", "Ångström", "jalapeño", "Zürich", "résumé", "Ελληνικά", "русский", "العربية",
             "中文", "日本語の文", "한국어", "東京タワー", "😀", "👍🏽", "🚀✨", "♥", "—", "…", "«quote»", "¿qué?", "¡sí!",
             "a\u00adb", "zero\u200bwidth", "tab\tsep", "new\nline", "cr\rlf", "nul\x00byte", "bell\x07", "rep\ufffdlace",
             "\x1fus", "nbsp\u00a0space", "ideo\u3000space", "line\u2028sep", "para\u2029sep", "soft\x85nl", "ﬁ", "Ⅻ", "²³", "½"]
    fixed = ["don't stop\tthe\x00music", "", " ", "   ", "\t\n", "　", "\x1f", "\x00", "\x00\x07", "a", "A.B.C.",
             "x" * 101, "y" * 100, "supercalifragilisticexpialidocious" * 3, " ".join(["word"] * 90),
             " ".join(f"token{i}" for i in range(50)), "中文字符测试", "Hello, World!", "  leading and trailing  "]
    out = list(fixed)
    while len(out) < 240:
        k = int(rng.randint(1, 14))
        parts = [str(rng.choice(words)) for _ in range(k)]
        seps = [str(rng.choice([" ", " ", " ", "", "\t", "\n", "  "])) for _ in range(k)]
        s = "".join(p + q for p, q in zip(parts, seps))
        if rng.rand() < 0.15:
            s = s.upper()
        if rng.rand() < 0.05:
            s = s * 12                                   # far over 77 pieces
        out.append(s)
    return out


def tok_cases(tk):
    cases = []
    for s in tok_strings():
        pieces, ids = ref_ids(tk, s)
        ws = bool(s) and not s.strip()
        if ws:   # the reference picks ONE special token by Python's (hash-seeded) set order of the special-token strings
            assert len(pieces) == 1 and pieces[0] in SPECIAL, (s, pieces)
        cases.append({"text": s, "pieces": pieces, "ids": ids, "whitespace_only": ws})
    return cases


def key_table(enc):
    return {"encoder." + k: list(v.shape) for k, v in enc.state_dict().items()}


def main():
    torch.set_grad_enabled(False)
    full, tk = ref_parts(False)
    mini, _ = ref_parts(True)
    for name, net in (("full", full), ("mini", mini)):
        json.dump(key_table(net), open(os.path.join(GOLD, f"keys_optimus_encoder_{name}.json"), "w"))

    cfg = bo.encoder_config(True)
    sd = bo.synth_encoder_sd({k: tuple(v.shape) for k, v in mini.state_dict().items()})
    mini.load_state_dict(sd, strict=True)
    sents = bo.golden_sentences()
    rows = [ref_ids(tk, s)[1] for s in sents]
    ids = bo.pad_ids(rows)
    assert max(len(r) for r in rows) == 79, "one golden sentence must be truncated at 77 pieces"
    z = ref_encode(mini, tk, sents)
    pooled = mini(ids, attention_mask=(ids > 0).float())[1]
    out = {"ids": ids.numpy().astype(np.int32), "pooled": pooled.numpy(), "z": z.numpy()}
    oz = bo.bert_encode(sd, ids, cfg)[1]
    print(f"mini: oracle vs reference z max rel err {float((oz - z).abs().max() / z.abs().max()):.2e}")

    fsd = bo.synth_encoder_sd({k: tuple(v.shape) for k, v in full.state_dict().items()})
    full.load_state_dict(fsd, strict=True)
    fs = bo.full_sentences()
    out["full_ids"] = bo.pad_ids([ref_ids(tk, s)[1] for s in fs]).numpy().astype(np.int32)
    out["full_z"] = ref_encode(full, tk, fs).numpy()
    np.savez_compressed(os.path.join(GOLD, "bert_mini.npz"), **out)

    cases = tok_cases(tk)
    used = {p for c in cases for p in c["pieces"]} | set(SPECIAL)
    used |= {p for s in bo.golden_sentences() + bo.full_sentences() for p in tk.tokenize(s.lower())}   # GPU tests encode them
    doc = {"vocab": {p: tk.vocab[p] for p in sorted(used)}, "cases": cases}
    with open(os.path.join(GOLD, "bert_tok.json.gz"), "wb") as fh:
        with gzip.GzipFile(fileobj=fh, mode="wb", mtime=0, filename="") as gz:     # byte-reproducible
            gz.write(json.dumps(doc, ensure_ascii=True, sort_keys=True, separators=(",", ":")).encode())
    print(f"wrote keys_optimus_encoder_{{full,mini}}.json, bert_mini.npz, bert_tok.json.gz ({len(cases)} cases, "
          f"{len(doc['vocab'])} vocabulary entries)")


def check():
    torch.set_grad_enabled(False)
    cfg = bo.encoder_config(True)
    net, tk = ref_parts(True)
    sd = bo.synth_encoder_sd({k: tuple(v.shape) for k, v in net.state_dict().items()}, seed=17)
    net.load_state_dict(sd, strict=True)
    sents = ["fresh words: zebra, quantum, saxophone!", "short", "", "émigré naïveté " * 30]
    z = ref_encode(net, tk, sents)
    ids = bo.pad_ids([ref_ids(tk, s)[1] for s in sents])
    pooled = net(ids, attention_mask=(ids > 0).float())[1]
    op, oz = bo.bert_encode(sd, ids, cfg)
    err = max(float((oz - z).abs().max() / z.abs().max()), float((op - pooled).abs().max() / pooled.abs().max()))
    assert err <= 2e-4, err
    print(f"oracle matches the reference (rel err {err:.2e})")


if __name__ == "__main__":
    check() if "--check" in sys.argv[1:] else main()
