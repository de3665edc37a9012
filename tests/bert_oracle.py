"""CPU fp32 restatement of the Optimus BERT text encoder (reference lib/model_zoo/optimus.py:729-743 on
optimus_models/optimus_bert.py:144-376, 1349-1439) — the oracle the text-encode tests compare the CUDA path against.

Like the reference it runs every padded row through all positions and masks the pad keys with an additive -10000 (the CUDA path
leaves them out).  Also the configs, synthetic-weight helpers and seeded sentences shared by tools/make_bert_golden.py and the
tests.
"""
import gzip
import json
import math
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from oracle import weights  # noqa: E402

WEIGHT_SEED = 7
CLS_ID, SEP_ID, PAD_ID, UNK_ID = 101, 102, 0, 100


def encoder_config(mini):
    """configs/model/optimus.yaml:7-31 (full) and the reduced encoder of the fast tests (width 128, 2 heads of 64, 2 layers,
    intermediate 512, the full 28996-entry vocabulary)"""
    c = dict(hidden_act="gelu", hidden_size=768, initializer_range=0.02, intermediate_size=3072, layer_norm_eps=1e-12,
             max_position_embeddings=512, num_attention_heads=12, num_hidden_layers=12, type_vocab_size=2, vocab_size=28996)
    if mini:
        c.update(hidden_size=128, num_attention_heads=2, num_hidden_layers=2, intermediate_size=512)
    return c


def synth_encoder_sd(shapes, seed=WEIGHT_SEED):
    """synthetic weights for the encoder's parameters (state_dict keys without the 'encoder.' prefix)"""
    return weights.synth_state_dict(shapes, seed)


def encoder_shapes(cfg, latent_size=768):
    """{key: shape} of BertForLatentConnector_XX's parameters, from the config alone"""
    C, I, L = cfg["hidden_size"], cfg["intermediate_size"], cfg["num_hidden_layers"]
    s = {"embeddings.word_embeddings.weight": (cfg["vocab_size"], C),
         "embeddings.position_embeddings.weight": (cfg["max_position_embeddings"], C),
         "embeddings.token_type_embeddings.weight": (cfg["type_vocab_size"], C),
         "embeddings.LayerNorm.weight": (C,), "embeddings.LayerNorm.bias": (C,)}
    for i in range(L):
        p = f"encoder.layer.{i}."
        for n in ("query", "key", "value"):
            s[p + f"attention.self.{n}.weight"], s[p + f"attention.self.{n}.bias"] = (C, C), (C,)
        s[p + "attention.output.dense.weight"], s[p + "attention.output.dense.bias"] = (C, C), (C,)
        s[p + "attention.output.LayerNorm.weight"], s[p + "attention.output.LayerNorm.bias"] = (C,), (C,)
        s[p + "intermediate.dense.weight"], s[p + "intermediate.dense.bias"] = (I, C), (I,)
        s[p + "output.dense.weight"], s[p + "output.dense.bias"] = (C, I), (C,)
        s[p + "output.LayerNorm.weight"], s[p + "output.LayerNorm.bias"] = (C,), (C,)
    s["pooler.dense.weight"], s["pooler.dense.bias"] = (C, C), (C,)
    s["linear.weight"] = (2 * latent_size, C)
    return s


def tokenizer_cases():
    """the reference tokenizer's cases of tests/golden/bert_tok.json.gz and the vocabulary entries they use"""
    with gzip.open(os.path.join(ROOT, "tests", "golden", "bert_tok.json.gz")) as fh:
        return json.load(fh)


def write_vocab(path):
    """the fixture's vocabulary entries at their line numbers (= ids) as a vocabulary file; the other lines hold strings no text
    can produce (they start with NUL, which the text cleaning drops) -> the path"""
    vocab = tokenizer_cases()["vocab"]
    lines = [f"\x00unused{i}" for i in range(max(vocab.values()) + 1)]
    for piece, i in vocab.items():
        lines[i] = piece
    with open(path, "w", encoding="utf-8") as fh:
        fh.write("\n".join(lines) + "\n")
    return str(path)


def golden_sentences():
    """the batch of the fixtures: different lengths, an empty string, accents / punctuation, and one sentence truncated at 77
    word pieces"""
    long = " ".join(f"word{i}, again" for i in range(60))
    return ["a man rides a horse on the beach.", "", "Héllo wörld! It's 3:45pm — don't stop.", "two words",
            long, "the quick brown fox jumps over the lazy dog near the river bank at dawn"]


def full_sentences():
    return ["a small dog plays in the park.", "", "A very long sentence " * 8]


def _ln(x, w, b, eps):
    return F.layer_norm(x, (x.shape[-1],), w, b, eps)


def pad_ids(rows):
    """pad_sequence(batch_first, padding_value=0) of id lists -> int64 [n, L]"""
    L = max(len(r) for r in rows)
    out = torch.full((len(rows), L), PAD_ID, dtype=torch.long)
    for i, r in enumerate(rows):
        out[i, :len(r)] = torch.tensor(r, dtype=torch.long)
    return out


@torch.no_grad()
def bert_encode(sd, ids, cfg, latent_size=768):
    """ids int64 [n, L] (0 = pad) -> (pooled [n, C], z_mu [n, latent]) with attention_mask = ids > 0"""
    g = lambda k: sd[k].float()
    C, H, eps = cfg["hidden_size"], cfg["num_attention_heads"], cfg["layer_norm_eps"]
    d = C // H
    n, L = ids.shape
    x = g("embeddings.word_embeddings.weight")[ids] + g("embeddings.position_embeddings.weight")[:L][None] \
        + g("embeddings.token_type_embeddings.weight")[0]
    x = _ln(x, g("embeddings.LayerNorm.weight"), g("embeddings.LayerNorm.bias"), eps)
    mask = (1.0 - (ids > 0).float())[:, None, None, :] * -10000.0
    for i in range(cfg["num_hidden_layers"]):
        p = f"encoder.layer.{i}."
        lin = lambda t, name: t @ g(p + name + ".weight").t() + g(p + name + ".bias")
        q, k, v = (lin(x, f"attention.self.{nm}").reshape(n, L, H, d).transpose(1, 2) for nm in ("query", "key", "value"))
        w = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(d) + mask, dim=-1)
        a = (w @ v).transpose(1, 2).reshape(n, L, C)
        x = _ln(lin(a, "attention.output.dense") + x, g(p + "attention.output.LayerNorm.weight"),
                g(p + "attention.output.LayerNorm.bias"), eps)
        f = lin(x, "intermediate.dense")
        f = f * 0.5 * (1.0 + torch.erf(f / math.sqrt(2.0)))
        x = _ln(lin(f, "output.dense") + x, g(p + "output.LayerNorm.weight"), g(p + "output.LayerNorm.bias"), eps)
    pooled = torch.tanh(x[:, 0] @ g("pooler.dense.weight").t() + g("pooler.dense.bias"))
    z = pooled @ g("linear.weight").t()
    return pooled, z[:, :latent_size]
