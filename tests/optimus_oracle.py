"""CPU fp32 restatement of the Optimus GPT-2 text decoder (reference lib/model_zoo/optimus.py:662-763 on
optimus_models/optimus_gpt2.py:99-246, 813-1112) — the oracle the text-decode tests compare the CUDA path against.

Like the reference it has no KV cache: every sampling step re-runs the whole prefix (teacher-forced logits of all positions).
`optimus_sample` replaces torch.multinomial by an inverse-CDF draw on given uniforms, so token sequences can be pinned.
Also the synthetic-weight helpers and seeded inputs shared by tools/make_optimus_golden.py and the tests.
"""
import json
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from oracle import weights  # noqa: E402

PAD_ID, BOS_ID, EOS_ID = 50257, 50258, 50259
VOCAB = 50260
MAX_LENGTH = 30
WEIGHT_SEED = 3


def decoder_config(mini):
    """configs/model/optimus.yaml:43-90 (full) and the reduced decoder of the fast tests (n_embd 128, 2 heads, 2 layers)"""
    c = dict(hidden_size=768, initializer_range=0.02, latent_size=768, layer_norm_epsilon=1e-05, max_position_embeddings=1024,
             n_ctx=1024, n_embd=768, n_head=12, n_layer=12, n_positions=1024, num_attention_heads=12, num_hidden_layers=12,
             vocab_size=VOCAB)
    if mini:
        c.update(hidden_size=128, n_embd=128, n_head=2, num_attention_heads=2, n_layer=2, num_hidden_layers=2)
    return c


def synth_decoder_sd(shapes, seed=WEIGHT_SEED):
    """synthetic weights for the decoder's parameters (the attention-mask buffers and the tied lm_head are not parameters)"""
    sd = weights.synth_state_dict({k: v for k, v in shapes.items() if not k.endswith(".attn.bias") and k != "lm_head.weight"},
                                  seed)
    sd["lm_head.weight"] = sd["transformer.wte.weight"]
    return sd


def synthetic_vocab(path):
    """a stand-in GPT-2 vocabulary json (id i -> ' w<i>'; 'Ġ' is GPT-2's byte character for a space) for tests that only need
    decode() to produce strings; returns the path"""
    with open(path, "w") as fh:
        json.dump({f"\u0120w{i}": i for i in range(PAD_ID)}, fh)
    return str(path)


def golden_inputs(kind):
    g = torch.Generator().manual_seed({"mini": 41, "full": 43}[kind])
    z = torch.randn(2, 768, generator=g)
    tokens = torch.randint(0, PAD_ID, (2, 12), generator=g)
    tokens[:, 0] = BOS_ID
    uniforms = torch.rand(3, MAX_LENGTH - 1, generator=g, dtype=torch.float64).numpy()
    return {"z": z, "tokens": tokens, "uniforms": uniforms}


def logit_columns():
    """the ~512 vocabulary columns kept in the fixtures: a fixed spread plus <PAD>, <BOS>, <EOS>"""
    cols = np.unique(np.concatenate([np.linspace(0, PAD_ID - 1, 509).round().astype(np.int64), [PAD_ID, BOS_ID, EOS_ID]]))
    return cols


def _ln(x, w, b, eps):
    return torch.nn.functional.layer_norm(x, (x.shape[-1],), w, b, eps)


def _gelu_tanh(x):
    return 0.5 * x * (1 + torch.tanh(math.sqrt(2 / math.pi) * (x + 0.044715 * torch.pow(x, 3))))


@torch.no_grad()
def gpt2_text_logits(sd, z, tokens, cfg):
    """Teacher-forced logits [n, T, vocab] of the decoder (state_dict keys without the 'decoder.' prefix) for latents z [n, 768]
    and tokens [n, T] starting with <BOS>: latent as embedding and as one memory slot per layer, positions from 1."""
    g = lambda k: sd[k].float()
    C, H, L, eps = cfg["n_embd"], cfg["n_head"], cfg["n_layer"], cfg["layer_norm_epsilon"]
    d = C // H
    z = z.float()
    n, T = tokens.shape
    lin = z @ g("transformer.linear.weight").t()                             # [n, L*C]: past key == past value per layer
    lemb = z @ g("transformer.linear_emb.weight").t()
    x = g("transformer.wte.weight")[tokens] + g("transformer.wpe.weight")[1:T + 1][None] + lemb[:, None]
    keep = torch.tril(torch.ones(T, T + 1), diagonal=1)                        # query i sees the memory slot and tokens 0..i
    for li in range(L):
        p = f"transformer.h.{li}."
        h = _ln(x, g(p + "ln_1.weight"), g(p + "ln_1.bias"), eps)
        qkv = h @ g(p + "attn.c_attn.weight") + g(p + "attn.c_attn.bias")
        q, k, v = (t.reshape(n, T, H, d).transpose(1, 2) for t in qkv.split(C, dim=2))
        mem = lin[:, li * C:(li + 1) * C].reshape(n, 1, H, d).transpose(1, 2)
        k = torch.cat([mem, k], dim=2)
        v = torch.cat([mem, v], dim=2)
        w = q @ k.transpose(-1, -2) / math.sqrt(d)
        w = w * keep - 1e4 * (1 - keep)
        a = (torch.softmax(w, dim=-1) @ v).transpose(1, 2).reshape(n, T, C)
        x = x + a @ g(p + "attn.c_proj.weight") + g(p + "attn.c_proj.bias")
        h = _ln(x, g(p + "ln_2.weight"), g(p + "ln_2.bias"), eps)
        m = _gelu_tanh(h @ g(p + "mlp.c_fc.weight") + g(p + "mlp.c_fc.bias"))
        x = x + m @ g(p + "mlp.c_proj.weight") + g(p + "mlp.c_proj.bias")
    x = _ln(x, g("transformer.ln_f.weight"), g("transformer.ln_f.bias"), eps)
    return x @ g("transformer.wte.weight").t()


def inverse_cdf(probs, u):
    """smallest i with cumsum(probs)[i] > u (float64 running sum in vocabulary order); the last non-zero entry if u is beyond"""
    c = np.cumsum(np.asarray(probs, dtype=np.float64))
    i = int(np.searchsorted(c, u, side="right"))
    if i >= len(c):
        i = int(np.nonzero(np.asarray(probs) > 0)[0][-1])
    return i


def top_p_filter(logits, top_p=1.0):
    """the reference's nucleus filter with top_k = 0 (optimus.py:690-720): masks the tokens past the first whose fp32 cumulative
    probability exceeds top_p — at top_p = 1.0 only tokens whose cumulative sum rounds above 1"""
    logits = logits.clone()
    sl, si = torch.sort(logits, descending=True)
    cp = torch.cumsum(torch.softmax(sl, dim=-1), dim=-1)
    rm = cp > top_p
    rm[..., 1:] = rm[..., :-1].clone()
    rm[..., 0] = 0
    logits[si[rm]] = -float("inf")
    return logits


@torch.no_grad()
def optimus_sample(sd, z, uniforms, temperature, cfg, use_filter=True):
    """sample_single_sequence_conditional per row with u = uniforms[row, step] as the multinomial draw -> list of id lists"""
    out = []
    for r in range(z.shape[0]):
        seq = [BOS_ID]
        for k in range(MAX_LENGTH - 1):
            last = gpt2_text_logits(sd, z[r:r + 1], torch.tensor([seq]), cfg)[0, -1] / temperature
            if use_filter:
                last = top_p_filter(last, 1.0)
            tok = inverse_cdf(torch.softmax(last, dim=-1).numpy(), float(uniforms[r, k]))
            seq.append(tok)
            if tok == EOS_ID:
                break
            if len(seq) >= MAX_LENGTH:
                seq[-1] = EOS_ID
                break
        out.append(seq)
    return out


def eos_uniforms(sd, z, uniforms, temperature, cfg, row, k):
    """uniforms with row `row`'s draw at step k moved inside <EOS>'s CDF interval (the sequence then stops at step k)"""
    u = np.array(uniforms, dtype=np.float64)
    seq = [BOS_ID]
    for j in range(k + 1):
        last = gpt2_text_logits(sd, z[row:row + 1], torch.tensor([seq]), cfg)[0, -1] / temperature
        p = torch.softmax(top_p_filter(last, 1.0), dim=-1).numpy()
        if j < k:
            seq.append(inverse_cdf(p, float(u[row, j])))
            assert seq[-1] != EOS_ID, "the draws before step k already end the sequence"
    c = np.cumsum(p.astype(np.float64))
    u[row, k] = 0.5 * (c[EOS_ID - 1] + c[EOS_ID])
    return u
