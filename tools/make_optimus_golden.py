"""Generates the Optimus text-decode fixtures under tests/golden/ by running the UNMODIFIED reference decoder and tokenizer on
CPU fp32 (through oracle/ref_shims.py, so it needs the reference tree) with the synthetic weights of tests/optimus_oracle.py.

    python tools/make_optimus_golden.py            # (re)writes the fixtures below
    python tools/make_optimus_golden.py --check    # oracle vs the live reference on weights and inputs unlike the fixtures'

Writes only these files (every other fixture is left alone):
  keys_optimus_full.json / keys_optimus_mini.json   state_dict key -> shape of the decoder (optimus_vae_next's 'decoder.*' keys,
                                                    the tied lm_head included), full size and the reduced test decoder
  optimus_mini.npz     reduced decoder: teacher-forced logits at logit_columns() + per-position logsumexp (2 rows x 12 positions),
                       token sequences at temperature 1.0 and 0.7 with torch.multinomial replaced by an inverse-CDF draw on the
                       golden uniforms, and one row whose draw at step EOS_STEP lands inside <EOS>'s interval
  gpt2_detok.json.gz    200 cases: ids -> the tokenizer's decode() string and the sentence optimus_vae_next.decode makes of it,
                        plus the vocabulary entries those ids use (so tests can detokenize without the reference tree)
"""
import gzip
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import ref_shims, weights  # noqa: E402
import optimus_oracle as oo  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
EOS_STEP = 4
TEMPERATURES = (1.0, 0.7)


def ref_decoder(mini):
    ns = ref_shims.load()
    with ref_shims._cwd(ref_shims.REF):
        cfg = ns.model_cfg_bank()("optimus_gpt2_decoder")
        if mini:
            c = oo.decoder_config(True)
            cfg.args.config.update({k: c[k] for k in ("hidden_size", "n_embd", "n_head", "num_attention_heads", "n_layer",
                                                      "num_hidden_layers")})
        net = ns.get_model()(cfg, verbose=False)
    net.eval()
    return net


def ref_tokenizer():
    ns = ref_shims.load()
    with ref_shims._cwd(ref_shims.REF):
        tk = ns.get_model()(ns.model_cfg_bank()("optimus_gpt2_tokenizer"), verbose=False)
    tk.add_special_tokens({'pad_token': '<PAD>', 'bos_token': '<BOS>', 'eos_token': '<EOS>'})   # optimus.py:30-34
    return tk


def key_table(net):
    return {"decoder." + k: list(v.shape) for k, v in net.state_dict().items()}


def ref_sample(net, z, uniforms, temperature):
    """the reference's sample_single_sequence_conditional with torch.multinomial drawing by inverse CDF on the given uniforms"""
    mod = sys.modules["lib.model_zoo.optimus"]
    out = []
    real = torch.multinomial
    try:
        for r in range(z.shape[0]):
            draws = iter(uniforms[r])
            torch.multinomial = lambda p, num_samples=1: torch.tensor([oo.inverse_cdf(p.numpy(), float(next(draws)))])
            seq = mod.sample_single_sequence_conditional(model=net, context=torch.LongTensor([oo.BOS_ID]), past=z[r],
                                                         temperature=temperature, top_k=0, top_p=1.0, max_length=oo.MAX_LENGTH,
                                                         eos_token=oo.EOS_ID)
            out.append([int(v) for v in seq])
    finally:
        torch.multinomial = real
    return out


def padded(seqs):
    a = np.full((len(seqs), oo.MAX_LENGTH), -1, dtype=np.int64)
    for i, s in enumerate(seqs):
        a[i, :len(s)] = s
    return a


def detok_cases(tk, vocab):
    rng = np.random.RandomState(2024)
    enc = {b: u for b, u in zip(range(256), _byte_chars())}
    high_bytes = [vocab[enc[b]] for b in range(128, 256)]                  # single-byte tokens: broken / partial UTF-8
    punct = [vocab[s] for s in ("Ġ.", "Ġ,", "Ġ?", "Ġ!", "Ġ'", "'", "Ġn't", "n't", "'m", "Ġ'm",
                                "'s", "Ġ's", "'ve", "Ġ've", "'re", "Ġ're", "Ġdo", "Ġnot", ".", ",", "!", "?")
             if s in vocab]
    special = [oo.PAD_ID, oo.BOS_ID, oo.EOS_ID]
    cases = []
    fixed = [[oo.BOS_ID, 15496, 11, 995, 13, oo.EOS_ID], [oo.BOS_ID, oo.EOS_ID], [oo.BOS_ID], [], [oo.EOS_ID],
             [oo.BOS_ID, vocab["Ġdo"], vocab["Ġnot"], oo.EOS_ID], [oo.BOS_ID, 50256, oo.EOS_ID]]
    cases.extend(fixed)
    for i in range(200 - len(fixed)):
        L = int(rng.randint(0, 20))
        body = []
        for _ in range(L):
            r = rng.rand()
            if r < 0.55:
                body.append(int(rng.randint(0, oo.PAD_ID)))
            elif r < 0.75:
                body.append(int(rng.choice(punct)))
            elif r < 0.92:
                body.append(int(rng.choice(high_bytes)))
            else:
                body.append(int(rng.choice(special)))
        start = [oo.BOS_ID] if i % 10 else []
        end = [oo.EOS_ID] if i % 7 else []
        cases.append(start + body + end)
    out = []
    for ids in cases:
        s = tk.decode(ids, clean_up_tokenization_spaces=True)
        out.append({"ids": ids, "decoded": s, "sentence": " ".join(s.split()[1:-1])})
    return out


def _byte_chars():
    from lib.model_zoo.optimus_models.tokenization_gpt2 import bytes_to_unicode   # the reference's table
    t = bytes_to_unicode()
    return [t[b] for b in range(256)]


def main():
    torch.set_grad_enabled(False)
    full, mini = ref_decoder(False), ref_decoder(True)
    for name, net in (("full", full), ("mini", mini)):
        json.dump(key_table(net), open(os.path.join(GOLD, f"keys_optimus_{name}.json"), "w"))
    del full

    cfg = oo.decoder_config(True)
    sd = oo.synth_decoder_sd(weights.param_shapes(mini))
    missing = mini.load_state_dict(sd, strict=False).missing_keys
    assert all(k.endswith(".attn.bias") for k in missing), missing
    gi = oo.golden_inputs("mini")
    z, tokens, uniforms = gi["z"], gi["tokens"], gi["uniforms"]
    cols = oo.logit_columns()
    logits = torch.cat([mini(input_ids=tokens[r:r + 1], past=z[r:r + 1])[0] for r in range(z.shape[0])])
    out = {"cols": cols, "logits": logits[..., cols].numpy(), "lse": torch.logsumexp(logits, dim=-1).numpy()}
    for T in TEMPERATURES:
        out[f"seq_t{T}"] = padded(ref_sample(mini, z, uniforms, T))
    ue = oo.eos_uniforms(sd, z, uniforms, 1.0, cfg, 0, EOS_STEP)
    out["eos_uniforms"] = ue[:1]
    out["eos_step"] = np.array(EOS_STEP)
    out["seq_eos"] = padded(ref_sample(mini, z[:1], ue[:1], 1.0))
    assert out["seq_eos"][0, EOS_STEP + 1] == oo.EOS_ID
    np.savez_compressed(os.path.join(GOLD, "optimus_mini.npz"), **out)

    tk = ref_tokenizer()
    vocab_src = os.path.join(ref_shims.REF, "lib/model_zoo/optimus_models/vocab/gpt2-vocab.json")
    vocab = json.load(open(vocab_src, encoding="utf-8"))
    cases = detok_cases(tk, vocab)
    used = {i for c in cases for i in c["ids"]}
    doc = {"vocab": {t: i for t, i in vocab.items() if i in used}, "cases": cases}
    with open(os.path.join(GOLD, "gpt2_detok.json.gz"), "wb") as fh:
        with gzip.GzipFile(fileobj=fh, mode="wb", mtime=0, filename="") as gz:     # byte-reproducible
            gz.write(json.dumps(doc, ensure_ascii=True, sort_keys=True, separators=(",", ":")).encode())
    print("wrote keys_optimus_{full,mini}.json, optimus_mini.npz, gpt2_detok.json.gz")


def check():
    torch.set_grad_enabled(False)
    cfg = oo.decoder_config(True)
    net = ref_decoder(True)
    sd = oo.synth_decoder_sd(weights.param_shapes(net), seed=17)
    net.load_state_dict(sd, strict=False)
    g = torch.Generator().manual_seed(5)
    z = torch.randn(1, 768, generator=g)
    tokens = torch.cat([torch.tensor([[oo.BOS_ID]]), torch.randint(0, oo.PAD_ID, (1, 7), generator=g)], dim=1)
    ref = net(input_ids=tokens, past=z)[0]
    err = float((oo.gpt2_text_logits(sd, z, tokens, cfg) - ref).abs().max() / ref.abs().max())
    assert err <= 2e-4, err
    u = torch.rand(1, oo.MAX_LENGTH - 1, generator=g, dtype=torch.float64).numpy()
    assert ref_sample(net, z, u, 0.8) == oo.optimus_sample(sd, z, u, 0.8, cfg)
    print(f"oracle matches the reference (logits rel err {err:.2e}, sequence equal)")


if __name__ == "__main__":
    check() if "--check" in sys.argv[1:] else main()
