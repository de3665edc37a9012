"""Optimus text VAE on vdb200 kernels — reference lib/model_zoo/optimus.py:17-52, 636-763,
optimus_models/optimus_gpt2.py:99-246, 813-1112 (decoder) and optimus_models/optimus_bert.py:144-376, 1349-1439 (encoder).

`optimus_vae_next.decode(z)` turns text latents [n, 768] into sentences like the reference's: a GPT-2 decoder that sees the
latent twice — `linear_emb(z)` added to every input embedding and one slice of `linear(z)` per layer used as a one-slot past
key AND value — samples up to 30 tokens from `<BOS>`.  The reference re-runs the whole prefix for every token and samples on
the host; here every layer keeps a bf16 KV cache, the sampler runs on the device, and the token step is one captured CUDA
graph replayed 28 times, so the host sees only the final [n, 30] token ids.

`optimus_vae_next.encode(sentences)` maps sentences to the latent mean z_mu [n, 768] like the reference: a clean-room BERT
WordPiece tokenizer on the host, one copy of the padded ids to the device, then a post-LN BERT-base encoder whose attention
leaves every sentence's pad keys out (vdb_attention_keylen_bf16), the tanh pooler on [CLS] and the first half of `linear`.

The module trees keep the reference's state_dict keys and shapes (`decoder.transformer.*`, `decoder.lm_head` tied to `wte`;
`encoder.embeddings.*`, `encoder.encoder.layer.N.*`, `encoder.pooler.dense`, `encoder.linear`).  The encoder is built only
when the VAE is given one (VDB_TEXT_ENCODER=1 in lib/cfg_helper.py): no app.py flow encodes text.
"""
import json
import os
import unicodedata

import torch
import torch.nn as nn

from lib.model_zoo.common.get_model import get_model, register
from .diffusion_utils import PackedMixin, bf16, f32, pack_epoch, require_cuda

symbol = 'optimus'

PAD_ID, BOS_ID, EOS_ID = 50257, 50258, 50259          # added after the 50257-entry GPT-2 vocabulary (optimus.py:30-34)
MAX_LENGTH = 30                                        # optimus.py:751
CACHE_SLOTS = 32                                       # KV-cache slots per (row, head), vdb_kv_decode_attention
D_HEAD = 64
DEFAULT_VOCAB = "lib/model_zoo/optimus_models/vocab/gpt2-vocab.json"
DEFAULT_BERT_VOCAB = "lib/model_zoo/optimus_models/vocab/bert-base-cased-vocab.txt"
BERT_PAD_ID = 0                                        # pad_sequence's padding_value (optimus.py:739); [PAD] in the vocabulary
BERT_MAX_PIECES = 510                                  # + [CLS] + [SEP] = the 512 rows of the position table


def _ops():
    from vdb200 import ops
    return ops


# ------------------------------------------------------------------------------------------------ module tree
class Conv1D(nn.Module):
    """GPT-2's transposed linear: y = x @ weight + bias, weight [in, out] (modeling_utils.Conv1D)."""

    def __init__(self, nf, nx):
        super().__init__()
        self.nf = nf
        self.weight = nn.Parameter(torch.empty(nx, nf).normal_(std=0.02))
        self.bias = nn.Parameter(torch.zeros(nf))


class Attention(nn.Module):
    def __init__(self, nx, n_ctx, n_head):
        super().__init__()
        self.register_buffer("bias", torch.tril(torch.ones(n_ctx, n_ctx)).view(1, 1, n_ctx, n_ctx))
        self.n_head = n_head
        self.c_attn = Conv1D(3 * nx, nx)
        self.c_proj = Conv1D(nx, nx)


class MLP(nn.Module):
    def __init__(self, n_state, nx):
        super().__init__()
        self.c_fc = Conv1D(n_state, nx)
        self.c_proj = Conv1D(nx, n_state)


class Block(nn.Module):
    def __init__(self, n_ctx, nx, n_head, eps):
        super().__init__()
        self.ln_1 = nn.LayerNorm(nx, eps=eps)
        self.attn = Attention(nx, n_ctx, n_head)
        self.ln_2 = nn.LayerNorm(nx, eps=eps)
        self.mlp = MLP(4 * nx, nx)


class GPT2Model_XX(nn.Module):
    def __init__(self, config):
        super().__init__()
        c = config
        self.wte = nn.Embedding(c["vocab_size"], c["n_embd"])
        self.wpe = nn.Embedding(c["n_positions"], c["n_embd"])
        self.h = nn.ModuleList([Block(c["n_ctx"], c["n_embd"], c["n_head"], c["layer_norm_epsilon"]) for _ in range(c["n_layer"])])
        self.ln_f = nn.LayerNorm(c["n_embd"], eps=c["layer_norm_epsilon"])
        self.latent_size = c.get("latent_size", 32)
        self.linear = nn.Linear(self.latent_size, c["hidden_size"] * c["n_layer"], bias=False)
        self.linear_emb = nn.Linear(self.latent_size, c["hidden_size"], bias=False)
        for m in self.modules():   # _init_weights of the reference (optimus_gpt2.py:855-866)
            if isinstance(m, (nn.Linear, nn.Embedding)):
                m.weight.data.normal_(mean=0.0, std=c.get("initializer_range", 0.02))


@register('optimus_gpt2_connector')
class GPT2ForLatentConnector_XX(PackedMixin, nn.Module):
    """Decoder with latent_as_gpt_emb = latent_as_gpt_memory = True (the reference's defaults, optimus_gpt2.py:1023-1033)."""

    def __init__(self, config, latent_size=32, latent_as_gpt_emb=True, latent_as_gpt_memory=True):
        super().__init__()
        if not (latent_as_gpt_emb and latent_as_gpt_memory):
            raise NotImplementedError("only latent_as_gpt_emb = latent_as_gpt_memory = True (the reference's decoder) is built")
        self.config = dict(config)
        self.transformer = GPT2Model_XX(self.config)
        self.lm_head = nn.Linear(self.config["n_embd"], self.config["vocab_size"], bias=False)
        self.lm_head.weight = self.transformer.wte.weight          # tie_weights (optimus_gpt2.py:1064-1069)
        self._states = {}

    def invalidate_packed(self):
        super().invalidate_packed()
        self._states = {}        # captured graphs read the packed weights

    def _pack(self):
        tr = self.transformer
        C = self.config["n_embd"]
        V = self.config["vocab_size"]
        vpad = (V + 63) // 64 * 64
        wte = torch.zeros(vpad, C, dtype=torch.bfloat16, device=tr.wte.weight.device)
        wte[:V] = tr.wte.weight.detach()
        layers = []
        for b in tr.h:
            layers.append(dict(
                ln1=(f32(b.ln_1.weight), f32(b.ln_1.bias)), ln2=(f32(b.ln_2.weight), f32(b.ln_2.bias)),
                attn_w=bf16(b.attn.c_attn.weight.t()), attn_b=f32(b.attn.c_attn.bias),
                proj_w=bf16(b.attn.c_proj.weight.t()), proj_b=f32(b.attn.c_proj.bias),
                fc_w=bf16(b.mlp.c_fc.weight.t()), fc_b=f32(b.mlp.c_fc.bias),
                mproj_w=bf16(b.mlp.c_proj.weight.t()), mproj_b=f32(b.mlp.c_proj.bias)))
        return dict(layers=layers, lnf=(f32(tr.ln_f.weight), f32(tr.ln_f.bias)), eps=tr.ln_f.eps, wte=wte, vocab=V,
                    wpe=f32(tr.wpe.weight), linear=bf16(tr.linear.weight), linear_emb=bf16(tr.linear_emb.weight),
                    heads=self.config["n_head"], width=C)

    # -------------------------------------------------------------- device state of one batch size
    def _state(self, n, device):
        st = self._states.get(n)
        if st is not None:
            return st
        pk = self.packed()
        C, L, H = pk["width"], len(pk["layers"]), pk["heads"]
        if C != H * D_HEAD:
            raise NotImplementedError(f"the decode kernels need d_head = {D_HEAD} (n_embd {C}, n_head {H})")
        kw = dict(device=device)
        st = dict(
            n=n, graphs={},
            zb=torch.empty(n, self.transformer.latent_size, dtype=torch.bfloat16, **kw),
            mem=torch.empty(n, L * C, dtype=torch.bfloat16, **kw),
            lemb=torch.empty(n, C, dtype=torch.float32, **kw),
            x=torch.empty(n, C, dtype=torch.bfloat16, **kw), x2=torch.empty(n, C, dtype=torch.bfloat16, **kw),
            h=torch.empty(n, C, dtype=torch.bfloat16, **kw), a=torch.empty(n, C, dtype=torch.bfloat16, **kw),
            qkv=torch.empty(n, 3 * C, dtype=torch.bfloat16, **kw), f=torch.empty(n, 4 * C, dtype=torch.bfloat16, **kw),
            logits=torch.empty(n, pk["wte"].shape[0], dtype=torch.float32, **kw),
            kc=torch.zeros(L, n, H, CACHE_SLOTS, D_HEAD, dtype=torch.bfloat16, **kw),
            vc=torch.zeros(L, n, H, CACHE_SLOTS, D_HEAD, dtype=torch.bfloat16, **kw),
            tokens=torch.full((n, CACHE_SLOTS), BOS_ID, dtype=torch.int32, **kw),
            step=torch.zeros(1, dtype=torch.int32, **kw),
            temperature=torch.ones(1, dtype=torch.float32, **kw),
            seed=torch.zeros(1, dtype=torch.int64, **kw),
            uniforms=torch.zeros(n, CACHE_SLOTS, dtype=torch.float32, **kw))
        self._states[n] = st
        return st

    def _prologue(self, st, z, pre_scale):
        """linear(z) -> memory slots, linear_emb(z) -> embedding offset, <BOS> input (optimus_gpt2.py:869-893, 941-951)."""
        ops, pk = _ops(), self.packed()
        ops.to_bf16(z.float().contiguous(), out=st["zb"])
        ops.gemm(st["zb"], pk["linear"], out=st["mem"], alpha=pre_scale)
        ops.gemm(st["zb"], pk["linear_emb"], out=st["lemb"], out_dtype=torch.float32, alpha=pre_scale)
        st["tokens"].fill_(BOS_ID)
        st["step"].zero_()
        ops.token_embed(st["tokens"], pk["wte"], pk["wpe"], st["lemb"], st["x"], pos_offset=1)

    def _blocks(self, st, logits):
        """the 12 pre-LN blocks, ln_f and the tied lm_head for the token at *step (optimus_gpt2.py:225-246, 1077-1082)"""
        ops, pk = _ops(), self.packed()
        C, H, eps = pk["width"], pk["heads"], pk["eps"]
        x, x2, h, a = st["x"], st["x2"], st["h"], st["a"]
        for li, ly in enumerate(pk["layers"]):
            ops.layernorm(x, *ly["ln1"], eps=eps, out=h)
            ops.gemm(h, ly["attn_w"], bias=ly["attn_b"], out=st["qkv"])
            ops.kv_decode_attention(st["qkv"], st["mem"][:, li * C:(li + 1) * C], st["kc"][li], st["vc"][li], st["step"], H, a,
                                    scale=D_HEAD ** -0.5)
            ops.gemm(a, ly["proj_w"], bias=ly["proj_b"], resid=x, out=x2)
            ops.layernorm(x2, *ly["ln2"], eps=eps, out=h)
            ops.gemm(h, ly["fc_w"], bias=ly["fc_b"], act=ops.ACT_GELU_TANH, out=st["f"])
            ops.gemm(st["f"], ly["mproj_w"], bias=ly["mproj_b"], resid=x2, out=x)
        ops.layernorm(x, *pk["lnf"], eps=eps, out=h)
        ops.gemm(h, pk["wte"], out=logits, out_dtype=torch.float32)

    def _token_step(self, st, use_uniforms):
        ops, pk = _ops(), self.packed()
        self._blocks(st, st["logits"])
        ops.sample_tokens(st["logits"], pk["vocab"], st["step"], st["tokens"], EOS_ID, temperature=st["temperature"],
                          seed=None if use_uniforms else st["seed"], uniforms=st["uniforms"] if use_uniforms else None,
                          max_len=MAX_LENGTH, wte=pk["wte"], wpe=pk["wpe"], emb_add=st["lemb"], x_next=st["x"])
        ops.add_int(st["step"], 1)

    @torch.no_grad()
    def sample_token_ids(self, z, temperature=1.0, uniforms=None, pre_scale=1.0, use_graph=True):
        """z [n, latent] -> int32 [n, 30] on the device: <BOS>, then sampled ids; every id after the first <EOS> is <EOS>.
        uniforms [n, 29] (optional) replaces the Philox draws (u of step k in column k)."""
        require_cuda(z, "optimus decode")
        n = z.shape[0]
        st = self._state(n, z.device)
        use_u = uniforms is not None
        if use_u:
            st["uniforms"][:, :MAX_LENGTH - 1].copy_(uniforms)
        else:
            # one 64-bit Philox key per decode from torch's CUDA generator: torch.manual_seed makes decodes reproducible
            st["seed"].copy_(torch.randint(0, 2 ** 62, (1,), device=z.device, dtype=torch.int64))
        st["temperature"].fill_(float(temperature))
        self._prologue(st, z, pre_scale)
        n0 = _ops().launch_count()
        self._token_step(st, use_u)                       # step 0 eager: packs, sizes the split-K workspace, warms modules
        self.last_step_launches = _ops().launch_count() - n0
        key = (pack_epoch(), use_u)
        g = st["graphs"].get(key) if use_graph else None
        if use_graph and g is None:
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):                     # capture records without executing: state stays at step 1
                self._token_step(st, use_u)
            st["graphs"] = {key: g}
        for _ in range(1, MAX_LENGTH - 1):
            if use_graph:
                g.replay()
            else:
                self._token_step(st, use_u)
        return st["tokens"][:, :MAX_LENGTH]

    @torch.no_grad()
    def logits_for(self, z, tokens, pre_scale=1.0):
        """Teacher forcing through the same launches: tokens int [n, L] (L <= 30, tokens[:, 0] = <BOS>) -> fp32 logits
        [n, L, vocab] of every position."""
        require_cuda(z, "optimus logits_for")
        ops, pk = _ops(), self.packed()
        n, L = tokens.shape
        if not 1 <= L <= MAX_LENGTH or bool((tokens[:, 0] != BOS_ID).any()):
            raise ValueError(f"logits_for: tokens must be [n, 1..{MAX_LENGTH}] starting with <BOS> ({BOS_ID})")
        st = self._state(n, z.device)
        forced = torch.full((n, CACHE_SLOTS), EOS_ID, dtype=torch.int32, device=z.device)
        forced[:, :L] = tokens.to(device=z.device, dtype=torch.int32)
        self._prologue(st, z, pre_scale)         # embeds <BOS> = forced[:, 0]
        st["tokens"].copy_(forced)
        vpad = pk["wte"].shape[0]
        out = torch.empty(n, L, vpad, dtype=torch.float32, device=z.device)
        for t in range(L):
            self._blocks(st, out[:, t, :])
            if t + 1 < L:
                ops.sample_tokens(None, 0, st["step"], st["tokens"], EOS_ID, forced=forced, max_len=MAX_LENGTH, wte=pk["wte"],
                                  wpe=pk["wpe"], emb_add=st["lemb"], x_next=st["x"])
                ops.add_int(st["step"], 1)
        return out[:, :, :pk["vocab"]]


# ------------------------------------------------------------------------------------------------ detokenizer
def _bytes_to_unicode():
    """GPT-2's reversible byte <-> printable-unicode table: printable Latin-1 bytes map to themselves, the other 68 bytes to
    code points 256 and up, in byte order."""
    keep = list(range(ord("!"), ord("~") + 1)) + list(range(ord("¡"), ord("¬") + 1)) + list(range(ord("®"), ord("ÿ") + 1))
    table, extra = {}, 0
    for b in range(256):
        if b in keep:
            table[b] = chr(b)
        else:
            table[b] = chr(256 + extra)
            extra += 1
    return table


@register('optimus_gpt2_tokenizer')
class GPT2Detokenizer(object):
    """Decoding half of the reference's GPT2Tokenizer with <PAD> <BOS> <EOS> added (tokenization_gpt2.py,
    tokenization_utils.py:701-815).  Needs only the vocabulary json; VDB_GPT2_VOCAB overrides its path."""
    added = {PAD_ID: "<PAD>", BOS_ID: "<BOS>", EOS_ID: "<EOS>"}

    def __init__(self, vocab_file=DEFAULT_VOCAB, merges_file=None, **kwargs):
        self.vocab_file = vocab_file
        self._decoder = None
        self._byte_decoder = {u: b for b, u in _bytes_to_unicode().items()}

    def _vocab(self):
        if self._decoder is None:
            path = os.environ.get("VDB_GPT2_VOCAB") or self.vocab_file
            if not os.path.exists(path):
                raise RuntimeError(f"GPT-2 vocabulary '{path}' is not available (cwd {os.getcwd()}): run from the tree that holds "
                                   f"{DEFAULT_VOCAB} or point VDB_GPT2_VOCAB at a gpt2-vocab.json")
            with open(path, encoding="utf-8") as fh:
                self._decoder = {v: k for k, v in json.load(fh).items()}
        return self._decoder

    def _bytes_text(self, pieces):
        return bytearray(self._byte_decoder[c] for c in "".join(pieces)).decode("utf-8", errors="replace")

    def decode(self, ids, clean_up_tokenization_spaces=True):
        """the reference's decode: byte-level runs decoded as UTF-8, every added token appended as ' ' + token"""
        dec = self._vocab()
        parts, run = [], []
        for i in ids:
            i = int(i)
            if i in self.added:
                if run:
                    parts.append(self._bytes_text(run))
                    run = []
                parts.append(" " + self.added[i])
            else:
                run.append(dec[i])
        if run:
            parts.append(self._bytes_text(run))
        text = "".join(parts)
        return self.clean_up_tokenization(text) if clean_up_tokenization_spaces else text

    @staticmethod
    def clean_up_tokenization(s):
        return (s.replace(" .", ".").replace(" ?", "?").replace(" !", "!").replace(" ,", ",").replace(" ' ", "'")
                .replace(" n't", "n't").replace(" 'm", "'m").replace(" do not", " don't").replace(" 's", "'s")
                .replace(" 've", "'ve").replace(" 're", "'re"))

    def sentence(self, ids):
        """optimus.py:758-760: decode, split on whitespace, drop the first and last word (the <BOS> / <EOS> words)"""
        return " ".join(self.decode(ids, clean_up_tokenization_spaces=True).split()[1:-1])


def truncate_at_eos(row):
    """ids up to and including the first <EOS> (the reference stops sampling there)"""
    row = [int(v) for v in row]
    return row[:row.index(EOS_ID) + 1] if EOS_ID in row else row


# ------------------------------------------------------------------------------------------------ BERT encoder
class _Linear(nn.Linear):
    def __init__(self, n_in, n_out, bias=True, std=0.02):
        super().__init__(n_in, n_out, bias=bias)
        self.weight.data.normal_(std=std)                  # _init_weights of the reference (optimus_bert.py:1371-1381)
        if bias:
            self.bias.data.zero_()


class BertEmbeddings(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.word_embeddings = nn.Embedding(c["vocab_size"], c["hidden_size"], padding_idx=0)
        self.position_embeddings = nn.Embedding(c["max_position_embeddings"], c["hidden_size"])
        self.token_type_embeddings = nn.Embedding(c["type_vocab_size"], c["hidden_size"])
        self.LayerNorm = nn.LayerNorm(c["hidden_size"], eps=c["layer_norm_eps"])
        for e in (self.word_embeddings, self.position_embeddings, self.token_type_embeddings):
            e.weight.data.normal_(std=c.get("initializer_range", 0.02))


class BertSelfAttention(nn.Module):
    def __init__(self, c):
        super().__init__()
        C, std = c["hidden_size"], c.get("initializer_range", 0.02)
        self.query, self.key, self.value = _Linear(C, C, std=std), _Linear(C, C, std=std), _Linear(C, C, std=std)


class BertSelfOutput(nn.Module):
    def __init__(self, c, n_in):
        super().__init__()
        self.dense = _Linear(n_in, c["hidden_size"], std=c.get("initializer_range", 0.02))
        self.LayerNorm = nn.LayerNorm(c["hidden_size"], eps=c["layer_norm_eps"])


class BertAttention(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.self = BertSelfAttention(c)
        self.output = BertSelfOutput(c, c["hidden_size"])


class BertIntermediate(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.dense = _Linear(c["hidden_size"], c["intermediate_size"], std=c.get("initializer_range", 0.02))


class BertLayer(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.attention = BertAttention(c)
        self.intermediate = BertIntermediate(c)
        self.output = BertSelfOutput(c, c["intermediate_size"])     # BertOutput: dense + LayerNorm, the same tree


class BertEncoder(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.layer = nn.ModuleList([BertLayer(c) for _ in range(c["num_hidden_layers"])])


class BertPooler(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.dense = _Linear(c["hidden_size"], c["hidden_size"], std=c.get("initializer_range", 0.02))


@register('optimus_bert_connector')
class BertForLatentConnector_XX(PackedMixin, nn.Module):
    """optimus_bert.py:1349-1439 as optimus_vae_next.encode uses it: post-LN BERT (exact-erf GELU), the tanh pooler on [CLS],
    and `linear` (hidden -> 2 * latent, no bias) whose first half is the latent mean."""

    def __init__(self, config, latent_size=32):
        super().__init__()
        self.config = dict(config)
        c = self.config
        if c.get("hidden_act", "gelu") != "gelu":
            raise NotImplementedError(f"hidden_act {c['hidden_act']!r}: only BERT's exact-erf 'gelu' is built")
        self.latent_size = latent_size
        self.embeddings = BertEmbeddings(c)
        self.encoder = BertEncoder(c)
        self.pooler = BertPooler(c)
        self.linear = _Linear(c["hidden_size"], 2 * latent_size, bias=False, std=c.get("initializer_range", 0.02))

    def _pack(self):
        c = self.config
        C, H = c["hidden_size"], c["num_attention_heads"]
        if C != H * D_HEAD or C % 128:
            raise NotImplementedError(f"the encode kernels need d_head = {D_HEAD} and a width that is a multiple of 128 "
                                      f"(hidden_size {C}, {H} heads)")
        e = self.embeddings
        layers = []
        for ly in self.encoder.layer:
            a = ly.attention
            wo = a.output.dense.weight.detach().float()
            layers.append(dict(
                wqk=bf16(torch.cat([a.self.query.weight.detach(), a.self.key.weight.detach()], 0)),
                bqk=f32(torch.cat([a.self.query.bias.detach(), a.self.key.bias.detach()], 0)),
                wv=bf16(a.self.value.weight),
                # softmax rows sum to 1 over the kept keys too, so P(V + 1 b_v^T) = PV + b_v: the V bias moves through the output
                wo=bf16(wo), bo=(a.output.dense.bias.detach().float() + wo @ a.self.value.bias.detach().float()).contiguous(),
                ln1=(f32(a.output.LayerNorm.weight), f32(a.output.LayerNorm.bias)),
                w1=bf16(ly.intermediate.dense.weight), b1=f32(ly.intermediate.dense.bias),
                w2=bf16(ly.output.dense.weight), b2=f32(ly.output.dense.bias),
                ln2=(f32(ly.output.LayerNorm.weight), f32(ly.output.LayerNorm.bias))))
        return dict(layers=layers, word=f32(e.word_embeddings.weight), pos=f32(e.position_embeddings.weight),
                    type0=f32(e.token_type_embeddings.weight[0]), emb_ln=(f32(e.LayerNorm.weight), f32(e.LayerNorm.bias)),
                    eps=float(c["layer_norm_eps"]), pool_w=bf16(self.pooler.dense.weight), pool_b=f32(self.pooler.dense.bias),
                    mu_w=bf16(self.linear.weight[:self.latent_size]), heads=H, width=C)

    @torch.no_grad()
    def encode_ids(self, ids, lengths, n_keys):
        """ids int32 [n, Lp] on the device (rows padded with 0 to Lp, a multiple of 8), lengths int32 [n] on the device (the
        ids of row b before its padding, [CLS] .. [SEP]), n_keys = max(lengths) on the host -> fp32 z_mu [n, latent].
        About 8 launches per layer plus 3."""
        require_cuda(ids, "optimus encode")
        ops, pk = _ops(), self.packed()
        n, Lp = ids.shape
        C, H, eps = pk["width"], pk["heads"], pk["eps"]
        if Lp % 8 or not 1 <= n_keys <= Lp:
            raise ValueError(f"encode_ids: padded length {Lp} must be a multiple of 8 and hold the {n_keys} keys")
        x = ops.bert_embed_ln(ids, pk["word"], pk["pos"], pk["type0"], *pk["emb_ln"], eps=eps)     # [n*Lp, C]
        o = torch.zeros(n * Lp, C, dtype=torch.bfloat16, device=ids.device)      # rows past n_keys are never written
        for ly in pk["layers"]:
            qk = ops.gemm(x, ly["wqk"], bias=ly["bqk"])                           # [n*Lp, 2C]: q | k
            vt = ops.gemm(ly["wv"], x)                                            # [C, n*Lp] = V^T (bias folded into bo)
            ops.attention(qk, qk, vt, o, n, H, n_keys, n_keys, D_HEAD, scale=D_HEAD ** -0.5, q_col0=0, k_col0=C,
                          q_bstride=Lp, kv_bstride=Lp, kv_len=lengths)
            h = ops.layernorm(ops.gemm(o, ly["wo"], bias=ly["bo"], resid=x), *ly["ln1"], eps=eps)
            f = ops.gemm(h, ly["w1"], bias=ly["b1"], act=ops.ACT_GELU)
            x = ops.layernorm(ops.gemm(f, ly["w2"], bias=ly["b2"], resid=h), *ly["ln2"], eps=eps)
        cls = x.view(n, Lp * C)[:, :C]                                            # the [CLS] rows: lda = Lp * C
        pooled = ops.gemm(cls, pk["pool_w"], bias=pk["pool_b"], act=ops.ACT_TANH)
        return ops.gemm(pooled, pk["mu_w"], out_dtype=torch.float32)


def _is_bert_whitespace(ch):
    return ch in " \t\n\r" or unicodedata.category(ch) == "Zs"


def _is_bert_control(ch):
    return ch not in "\t\n\r" and unicodedata.category(ch).startswith("C")


def _is_bert_punctuation(ch):
    cp = ord(ch)
    return 33 <= cp <= 47 or 58 <= cp <= 64 or 91 <= cp <= 96 or 123 <= cp <= 126 or unicodedata.category(ch).startswith("P")


_CJK_RANGES = ((0x4E00, 0x9FFF), (0x3400, 0x4DBF), (0x20000, 0x2A6DF), (0x2A700, 0x2B73F), (0x2B740, 0x2B81F),
               (0x2B820, 0x2CEAF), (0xF900, 0xFAFF), (0x2F800, 0x2FA1F))


def _is_cjk(ch):
    cp = ord(ch)
    return any(lo <= cp <= hi for lo, hi in _CJK_RANGES)


@register('optimus_bert_tokenizer')
class BertTokenizer(object):
    """What optimus_vae_next.encode uses of the reference's BertTokenizer (tokenization_bert.py, tokenization_utils.py:576-625)
    with do_lower_case = False: text cleaning (NUL, U+FFFD and control characters dropped, whitespace -> ' '), CJK characters
    split out, whitespace and punctuation splits, accents kept, then greedy longest-match-first WordPiece ('##' continuations,
    [UNK] for a word that cannot be covered or is longer than 100 characters).  Needs only the vocabulary file (one piece per
    line, the line number is the id); VDB_BERT_VOCAB overrides its path.

    A text that is all whitespace (but not empty) comes out of the reference as ONE special token picked by Python's set order
    of the special-token strings, which changes with the hash seed of the process; here it is always [UNK]."""
    max_input_chars_per_word = 100

    def __init__(self, vocab_file=DEFAULT_BERT_VOCAB, do_lower_case=False, **kwargs):
        if do_lower_case:
            raise NotImplementedError("only the cased tokenizer of the Optimus encoder (do_lower_case = False) is built")
        self.vocab_file = vocab_file
        self._vocab_map = None

    def vocab(self):
        if self._vocab_map is None:
            path = os.environ.get("VDB_BERT_VOCAB") or self.vocab_file
            if not os.path.exists(path):
                raise RuntimeError(f"BERT vocabulary '{path}' is not available (cwd {os.getcwd()}): run from the tree that holds "
                                   f"{DEFAULT_BERT_VOCAB} or point VDB_BERT_VOCAB at a bert-base-cased-vocab.txt")
            with open(path, encoding="utf-8") as fh:
                self._vocab_map = {line.rstrip("\n"): i for i, line in enumerate(fh)}
        return self._vocab_map

    def _id(self, piece):
        v = self.vocab()
        return v.get(piece, v["[UNK]"])

    @property
    def cls_token_id(self):
        return self._id("[CLS]")

    @property
    def sep_token_id(self):
        return self._id("[SEP]")

    @staticmethod
    def basic_tokenize(text):
        out = []
        for ch in text:
            if ch == "\x00" or ch == "\ufffd" or _is_bert_control(ch):
                continue
            if _is_bert_whitespace(ch):
                out.append(" ")
            elif _is_cjk(ch):
                out.append(" " + ch + " ")
            else:
                out.append(ch)
        words = []
        for word in "".join(out).split():
            cur = ""
            for ch in word:
                if _is_bert_punctuation(ch):
                    if cur:
                        words.append(cur)
                        cur = ""
                    words.append(ch)
                else:
                    cur += ch
            if cur:
                words.append(cur)
        return words

    def wordpiece(self, word):
        if len(word) > self.max_input_chars_per_word:
            return ["[UNK]"]
        vocab = self.vocab()
        pieces, start = [], 0
        while start < len(word):
            for end in range(len(word), start, -1):
                piece = word[start:end] if start == 0 else "##" + word[start:end]
                if piece in vocab:
                    break
            else:
                return ["[UNK]"]
            pieces.append(piece)
            start = end
        return pieces

    def tokenize(self, text):
        if text and not text.strip():
            return ["[UNK]"]
        return [p for w in self.basic_tokenize(text) for p in self.wordpiece(w)]

    def convert_tokens_to_ids(self, pieces):
        return [self._id(p) for p in pieces]

    def encode_sentences(self, sentences, max_length=77):
        """optimus.py:729-738: lower-case, tokenize, keep the first max_length pieces, add [CLS] .. [SEP] -> list of id lists"""
        cls, sep = self.cls_token_id, self.sep_token_id
        return [[cls] + self.convert_tokens_to_ids(self.tokenize(s.lower())[:max_length]) + [sep] for s in sentences]


# ------------------------------------------------------------------------------------------------ the VAE surface
@register('optimus_vae_next')
class optimus_vae_next(nn.Module):
    def __init__(self, encoder=None, decoder=None, tokenizer_encoder=None, tokenizer_decoder=None, args=None):
        super().__init__()
        if encoder is not None:
            self.encoder = encoder if isinstance(encoder, nn.Module) else get_model()(encoder, verbose=False)
            self.tokenizer_encoder = tokenizer_encoder if isinstance(tokenizer_encoder, BertTokenizer) \
                else get_model()(tokenizer_encoder, verbose=False)
        self.decoder = decoder if isinstance(decoder, nn.Module) else get_model()(decoder, verbose=False)
        self.tokenizer_decoder = tokenizer_decoder if isinstance(tokenizer_decoder, GPT2Detokenizer) \
            else get_model()(tokenizer_decoder, verbose=False)
        self.args = args
        self.nz = (args or {}).get("latent_size", self.decoder.transformer.latent_size)
        self.eos_token_id, self.pad_token_id = EOS_ID, PAD_ID

    def get_device(self):
        return self.decoder.transformer.linear.weight.device

    @torch.no_grad()
    def encode(self, text, max_length=77):
        """optimus.py:729-743: sentences (a list of str; a single str is one sentence) -> fp32 z_mu [n, latent] on the device.
        Each sentence keeps its first max_length word pieces; the rows are padded to the longest, rounded up to 8."""
        if getattr(self, "encoder", None) is None:
            raise NotImplementedError("Optimus text encoding (the BERT encoder, vae_encode(x, 'text')) is not built in this VAE: "
                                      "construct it with an encoder (VDB_TEXT_FLOWS=1 VDB_TEXT_ENCODER=1 in the config bank)")
        if not 0 <= max_length <= BERT_MAX_PIECES:
            raise ValueError(f"max_length {max_length}: at most {BERT_MAX_PIECES} pieces fit the 512 positions with [CLS] and [SEP]")
        sentences = [text] if isinstance(text, str) else list(text)
        if not sentences:
            raise ValueError("encode: no sentences")
        rows = self.tokenizer_encoder.encode_sentences(sentences, max_length)
        n, keys = len(rows), max(len(r) for r in rows)
        Lp = (keys + 7) // 8 * 8                         # the attention's per-item row stride must stay 16-byte aligned
        host = torch.full((n * Lp + n,), BERT_PAD_ID, dtype=torch.int32)
        for b, r in enumerate(rows):
            host[b * Lp:b * Lp + len(r)] = torch.tensor(r, dtype=torch.int32)
            host[n * Lp + b] = len(r)
        dev = self.encoder.linear.weight.device
        require_cuda(self.encoder.linear.weight, "optimus encode")
        buf = host.to(dev)                               # ids and lengths in one host-to-device copy
        return self.encoder.encode_ids(buf[:n * Lp].view(n, Lp), buf[n * Lp:], keys)

    @torch.no_grad()
    def decode_tokens(self, z, temperature=1.0, uniforms=None, pre_scale=1.0, use_graph=True):
        """z [n, latent] -> int64 numpy-ready CPU tensor [n, 30] (one device-to-host copy)"""
        return self.decoder.sample_token_ids(z, temperature, uniforms, pre_scale, use_graph).to("cpu", torch.int64)

    @torch.no_grad()
    def logits_for(self, z, tokens, pre_scale=1.0):
        return self.decoder.logits_for(z, tokens, pre_scale)

    @torch.no_grad()
    def decode(self, z, temperature=1.0, pre_scale=1.0):
        """optimus.py:745-763: one sentence per latent row"""
        ids = self.decode_tokens(z, temperature, pre_scale=pre_scale)
        return [self.tokenizer_decoder.sentence(truncate_at_eos(r)) for r in ids.tolist()]
