"""Optimus text VAE (decoder side) on vdb200 kernels — reference lib/model_zoo/optimus.py:17-52, 645-763 and
optimus_models/optimus_gpt2.py:99-246, 813-1112.

`optimus_vae_next.decode(z)` turns text latents [n, 768] into sentences like the reference's: a GPT-2 decoder that sees the
latent twice — `linear_emb(z)` added to every input embedding and one slice of `linear(z)` per layer used as a one-slot past
key AND value — samples up to 30 tokens from `<BOS>`.  The reference re-runs the whole prefix for every token and samples on
the host; here every layer keeps a bf16 KV cache, the sampler runs on the device, and the token step is one captured CUDA
graph replayed 28 times, so the host sees only the final [n, 30] token ids.

The module tree keeps the reference's state_dict keys and shapes (`decoder.transformer.*`, `decoder.lm_head` tied to
`wte`); only the decoder is built.  The BERT encoder (`vae_encode(., 'text')`) is used by no app.py flow.
"""
import json
import os

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


# ------------------------------------------------------------------------------------------------ the VAE surface
@register('optimus_vae_next')
class optimus_vae_next(nn.Module):
    def __init__(self, encoder=None, decoder=None, tokenizer_encoder=None, tokenizer_decoder=None, args=None):
        super().__init__()
        self.decoder = decoder if isinstance(decoder, nn.Module) else get_model()(decoder, verbose=False)
        self.tokenizer_decoder = tokenizer_decoder if isinstance(tokenizer_decoder, GPT2Detokenizer) \
            else get_model()(tokenizer_decoder, verbose=False)
        self.args = args
        self.nz = (args or {}).get("latent_size", self.decoder.transformer.latent_size)
        self.eos_token_id, self.pad_token_id = EOS_ID, PAD_ID

    def get_device(self):
        return self.decoder.transformer.linear.weight.device

    def encode(self, text, max_length=77):
        raise NotImplementedError("Optimus text encoding (the BERT encoder, vae_encode(x, 'text')) is not built: no app.py flow "
                                  "uses it; only decode() is available")

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
