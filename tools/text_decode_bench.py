"""Optimus text decode at FULL size on one GPU (app.py's i2t / t2t shape: n = 4 latents, 30 tokens): time of one decode(), of one
token step in the replayed CUDA graph, launches per step, and the weight bytes a token step streams against the HBM peak; then
the whole inference_i2t-shaped flow (50-step text-latent DDIM with CFG on a CLIP-image context, then vae_decode(x, 'text')).
Random-init weights and a synthetic context.  Without VDB_GPT2_VOCAB the ids are turned into strings through a stand-in vocabulary
written to a temporary directory (the detokenizer's cost does not depend on the strings).
    python tools/text_decode_bench.py            (sets VDB_TEXT_FLOWS=1 itself)"""
import json
import os
import subprocess
import sys
import tempfile
import time

os.environ["VDB_TEXT_FLOWS"] = "1"
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
if "VDB_GPT2_VOCAB" not in os.environ:
    os.environ["VDB_GPT2_VOCAB"] = os.path.join(tempfile.mkdtemp(), "gpt2-vocab.json")
    json.dump({f"\u0120w{i}": i for i in range(50257)}, open(os.environ["VDB_GPT2_VOCAB"], "w"))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "versatile-diffusion_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from lib.cfg_helper import model_cfg_bank  # noqa: E402
from lib.model_zoo import get_model  # noqa: E402
from lib.model_zoo.ddim import DDIMSampler  # noqa: E402
from lib.model_zoo.optimus import MAX_LENGTH  # noqa: E402

dev = torch.device("cuda", 0)
cfg = model_cfg_bank()('vd_four_flow_v1-0')
cfg.args.ctx_cfg_list = []
cfg.args.vae_cfg_list = [v for v in cfg.args.vae_cfg_list if v[0] == "text"]
torch.manual_seed(0)
t0 = time.time()
with torch.device(dev):
    net = get_model()(cfg, verbose=False)
g = torch.Generator(device=dev).manual_seed(1)
with torch.no_grad():
    for _, p in net.named_parameters():
        if p.ndim == 1 or not bool(p.any()):
            if p.ndim == 1 and p.shape[0] > 0 and bool((p == 1).all()):
                continue
            p.normal_(0.0, 0.02, generator=g)
net.eval()
net.to(dev)
vae = net.vae["text"]
dec = vae.decoder
print(f"built in {time.time() - t0:.1f} s", flush=True)

n = 4
gq = torch.Generator().manual_seed(3)
z = torch.randn(n, 768, generator=gq).to(dev)
ev = lambda: torch.cuda.Event(enable_timing=True)


def median_ms(fn, reps, pre=None):
    ts = []
    for _ in range(reps):
        if pre is not None:
            pre()
        e0, e1 = ev(), ev()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))


with torch.no_grad():
    for _ in range(3):
        vae.decode(z)
    torch.cuda.synchronize()
    ms_decode = median_ms(lambda: vae.decode(z), 25)                  # ids to the host + detokenization included
    ms_tokens = median_ms(lambda: vae.decode_tokens(z), 25)
    st = dec._states[n]
    graph = next(iter(st["graphs"].values()))

    def replay_all():
        for _ in range(1, MAX_LENGTH - 1):
            graph.replay()
    def rewind():                # back to step 1 with no finished row, so every replay samples all rows
        st["step"].fill_(1)
        st["tokens"][:, 1:].fill_(0)
    ms_replay = median_ms(replay_all, 25, pre=rewind)
    us_step = ms_replay / (MAX_LENGTH - 2) * 1e3
    pk = dec.packed()
    wbytes = sum(ly[k].numel() * ly[k].element_size() for ly in pk["layers"] for k in ("attn_w", "proj_w", "fc_w", "mproj_w"))
    wbytes += pk["vocab"] * pk["width"] * 2                              # lm_head (tied wte), bf16
    sentences = vae.decode(z)

    g2 = torch.Generator().manual_seed(5)
    c = (torch.randn(n, 257, 768, generator=g2) * 0.5).to(dev)
    u = torch.zeros(n, 257, 768, device=dev)
    S = DDIMSampler(net)
    kw = dict(steps=50, shape=[n, 768], x_info={"type": "text"},
              c_info={"type": "image", "conditioning": c, "unconditional_conditioning": u, "unconditional_guidance_scale": 7.5},
              verbose=False, eta=0.)

    def i2t():
        x, _ = S.sample(**kw)
        return net.vae_decode(x, which='text', temperature=1)
    for _ in range(2):
        i2t()
    torch.cuda.synchronize()
    ms_ddim = median_ms(lambda: S.sample(**kw), 5)
    ms_i2t = median_ms(i2t, 5)

peak, peak_src = 6571.9, "fallback"
try:
    peak, peak_src = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "MEASURED_PEAKS.json"
except Exception:
    pass
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except Exception as ex:
    power = f"unavailable ({type(ex).__name__})"
print(json.dumps({
    "workload": "Optimus GPT-2 text decode, full size (12 x 768, vocab 50260), n = 4 latents x 30 tokens, bf16 weights, random init",
    "gpu": torch.cuda.get_device_name(0), "power_limit": power,
    "ms_per_decode": round(ms_decode, 3), "ms_per_decode_tokens_only": round(ms_tokens, 3),
    "us_per_token_step_graph": round(us_step, 2), "launches_per_step": dec.last_step_launches,
    "weight_bytes_per_step": wbytes, "step_weight_gbs": round(wbytes / us_step / 1e3, 1), "hbm_peak_gbs": peak,
    "hbm_peak_source": peak_src, "frac_of_hbm_peak": round(wbytes / us_step / 1e3 / peak, 3),
    "ddim50_text_ms": round(ms_ddim, 2), "i2t_ddim50_plus_decode_ms": round(ms_i2t, 2),
    "sample_sentence": sentences[0][:80]}))
