"""Optimus BERT text encode at FULL size on one GPU: median CUDA-event time of one net.vae_encode(sentences, 'text') call (host
tokenization, the one id copy and the ~100 launches of the 12-layer encoder) and of the device part alone (encode_ids), for
n = 1, 4, 8 sentences of 79 tokens ([CLS] + 77 word pieces + [SEP], the longest encode() builds); launches per call; the bf16
weights one call streams.  Random-init weights.  Without VDB_BERT_VOCAB the sentences are words of a stand-in vocabulary written
to a temporary directory (WordPiece's cost does not depend on the vocabulary's content).  One JSON line per batch size, with the
card's name and power limit read in the same run.
    python tools/text_encode_bench.py [--reps 60]      (sets VDB_TEXT_FLOWS=1 VDB_TEXT_ENCODER=1 itself)"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

os.environ["VDB_TEXT_FLOWS"] = "1"
os.environ["VDB_TEXT_ENCODER"] = "1"
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
WORDS = [f"w{i}" for i in range(2000)]
if "VDB_BERT_VOCAB" not in os.environ:
    os.environ["VDB_BERT_VOCAB"] = os.path.join(tempfile.mkdtemp(), "bert-vocab.txt")
    lines = [f"[unused{i}]" for i in range(28996)]
    lines[0], lines[100], lines[101], lines[102], lines[103] = "[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]"
    lines[1000:1000 + len(WORDS)] = WORDS
    open(os.environ["VDB_BERT_VOCAB"], "w").write("\n".join(lines) + "\n")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "versatile-diffusion_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from lib.cfg_helper import model_cfg_bank  # noqa: E402
from lib.model_zoo import get_model  # noqa: E402
from vdb200 import ops  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=60)
opt = ap.parse_args()

dev = torch.device("cuda", 0)
cfg = model_cfg_bank()("optimus_v1")
torch.manual_seed(0)
with torch.device(dev):
    vae = get_model()(cfg, verbose=False)
vae.eval().to(dev)
enc = vae.encoder
ev = lambda: torch.cuda.Event(enable_timing=True)


def median_ms(fn, reps):
    ts = []
    for _ in range(reps):
        e0, e1 = ev(), ev()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(np.percentile(ts, 10)), float(np.percentile(ts, 90))


try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except Exception as ex:
    power = f"unavailable ({type(ex).__name__})"
pk = enc.packed()
wbytes = sum(ly[k].numel() * 2 for ly in pk["layers"] for k in ("wqk", "wv", "wo", "w1", "w2")) + pk["pool_w"].numel() * 2 \
    + pk["mu_w"].numel() * 2
rng = np.random.RandomState(0)
with torch.no_grad():
    for n in (1, 4, 8):
        sents = [" ".join(rng.choice(WORDS, 77)) for _ in range(n)]
        rows = vae.tokenizer_encoder.encode_sentences(sents)
        assert all(len(r) == 79 for r in rows), [len(r) for r in rows]
        for _ in range(5):                                  # warm-up: module loads, packing, split-K workspace
            vae.encode(sents)
        torch.cuda.synchronize()
        n0 = ops.launch_count()
        vae.encode(sents)
        launches = ops.launch_count() - n0
        ms_call = median_ms(lambda: vae.encode(sents), opt.reps)
        Lp = 80
        host = torch.zeros(n * Lp + n, dtype=torch.int32)
        for b, r in enumerate(rows):
            host[b * Lp:b * Lp + len(r)] = torch.tensor(r, dtype=torch.int32)
            host[n * Lp + b] = len(r)
        buf = host.to(dev)
        ms_dev = median_ms(lambda: enc.encode_ids(buf[:n * Lp].view(n, Lp), buf[n * Lp:], 79), opt.reps)
        us = ms_dev[0] * 1e3
        print(json.dumps({
            "workload": f"Optimus BERT text encode, full size (12 x 768, 12 heads), n = {n} sentences x 79 tokens, bf16 weights, "
                        "random init",
            "gpu": torch.cuda.get_device_name(0), "power_limit": power, "reps": opt.reps,
            "ms_per_vae_encode_median": round(ms_call[0], 4), "ms_per_vae_encode_p10_p90": [round(ms_call[1], 4), round(ms_call[2], 4)],
            "ms_device_encode_ids_median": round(ms_dev[0], 4), "ms_device_encode_ids_p10_p90": [round(ms_dev[1], 4), round(ms_dev[2], 4)],
            "launches_per_call": launches, "us_per_launch_device": round(us / launches, 2),
            "weight_bytes_per_call": wbytes, "weight_gbs_device": round(wbytes / us / 1e3, 1)}), flush=True)
