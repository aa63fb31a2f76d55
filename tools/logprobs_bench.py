"""Cost of token log-probabilities: the kernel against the device sampler, and the scheduler's throughput with and without.

    python tools/logprobs_bench.py [--iters 200] [--waves 2] [--out profiles/logprobs_bench.json]

1. cl_op_logprobs (top_n 0 and 20) and cl_op_sample (Ollama defaults) at B = 1, 8, 64, 128 rows of V = 128 256 fp32
   logits: mean of `iters` CUDA-event-timed launches that rotate over copies of the logits larger than the 126 MB L2.
2. tools/sched_probe.py at max_batch 64 and 128 (Llama-3-8B synthetic weights, 146-token prompts, 128 tokens, greedy,
   as many closed-loop clients as max_batch) with every request at top_logprobs 5 against none, alternated twice in one
   process per max_batch.
The card's name and power limit are read in the same run and written beside the numbers.
"""
import argparse
import json
import re
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from crowdllama_b200 import engine as eng  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def kernel_times(iters):
    V = 128256
    rng = np.random.default_rng(0)
    out = {}
    for B in (1, 8, 64, 128):
        x = (rng.standard_normal((B, V)) * 3.0).astype(np.float32)
        chosen = rng.integers(0, V, B).astype(np.int32)
        row = {}
        for n in (0, 20):
            row[f"logprobs_top{n}"] = eng.op_logprobs(x, chosen, n, iters=iters)[3] * 1e3
        sps = [eng.ollama_default_sampling(seed=b) for b in range(B)]
        row["sample"] = eng.op_sample(x, sps, [rng.integers(0, V, 64) for _ in range(B)], [0] * B, iters=iters)[1] * 1e3
        out[B] = row
        print(f"B={B:4d} V={V}: logprobs top_n 0 {row['logprobs_top0']:7.1f} us  top_n 20 {row['logprobs_top20']:7.1f} us  "
              f"sampler {row['sample']:7.1f} us", flush=True)
    return out


def sched(max_batch, waves):
    cmd = [sys.executable, str(ROOT / "tools" / "sched_probe.py"), "--max-batch", str(max_batch), "--conc", str(max_batch),
           "--waves", str(waves), "--gen", "128", "--top-logprobs", "none,5,none,5"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode:
        raise SystemExit(r.stderr[-3000:])
    lines = [l for l in r.stdout.splitlines() if "req/s" in l][4:]           # the first four are the warm-up runs
    res = {"none": [], "5": []}
    for l in lines:
        print(f"max_batch={max_batch} {l}", flush=True)
        top = re.search(r"top_logprobs\s+(\S+)", l).group(1)
        res[top].append({"req_per_s": float(re.search(r"([\d.]+) req/s", l).group(1)),
                         "decode_ms_per_step": float(re.search(r"decode ([\d.]+) ms/step", l).group(1))})
    a, b = (max(x["req_per_s"] for x in res[k]) for k in ("none", "5"))
    print(f"max_batch={max_batch}: top_logprobs 5 costs {100 * (1 - b / a):.2f} % of req/s (best of two each)", flush=True)
    return {"runs": res, "cost_pct": 100 * (1 - b / a)}


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--waves", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    c = card()
    print("card:", c, flush=True)
    res = {"card (name, power limit, max SM clock)": c, "kernel_us": kernel_times(a.iters),
           "sched": {mb: sched(mb, a.waves) for mb in (64, 128)}}
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))
