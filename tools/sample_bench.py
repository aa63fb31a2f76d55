"""Device sampler cost: the kernel alone, and the sampled decode step against the greedy one.

    python tools/sample_bench.py [--iters 200] [--steps 32] [--out profiles/sample_bench.json]

1. cl_op_sample at B = 1, 8, 64, 128 rows of V = 128 256 fp32 logits with the Ollama defaults (temperature 0.8, top_k 40,
   top_p 0.9, repeat_penalty 1.1 over a 64-id window): mean of `iters` CUDA-event-timed launches that rotate over copies
   of the logits larger than the 126 MB L2.
2. Llama-3-8B (synthetic weights), B = 8 / 64 / 128 sequences after a 128-token prompt: device ms per step of
   cl_decode_greedy_batch against cl_decode_sample_batch (Ollama defaults), alternated, two rounds each.
The card's name and power limit are read in the same run and written beside the numbers.
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
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
        sps = [eng.ollama_default_sampling(seed=b) for b in range(B)]
        wins = [rng.integers(0, V, 64) for _ in range(B)]
        _, ms = eng.op_sample(x, sps, wins, [0] * B, iters=iters)
        out[B] = ms * 1e3
        print(f"sampler kernel B={B:4d} V={V}: {ms * 1e3:8.1f} us", flush=True)
    return out


def step_times(steps):
    out = {}
    with eng.Engine(preset="llama3-8b", seed=1234, max_batch=128) as e:
        V = e.cfg["vocab_size"]
        for B in (8, 64, 128):
            prompts = [np.array([(i * 7919 + 104729 * b) % (V - 1000) + 500 for i in range(128)], np.int32) for b in range(B)]
            sps = [eng.ollama_default_sampling(seed=b) for b in range(B)]
            res = {"greedy": [], "sampled": []}
            for rnd in range(2):
                for mode in ("greedy", "sampled"):
                    seqs = [e.seq_create() for _ in range(B)]
                    first = []
                    for s, p in zip(seqs, prompts):
                        lg = e.prefill(s, p)
                        first.append(int(lg.argmax()))
                    if mode == "greedy":
                        _, ms = e.decode_greedy_batch(seqs, first, steps)
                    else:
                        _, ms = e.decode_sample_batch(seqs, first, sps, [1] * B, steps)
                    res[mode].append(ms / steps)
                    for s in seqs:
                        e.seq_free(s)
            g, s_ = min(res["greedy"]), min(res["sampled"])
            out[B] = {"greedy_ms_per_step": res["greedy"], "sampled_ms_per_step": res["sampled"], "overhead_pct": 100 * (s_ / g - 1)}
            print(f"decode step B={B:4d}: greedy {g:.3f} ms  sampled {s_:.3f} ms  (+{100 * (s_ / g - 1):.2f} %)  runs {res}", flush=True)
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    c = card()
    print("card:", c, flush=True)
    res = {"card (name, power limit, max SM clock)": c, "kernel_us": kernel_times(a.iters), "step": step_times(a.steps)}
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))
