"""Scheduler probe: closed-loop clients straight on the C-ABI (no sockets, no gateway), scheduler accounting per run.

    python tools/sched_probe.py [--max-batch 32] [--gen 256] [--prompt 146] [--conc 32,33,64] [--waves 6] [--sampling greedy|ollama]
                                [--top-logprobs none,5]

--sampling ollama sends every request with the Ollama defaults (temperature 0.8, top_k 40, top_p 0.9, repeat_penalty 1.1
over 64 tokens; seed = request index); CL_SCHED_DEVICE_SAMPLE=0/1 in the environment picks the host or the device sampler.
--top-logprobs takes a comma list of `none` (no log-probabilities) and 0..20 (every request asks for the log-probabilities
of its tokens with that many alternatives); the values are run one after the other at every concurrency, in list order.
"""
import argparse
import sys
import threading
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from crowdllama_b200 import engine as eng  # noqa: E402

KEYS = ("tokens_generated", "requests_completed", "preemptions", "sched_decode_steps", "sched_decode_ns", "sched_prefill_calls",
        "sched_prefill_tokens", "sched_prefill_ns")


def run(e, conc, n_req, prompt_len, gen, vocab, jitter=0, sampling="greedy", top=None):
    st0 = e.stats()
    sem = threading.Semaphore(conc)
    lat = []

    def one(i):
        ids = (np.arange(prompt_len, dtype=np.int64) * 7919 + i * 104729) % (vocab - 1000) + 500
        n = gen + ((i * 37) % (2 * jitter + 1) - jitter if jitter else 0)
        if sampling == "ollama":
            sp = eng.ollama_default_sampling(seed=i, max_new_tokens=n)
            sp.ignore_eos = 1
        else:
            sp = eng.greedy(n, ignore_eos=True)
        t0 = time.time()
        e.generate_ids(ids.astype(np.int32), sp, top_logprobs=top)
        lat.append(time.time() - t0)
        sem.release()
    th = []
    t0 = time.time()
    for i in range(n_req):
        sem.acquire()
        t = threading.Thread(target=one, args=(i,))
        t.start()
        th.append(t)
    for t in th:
        t.join()
    dt = time.time() - t0
    st1 = e.stats()
    a = {k: st1[k] - st0[k] for k in KEYS}
    steps = max(a["sched_decode_steps"], 1)
    print(f"{sampling:6s} top_logprobs {'none' if top is None else top:>4} conc {conc:4d} jitter {jitter:3d}: {n_req / dt:6.2f} req/s  p50 {np.median(lat):.3f}s  mean batch {a['tokens_generated'] / steps:5.2f}  decode {a['sched_decode_ns'] / steps * 1e-6:.3f} ms/step "
          f"({a['sched_decode_ns'] * 1e-9:.2f}s)  prefill {a['sched_prefill_ns'] / max(a['sched_prefill_calls'], 1) * 1e-6:.3f} ms/call x {a['sched_prefill_calls']} "
          f"({a['sched_prefill_ns'] * 1e-9:.2f}s)  wall {dt:.2f}s  preempt {a['preemptions']}", flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--max-batch", type=int, default=32)
    ap.add_argument("--gen", type=int, default=256)
    ap.add_argument("--prompt", type=int, default=146)
    ap.add_argument("--conc", default="32,33,48,64,96")
    ap.add_argument("--waves", type=int, default=6)
    ap.add_argument("--preset", default="llama3-8b")
    ap.add_argument("--jitter", default="0", help="comma list: max_new = gen +- jitter (desynchronises the requests)")
    ap.add_argument("--sampling", choices=("greedy", "ollama"), default="greedy")
    ap.add_argument("--top-logprobs", default="none", help="comma list of none | 0..20, run in turn at every concurrency")
    a = ap.parse_args()
    tops = [None if x == "none" else int(x) for x in a.top_logprobs.split(",")]
    with eng.Engine(preset=a.preset, device=0, seed=1234, max_batch=a.max_batch, max_seqs=a.max_batch + 2, start_scheduler=True) as e:
        V = e.cfg["vocab_size"]
        for t in tops:
            run(e, a.max_batch, a.max_batch, a.prompt, 32, V, sampling=a.sampling, top=t)          # warm-up
        for c in [int(x) for x in a.conc.split(",")]:
            for j in [int(x) for x in a.jitter.split(",")]:
                for t in tops:
                    run(e, c, a.waves * a.max_batch, a.prompt, a.gen, V, j, a.sampling, t)
