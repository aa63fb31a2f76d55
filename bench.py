#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 worker decode engine (contract: DESIGN.md §6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Metric (BASELINE.json): "decode tokens/sec/GPU (Llama-3-8B, seq 4K) + box req/s at 1/2/4/8 peers".

First half — `value`, `roofline`, `e2e` (BASELINE.json configs[2]): Llama-3-8B shapes, bf16 synthetic seeded weights
(no checkpoints exist offline), a 4096-token prompt is prefilled, then a greedy 1-token decode loop.  One "step" = one
decoded token = one pass of the whole token step over all weights (15 GB) and the KV cache of the sequence.  N GPUs =
N independent replicas (one process per GPU, no collective on the data path — SURVEY.md §8e): weak scaling,
value = N*K tokens / max-over-ranks device time.  `roofline` describes the step's dominant kernel
(decode_mega_kernel: algorithmic bytes per launch / CUDA-event time per launch, measured live on the launching
stream); the whole-step figure sits beside it in `roofline.step`.

Second half — `box` (configs[3]): every rank also serves as a worker peer (WorkerServer over the length-prefixed
protobuf protocol, pkg/peer/peer.go:190-256) and a load generator next to rank 0 drives the gateway stand-in
(/api/chat -> FindBestWorker, pkg/peermanager/manager.go:338-387 -> RequestInference, pkg/gateway/gateway.go:243-293
-> cl_handle_message -> continuous-batching scheduler): 64 concurrent chats x 256 greedy tokens as BASELINE states,
and a saturating load (BOX_MAX_BATCH = 128 concurrent chats per peer).  Reported: req/s, tok/s, per-worker request counts.

`--impl reference` times the reference arm: the reference worker's CPU path.  The reference's own implementation
(Ollama v0.9.6) cannot be built or installed offline, so the arm runs the CPU oracle port of the same token step
(oracle/, OpenMP over all host cores) on the same config.
"""
from __future__ import annotations

import argparse
import json
import os
import socket
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

PRESET = "llama3-8b"
MODEL_NAME = "llama3:8b"
CTX = 4096
SEED = 1234
METRIC = "decode tokens/sec (Llama-3-8B bf16, seq 4K; aggregate over local worker peers)"
BOX_MAX_BATCH = int(os.environ.get("CL_BOX_MAX_BATCH", "128"))   # sequences per worker peer's decode batch (one peer, saturated: 25 req/s at 32, 46 at 64, 68 at 128)
BOX_GEN = 256


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            d = json.loads(p.read_text())
            return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", 1453.9)), "measured"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, 1400.0, "fallback"


def ncu_traffic(kernel: str):
    """DRAM traffic per launch of the dominant kernel from the committed ncu --set full capture (bench.py cannot run
    ncu): profiles/ncu_traffic.json, written by tools/ncu_summary.py from the same command under the profiler."""
    p = ROOT / "profiles" / "ncu_traffic.json"
    try:
        return json.loads(p.read_text()).get(kernel)
    except Exception:  # noqa: BLE001
        return None


def model_bytes(cfg):
    layer = ((cfg["n_heads"] + 2 * cfg["n_kv_heads"]) * cfg["head_dim"] * cfg["d_model"] + cfg["d_model"] * cfg["n_heads"] * cfg["head_dim"]
             + 3 * cfg["d_ff"] * cfg["d_model"] + 2 * cfg["d_model"])
    p_read = cfg["n_layers"] * layer + cfg["d_model"] + cfg["vocab_size"] * cfg["d_model"]
    kv_tok = 2 * cfg["n_layers"] * cfg["n_kv_heads"] * cfg["head_dim"] * 2
    return p_read, kv_tok, cfg["n_layers"] * layer


def prompt_ids(n, vocab):
    return np.array([(i * 7919 + 13) % vocab for i in range(n)], np.int32)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---- CPU arms (the only places that execute oracle/) ---------------------------------------------------------------
def cpu_baseline(steps_cap_s=12.0, max_tokens=64, warm=2):
    """The CPU oracle port on this box's host cores: Llama-3-8B shapes, synthetic weights, KV cache
    pre-filled to 4096 positions (timing only), greedy decode steps for about 12 s (bounded sample of the workload)."""
    from oracle import oracle as oc
    cfg = dict(oc.PRESETS[PRESET])
    cfg["max_seq_len"] = CTX + 64
    threads = oc.effective_cpus()
    oc.set_threads(threads)
    t0 = time.time()
    m = oc.Model(cfg, seed=SEED)
    gen_s = time.time() - t0
    s = m.new_seq(CTX + 64)
    s.fake_fill(CTX)
    tok = 17
    for _ in range(warm):
        lg = s.forward([tok]); tok = int(lg.argmax())
    t0 = time.time()
    n = 0
    while n < max_tokens and (time.time() - t0) < steps_cap_s:
        lg = s.forward([tok]); tok = int(lg.argmax()); n += 1
    dt = time.time() - t0
    return {"value": round(n / dt, 4), "unit": "tokens/s", "cores": threads, "kind": "port",
            "sample": f"{n} greedy decode steps at ctx {CTX} (KV pre-filled with a synthetic pattern), Llama-3-8B shapes, "
                      f"seeded bf16 weights generated in {gen_s:.1f}s; oracle/llama_oracle.c with OpenMP x{threads}",
            "ms_per_step": round(dt / max(n, 1) * 1e3, 2)}, m, s


def cpu_config1():
    """BASELINE.json configs[0] stand-in (SURVEY.md §8d "Config 1"): TinyLlama-1.1B shapes on the CPU oracle port,
    16-id prompt, 32 greedy tokens — the reference's own CPU-runnable case."""
    from oracle import oracle as oc
    cfg = dict(oc.PRESETS["tinyllama-1.1b"])
    cfg["max_seq_len"] = 128
    threads = oc.effective_cpus()
    oc.set_threads(threads)
    m = oc.Model(cfg, seed=SEED)
    s = m.new_seq(128)
    ids = prompt_ids(16, cfg["vocab_size"])
    t0 = time.time()
    first = int(s.forward(ids).argmax())
    t1 = time.time()
    out, _ = s.greedy(first, 32)
    t2 = time.time()
    s.close(); m.close()
    return {"tokens_per_s": round(32 / (t2 - t1), 2), "prefill_s": round(t1 - t0, 3), "cores": threads, "kind": "port", "ids_head": [int(x) for x in out[:4]]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cb, m, s = cpu_baseline(steps_cap_s=0.0, max_tokens=0, warm=0)  # builds model + pre-filled cache
    tok, t_first = 17, time.time()
    lg = s.forward([tok]); tok = int(lg.argmax())
    t_tok = time.time() - t_first
    warm = max(0, min(args.warmup, 2) - 1)
    for _ in range(warm):
        lg = s.forward([tok]); tok = int(lg.argmax())
    steps = max(3, min(args.steps, int(150.0 / max(t_tok, 1e-3))))
    t0 = time.time()
    for _ in range(steps):
        lg = s.forward([tok]); tok = int(lg.argmax())
    dt = time.time() - t0
    val = steps / dt
    cb.update(value=round(val, 4), ms_per_step=round(dt / steps * 1e3, 2),
              sample=f"{steps} greedy decode steps at ctx {CTX} (bounded from --steps {args.steps}); " + cb["sample"].split(";", 1)[-1].strip())
    line = {"impl": "reference", "metric": METRIC, "value": round(val, 4), "unit": "tokens/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warm + 1, "ms_per_step": round(dt / steps * 1e3, 2), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"configs[2]: Llama-3-8B bf16 shapes, ctx {CTX}, 1-token greedy decode loop", "preset": PRESET,
                       "ctx": CTX, "weights": f"synthetic seed {SEED}", "note": "reference arm = CPU oracle port of the worker's "
                       "model step (Ollama v0.9.6 cannot be built offline); rank 0 only"},
            "cpu_baseline": cb, "e2e": {"value": round(val, 4), "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


# ---- box: the load generator (a process of its own next to rank 0, so that it shares no GIL with worker 0) -----------
def _wait_port(addr, timeout_s):
    t0 = time.time()
    while time.time() - t0 < timeout_s:
        try:
            with socket.create_connection(addr, timeout=2):
                return True
        except OSError:
            time.sleep(0.25)
    return False


BOX_PROMPT = ("Explain, step by step, why the sky appears blue during the day and red at sunset, and what changes on Mars. " * 2)[:118]
BOX_SHARD_CLIENTS = int(os.environ.get("CL_BOX_SHARD_CLIENTS", "128"))   # closed-loop clients per gateway stand-in process (one Python GIL each)


def run_box_shard(addrs, port, concurrency, n_req, first_id, start_at):
    """One gateway stand-in (own metadata table, FindBestWorker routing) + `concurrency` closed-loop clients sending
    `n_req` chats through it.  Returns raw observations; the caller aggregates over shards."""
    from crowdllama_b200 import gateway
    gw = gateway.make_server(addrs, port=port)
    threading.Thread(target=gw.serve_forever, daemon=True).start()
    lat, errs = [], []
    nxt, nxt_lock = [0], threading.Lock()

    def client():
        # one closed-loop client = one thread with one keep-alive HTTP connection (the gateway stand-in speaks HTTP/1.1):
        # no thread or connection set-up per request on either side of the gateway
        import http.client
        conn = None
        while True:
            with nxt_lock:
                i = nxt[0]
                nxt[0] += 1
            if i >= n_req:
                break
            body = json.dumps({"model": MODEL_NAME, "messages": [{"role": "user", "content": f"{first_id + i:04d} {BOX_PROMPT}"}], "stream": False}).encode()
            t0 = time.time()
            try:
                if conn is None:
                    conn = http.client.HTTPConnection("127.0.0.1", port, timeout=900)
                conn.request("POST", "/api/chat", body, {"Content-Type": "application/json"})
                o = json.loads(conn.getresponse().read())
                assert o["done"] and o["model"] == MODEL_NAME and o["message"]["role"] == "assistant" and o["message"]["content"]
                lat.append(time.time() - t0)
            except Exception as ex:  # noqa: BLE001
                errs.append(str(ex))
                try:
                    conn and conn.close()
                finally:
                    conn = None
        if conn:
            conn.close()
    while time.time() < start_at:
        time.sleep(0.005)
    threads = [threading.Thread(target=client) for _ in range(min(concurrency, n_req))]
    t0 = time.time()
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    t1 = time.time()
    res = {"lat": lat, "errors": errs[:3], "n_err": len(errs), "t0": t0, "t1": t1, "counts": dict(gw.counts),
           "advertised": {r.peer_id: [r.tokens_throughput, r.load] for r in gw.table.peers.values()}}
    gw.table.stop()
    gw.shutdown()
    gw.server_close()
    return res


def run_box_client(args):
    """Load generator of the box leg: gateway stand-ins + closed-loop HTTP clients against already running worker peers.
    Up to BOX_SHARD_CLIENTS clients share one gateway stand-in process; larger scenarios are sharded over several such
    processes (every shard routes with FindBestWorker over its own metadata table), because one Python process tops out
    near 500 req/s (measured against instant mock peers) — below what eight peers deliver.  Prints one JSON object."""
    from crowdllama_b200 import gateway
    from crowdllama_b200.worker import STOP_PROTOCOL, STATS_PROTOCOL
    addrs = [("127.0.0.1", args.base_port + i) for i in range(args.workers)]
    if args.box_shard:                                      # child process: one shard of one scenario
        conc, n_req, first_id, port, start_at = args.box_shard.split(",")
        print(json.dumps(run_box_shard(addrs, int(port), int(conc), int(n_req), int(first_id), float(start_at))), flush=True)
        return 0
    out = {"workers": args.workers, "gen_tokens": BOX_GEN, "max_batch_per_worker": BOX_MAX_BATCH, "router": "find_best_worker (manager.go:338-387), "
           "metadata refreshed every 2 s, load-independent capacity in half-octave buckets + two-level load (router.py)",
           "clients_per_gateway_process": BOX_SHARD_CLIENTS}
    try:
        for a in addrs:
            if not _wait_port(a, 600):
                raise RuntimeError(f"worker {a} did not come up")
        for a in addrs:                                  # warm every worker directly: prefill workspaces, every batch size once
            th = [threading.Thread(target=gateway.request_inference, args=(a, MODEL_NAME, f"warm {i} " + BOX_PROMPT, False)) for i in range(BOX_MAX_BATCH)]
            [t.start() for t in th]
            [t.join() for t in th]

        def worker_stats():
            res = []
            for a in addrs:
                with socket.create_connection(a, timeout=5) as sk:
                    sk.sendall((STATS_PROTOCOL + "\n").encode())
                    data = b""
                    while chunk := sk.recv(65536):
                        data += chunk
                res.append(json.loads(data))
            return res

        def scenario(concurrency, n_req):
            n_sh = max(1, min(8, -(-concurrency // BOX_SHARD_CLIENTS)))
            st0 = worker_stats()
            if n_sh == 1:
                parts = [run_box_shard(addrs, args.base_port - 1, concurrency, n_req, 0, time.time())]
            else:
                start_at = time.time() + 3.0                # the shards import, probe the peers, then start together
                procs, first = [], 0
                for i in range(n_sh):
                    c = concurrency // n_sh + (1 if i < concurrency % n_sh else 0)
                    r = n_req // n_sh + (1 if i < n_req % n_sh else 0)
                    procs.append(subprocess.Popen([sys.executable, str(ROOT / "bench.py"), "--box-client", "--workers", str(args.workers), "--base-port", str(args.base_port),
                                                   "--box-shard", f"{c},{r},{first},{args.base_port - 1 - i},{start_at}"],
                                                  stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""}))
                    first += r
                parts = []
                for pr in procs:
                    so, se = pr.communicate(timeout=1200)
                    if pr.returncode != 0 or not so.strip():
                        raise RuntimeError(f"box shard failed: {se[-400:]}")
                    parts.append(json.loads(so.strip().splitlines()[-1]))
            st1 = worker_stats()
            lat = [x for p_ in parts for x in p_["lat"]]
            dt = max(p_["t1"] for p_ in parts) - min(p_["t0"] for p_ in parts)
            counts, adv = {}, {}
            for p_ in parts:
                for k, v in p_["counts"].items():
                    counts[k] = counts.get(k, 0) + v
                adv.update(p_["advertised"])
            ok = len(lat)
            acc = {k: sum(b.get(k, 0) - a.get(k, 0) for a, b in zip(st0, st1)) for k in ("tokens_generated", "requests_completed", "preemptions", "sched_decode_steps",
                                                                            "sched_decode_ns", "sched_prefill_calls", "sched_prefill_tokens", "sched_prefill_ns")}
            sched = {"mean_batch": round(acc["tokens_generated"] / max(acc["sched_decode_steps"], 1), 2),
                     "decode_ms_per_step": round(acc["sched_decode_ns"] / max(acc["sched_decode_steps"], 1) * 1e-6, 3),
                     "prefill_ms_per_call": round(acc["sched_prefill_ns"] / max(acc["sched_prefill_calls"], 1) * 1e-6, 3),
                     "prefill_tokens_per_call": round(acc["sched_prefill_tokens"] / max(acc["sched_prefill_calls"], 1), 1),
                     "decode_s_per_worker": round(acc["sched_decode_ns"] * 1e-9 / len(addrs), 3),
                     "prefill_s_per_worker": round(acc["sched_prefill_ns"] * 1e-9 / len(addrs), 3), "preemptions": acc["preemptions"]}
            return {"scheduler": sched, "concurrency": concurrency, "requests": n_req, "ok": ok, "errors": [e for p_ in parts for e in p_["errors"]][:3],
                    "wall_s": round(dt, 3), "req_per_s": round(ok / dt, 3), "tok_per_s": round(ok * BOX_GEN / dt, 1),
                    "p50_latency_s": round(float(np.median(lat)), 3) if lat else None, "gateway_processes": n_sh,
                    "per_worker_requests": dict(sorted(counts.items())), "advertised_at_end": dict(sorted(adv.items()))}
        # untimed warm-up THROUGH the gateway (the first scenario otherwise pays for cold HTTP / thread / routing paths and
        # starts desynchronised: 21.2 req/s first against 25.0 for the same scenario run later, r2o)
        out["warmup"] = {k: v for k, v in scenario(min(BOX_MAX_BATCH * args.workers, BOX_SHARD_CLIENTS), 2 * BOX_MAX_BATCH * args.workers).items()
                         if k in ("requests", "ok", "wall_s")}
        # BASELINE.json configs[3]: 64 concurrent chats.  Long enough for request-level statistics: >= 6 waves per worker slot.
        for i, tag in enumerate(os.environ.get("CL_BOX_SCENARIOS", "config4,saturated").split(",")):   # the default is the contract
            key = tag if tag not in out else f"{tag}#{i}"
            if tag == "config4":
                out[key] = scenario(64, max(384, 96 * args.workers))
            elif tag == "saturated":
                out[key] = scenario(BOX_MAX_BATCH * args.workers, 6 * BOX_MAX_BATCH * args.workers)
            elif tag.startswith("c"):                                         # c<concurrency>: diagnostics
                out[key] = scenario(int(tag[1:]), 6 * BOX_MAX_BATCH * args.workers)
    except Exception as ex:  # noqa: BLE001
        out["error"] = repr(ex)
    for a in addrs:
        try:
            with socket.create_connection(a, timeout=5) as s:
                s.sendall((STOP_PROTOCOL + "\n").encode())
        except OSError:
            pass
    print(json.dumps(out), flush=True)
    return 0


def run_box(e, rank, n_gpus, base_port):
    """Every rank: serve as a worker peer until the load generator says stop.  Rank 0 also launches the generator."""
    from crowdllama_b200 import engine as eng
    from crowdllama_b200.worker import WorkerServer
    srv = WorkerServer(("127.0.0.1", base_port + rank), e, peer_id=f"b200-worker-{rank}", sampling=eng.greedy(BOX_GEN, ignore_eos=True))
    threading.Thread(target=srv.serve_forever, kwargs={"poll_interval": 0.1}, daemon=True).start()
    res, client = None, None
    if rank == 0:
        client = subprocess.Popen([sys.executable, str(ROOT / "bench.py"), "--box-client", "--workers", str(n_gpus), "--base-port", str(base_port)],
                                  stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                                  env={**os.environ, "CUDA_VISIBLE_DEVICES": "", "RANK": "0", "WORLD_SIZE": "1"})
    stopped = srv.stop_event.wait(900)           # CPU-side wait: no NCCL kernel may sit on the GPU while the peers serve
    if client is not None:
        try:
            so, se = client.communicate(timeout=60)
            res = json.loads(so.strip().splitlines()[-1])
        except Exception as ex:  # noqa: BLE001
            client.kill()
            res = {"error": f"load generator failed: {ex!r}"}
    if not stopped and res is None:
        res = {"error": "timeout"}
    srv.shutdown()
    srv.server_close()
    return res


# ---- our arm ---------------------------------------------------------------------------------------------------------
def run_ours(args):
    from crowdllama_b200 import engine as eng
    hbm, tflops, peak_src = load_peaks()
    from crowdllama_b200.distutil import Group
    grp = Group()
    rank, local, world = grp.rank, grp.local_rank, grp.world
    if world != args.gpus and world > 1:
        print(f"warning: WORLD_SIZE={world} != --gpus {args.gpus}", file=sys.stderr)
    n_gpus = max(world, 1)
    K, W = args.steps, max(args.warmup, 3)
    t0 = time.time()
    e = eng.Engine(preset=args.preset, model_name=MODEL_NAME, device=local, seed=SEED, max_batch=BOX_MAX_BATCH, max_seqs=BOX_MAX_BATCH + 2,
                   start_scheduler=True)
    init_s = time.time() - t0
    cfg = e.cfg
    p_read, kv_tok, layer_bytes_elems = model_bytes(cfg)
    KD = min(64, max(8, K))                                     # eagerly launched steps of the dominant-kernel timing
    ctx = min(args.ctx, cfg["max_seq_len"] - (K + W + KD + 8))
    ids = prompt_ids(ctx, cfg["vocab_size"])

    # ---- prefill (tcgen05 path) through the C-ABI with a host prompt
    s = e.seq_create()
    t0 = time.time()
    lg = e.prefill(s, ids)
    prefill_ms_first = (time.time() - t0) * 1e3
    first = int(lg.argmax())
    time.sleep(1.0)   # let the board's power state settle after the prefill burst (r2h: sw_power_cap right after a 58 ms prefill cost 1.7 %)
    # ---- warm-up decode steps (also captures the CUDA graph)
    wids, _ = e.decode_greedy(s, first, W)
    nxt = int(wids[-1])
    launches0 = e.stats()["kernel_launches"]
    # ---- timed region: exactly K steps, device time from CUDA events on the launching stream
    grp.barrier()
    clk = ClockSampler(local)
    clk.start()
    out_ids, ms = e.decode_greedy(s, nxt, K)
    grp.barrier()
    clocks = clk.stop()
    launches = e.stats()["kernel_launches"] - launches0
    if args.dump_outputs and rank == 0:
        # what cl_decode_greedy returned for the timed steps; prompt, weights and warm-up depend only on the arguments
        out_dir = Path(args.dump_outputs)
        out_dir.mkdir(parents=True, exist_ok=True)
        np.save(out_dir / "decode_ids.npy", out_ids.astype(np.float64))
    ms_max = grp.max(ms)
    value = n_gpus * K / (ms_max * 1e-3)
    mean_ctx = ctx + W + K / 2.0
    step_bytes = 2 * p_read + kv_tok * (mean_ctx + 1)
    achieved = step_bytes / (ms / K * 1e-3) / 1e9

    # ---- the step's dominant kernel, timed live: CUDA-event pair around each of its launches (same stream), KD steps
    kern = None
    try:
        k_ms, k_step_ms = e.time_dominant_kernel(s, int(out_ids[-1]), KD)
        k_ctx = ctx + W + K + KD / 2.0
        k_bytes = 2 * layer_bytes_elems + kv_tok * (k_ctx + 1)            # all layer weights + the sequence's K/V, bf16
        mega = os.environ.get("CL_MEGA", "1") != "0"
        name = "decode_mega_kernel" if mega else "per-op layer stack (gemv_ring_kernel x4 + attn_decode_kernel per layer)"
        tr = ncu_traffic("decode_mega_kernel") if mega else None
        kern = {"name": name, "launches_timed": KD, "ms": round(k_ms, 5), "algorithmic_bytes": int(k_bytes), "achieved": round(k_bytes / (k_ms * 1e-3) / 1e9, 1),
                "share_of_step_time": round(k_ms / k_step_ms, 4), "eager_step_ms": round(k_step_ms, 4), "traffic": tr}
    except Exception as ex:  # noqa: BLE001
        kern = {"error": str(ex)}
    e.seq_free(s)

    # ---- e2e: the request path (cl_generate_ids -> continuous-batching scheduler), HOST prompt in, HOST ids out,
    #      every step's token read back to the host; prefill measured separately inside the same call
    r = e.generate_ids(ids, eng.greedy(K, ignore_eos=True))     # warm (prefill workspace etc. already hot)
    grp.barrier()
    r = e.generate_ids(ids, eng.greedy(K, ignore_eos=True))
    grp.barrier()
    dec_s = grp.max(r.decode_ns * 1e-9)
    e2e_val = n_gpus * (r.n_generated - 1) / dec_s
    req_s = n_gpus / grp.max(r.total_ns * 1e-9)
    prefill_ms = r.prefill_ns * 1e-6
    prefill_flops = 2.0 * ctx * (p_read - cfg["vocab_size"] * cfg["d_model"]) + 4.0 * cfg["n_layers"] * cfg["n_heads"] * cfg["head_dim"] * ctx * ctx / 2

    # ---- configs[1]: 128-token prompt, 256 greedy tokens through the request path (every rank; rank 0 reports)
    c2 = None
    if not args.no_extra_configs:
        p2 = prompt_ids(128, cfg["vocab_size"])
        e.generate_ids(p2, eng.greedy(8, ignore_eos=True))
        r2 = e.generate_ids(p2, eng.greedy(256, ignore_eos=True))
        mean2 = 128 + 128
        c2 = {"workload": "configs[1]: 128-token prompt, 256 greedy tokens, cl_generate_ids", "prefill_ms": round(r2.prefill_ns * 1e-6, 3),
              "decode_tokens_per_s": round((r2.n_generated - 1) / (r2.decode_ns * 1e-9), 2),
              "roofline_frac": round((2 * p_read + kv_tok * (mean2 + 1)) * (r2.n_generated - 1) / (r2.decode_ns * 1e-9) / 1e9 / hbm, 4),
              "requests_per_s": round(1.0 / (r2.total_ns * 1e-9), 3)}

    # ---- box req/s (configs[3]): the ranks become worker peers; no NCCL traffic until the load generator is done
    box = None
    if not args.no_box:
        grp.barrier()
        base_port = 21000 + (int(os.environ.get("MASTER_PORT", "29500")) % 500) * 16 + 1
        box = run_box(e, rank, n_gpus, base_port)
        grp.barrier()
    e.close()

    # ---- configs[0] on the GPU: TinyLlama shapes, 16-id prompt, 32 greedy tokens (per-op kernels: other shape)
    c1 = None
    if rank == 0 and n_gpus == 1 and not args.no_extra_configs:
        try:
            with eng.Engine(preset="tinyllama-1.1b", device=local, seed=SEED, max_batch=1, start_scheduler=True) as t:
                tp = prompt_ids(16, t.cfg["vocab_size"])
                t.generate_ids(tp, eng.greedy(32, ignore_eos=True))
                rt = t.generate_ids(tp, eng.greedy(32, ignore_eos=True))
                tb, tk, _ = model_bytes(t.cfg)
                tps = (rt.n_generated - 1) / (rt.decode_ns * 1e-9)
                c1 = {"workload": "configs[0] shapes on the GPU: TinyLlama-1.1B bf16, 16-id prompt, 32 greedy tokens", "decode_tokens_per_s": round(tps, 1),
                      "prefill_ms": round(rt.prefill_ns * 1e-6, 3), "roofline_frac": round((2 * tb + tk * 33) * tps / 1e9 / hbm, 4)}
        except Exception as ex:  # noqa: BLE001
            c1 = {"error": str(ex)}
    grp.close()

    if rank != 0:
        return 0
    cb = None
    if n_gpus == 1 and not args.no_cpu_baseline:
        try:
            cb, _m, _s = cpu_baseline()
            _s.close(); _m.close()
            del _m, _s
            if c1 is not None and not args.no_extra_configs:
                c1["cpu_reference_path"] = cpu_config1()
        except Exception as ex:  # noqa: BLE001
            cb = {"value": None, "unit": "tokens/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}
    k_ok = isinstance(kern, dict) and "achieved" in kern
    traffic = kern["traffic"]["dram_bytes_per_launch"] if k_ok and kern.get("traffic") else None
    line = {
        "metric": METRIC, "value": round(value, 2), "unit": "tokens/s", "n_gpus": n_gpus, "steps": K, "warmup": W,
        "ms_per_step": round(ms_max / K, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": f"configs[2]: Llama-3-8B bf16, {ctx}-token prefill then 1-token greedy decode loop, batch 1 per GPU",
                   "preset": args.preset, "ctx": ctx, "weights": f"synthetic counter-based seed {SEED}", "page_size": 32,
                   "replicas": n_gpus, "l2": "inputs larger than L2: every step streams 15 GB of weights (L2 = 126 MB)",
                   "decode_path": "persistent kernel" if os.environ.get("CL_MEGA", "1") != "0" else "per-op kernels"},
        "per_gpu_tokens_per_s": round(value / n_gpus, 2),
        # the dominant kernel of the timed graph (92 % of the step), timed live
        "roofline": {"bound": "hbm", "kernel": kern.get("name") if isinstance(kern, dict) else None,
                     "achieved": kern["achieved"] if k_ok else round(achieved, 1), "peak": hbm, "unit": "GB/s",
                     "frac": round((kern["achieved"] if k_ok else achieved) / hbm, 4), "traffic": traffic, "peak_source": peak_src,
                     "detail": kern,
                     "step": {"scope": "whole token step (one CUDA-graph launch: embed + persistent kernel + LM head + argmax)",
                              "achieved": round(achieved, 1), "frac": round(achieved / hbm, 4), "algorithmic_bytes_per_step": int(step_bytes)},
                     "prefill": {"bound": "tensor", "achieved": round(prefill_flops / (prefill_ms * 1e-3) / 1e12, 1), "peak": tflops, "unit": "TFLOP/s",
                                 "frac": round(prefill_flops / (prefill_ms * 1e-3) / 1e12 / tflops, 4), "tokens": ctx, "ms": round(prefill_ms, 2),
                                 "algorithmic_tflop": round(prefill_flops / 1e12, 2)}},
        "cpu_baseline": cb,
        "e2e": {"value": round(e2e_val, 2), "unit": "tokens/s", "h2d_bytes_per_step": round(ctx * 4 / K, 1),
                "d2h_bytes_per_step": 4 * 2, "path": "cl_generate_ids -> scheduler; host prompt ids in, one token id read back per step",
                "prefill_ms": round(prefill_ms, 2), "prefill_tflops": round(prefill_flops / (prefill_ms * 1e-3) / 1e12, 1),
                "requests_per_s": round(req_s, 4)},
        "box": box,
        "configs": {"config1": c1, "config2": c2},
        "gpu_launches": int(launches), "clocks": clocks,
        "extra": {"init_s": round(init_s, 1), "first_prefill_ms_incl_workspace_alloc": round(prefill_ms_first, 1),
                  "bf16_tflops_sustained_peak": tflops},
    }
    print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--preset", default=PRESET)
    ap.add_argument("--ctx", type=int, default=CTX)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-box", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the token ids of the timed decode steps to DIR/decode_ids.npy (float64), to compare two builds")
    ap.add_argument("--box-client", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--box-shard", default="", help=argparse.SUPPRESS)
    ap.add_argument("--workers", type=int, default=1, help=argparse.SUPPRESS)
    ap.add_argument("--base-port", type=int, default=21001, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU decode path computed; it needs --impl ours")
    if args.box_client:
        return run_box_client(args)
    return run_reference(args) if args.impl == "reference" else run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
