"""Device sampler (sample_kernels.cu) against the host sampler cl_sample_token: the single-op entry point draw for draw,
the device decode loop against a host replay of the same batched steps, and the scheduler with the device path on
and off."""
import threading
import zlib

import numpy as np
import pytest

from crowdllama_b200 import engine as eng

pytestmark = pytest.mark.gpu


def _sampling(temperature, top_k, top_p, penalty, last_n=64, seed=0, max_new=-1):
    s = eng.Sampling()
    s.temperature, s.top_k, s.top_p, s.repeat_penalty, s.repeat_last_n = temperature, top_k, top_p, penalty, last_n
    s.seed, s.max_new_tokens = seed, max_new
    return s


def _rows(rng, n, vocab, top_k):
    """Logits rows with the awkward cases: ties straddling the k-th place, a constant row, -inf entries, negatives."""
    x = (rng.standard_normal((n, vocab)) * 3.0).astype(np.float32)
    for r in range(n):
        kind = r % 5
        if kind == 1:                                   # a run of equal values across the k-th place
            order = np.argsort(-x[r], kind="stable")
            lo, hi = max(0, top_k - 4), min(vocab, top_k + 4)
            x[r, order[lo:hi]] = x[r, order[lo]]
        elif kind == 2:                                 # constant row
            x[r] = np.float32(0.25)
        elif kind == 3:                                 # -inf entries (enough finite ones to fill the top k)
            mask = rng.random(vocab) < 0.3
            mask[rng.permutation(vocab)[: top_k + 8]] = False
            x[r, mask] = -np.inf
        elif kind == 4:                                 # all negative, small spread (the penalty multiplies)
            x[r] = -np.abs(x[r]) * 0.1 - 0.5
    return x


CL_W = eng.SAMPLE_MAX_WINDOW


def _window(rng, row, vocab):
    """A history of up to 64 ids drawn mostly from the row's best entries, with duplicates (and an id out of range)."""
    n = int(rng.integers(0, CL_W + 1))
    best = np.argpartition(-row, 48)[:48] if row.size > 48 else np.arange(row.size)
    w = np.where(rng.random(n) < 0.7, rng.choice(best, n), rng.integers(0, vocab, n)).astype(np.int32)
    if n > 4:
        w[n // 2] = w[1]                                # duplicate
    if n > 8 and rng.random() < 0.2:
        w[3] = -1                                       # the host skips ids outside the vocabulary
    return w


@pytest.mark.parametrize("vocab", [128256, 32003, 64])
def test_op_sample_matches_host_sampler(vocab):
    temps = (0.3, 0.8, 1.5)
    top_ks = [k for k in (1, 40, eng.SAMPLE_MAX_TOP_K) if k < vocab] + ([vocab - 1] if vocab <= eng.SAMPLE_MAX_TOP_K else [])
    top_ps = (0.0, 0.5, 0.9, 1.0)
    pens = (1.0, 1.1, 0.8)
    combos = [(t, k, p, q) for t in temps for k in top_ks for p in top_ps for q in pens]
    # draws per vocabulary: ~6e3 (128256), ~1.2e4 (32003), ~8.6e4 (64): over 1e5 in all
    rounds, batch = {128256: (48, 128), 32003: (96, 128), 64: (100, 864)}[vocab]
    rng = np.random.default_rng(zlib.crc32(f"op_sample/{vocab}".encode()))
    total = 0
    for rnd in range(rounds):
        sps, steps = [], []
        for r in range(batch):
            t, k, p, q = combos[(rnd * batch + r) % len(combos)]
            last_n = int(rng.integers(1, CL_W + 1)) if r % 4 == 0 else 64
            sps.append(_sampling(t, k, p, q, last_n, seed=int(rng.integers(0, 2**63))))
            steps.append(int(rng.integers(0, 1 << 20)))
        x = _rows(rng, batch, vocab, max(s.top_k for s in sps))
        wins = [_window(rng, x[r], vocab) for r in range(batch)]
        ids, _ = eng.op_sample(x, sps, wins, steps)
        for r in range(batch):
            want = eng.sample_token(x[r], sps[r], wins[r], steps[r])
            assert ids[r] == want, (vocab, rnd, r, sps[r].temperature, sps[r].top_k, sps[r].top_p, sps[r].repeat_penalty,
                                    sps[r].repeat_last_n, list(wins[r]), steps[r], int(ids[r]), want)
        total += batch
    assert total >= {128256: 6000, 32003: 12000, 64: 80000}[vocab]


def test_op_sample_rejects_rows_outside_the_limits():
    x = np.zeros((1, 1000), np.float32)
    for sp in (_sampling(0.8, 0, 0.9, 1.1),                                 # top_k 0: full-vocabulary sort
               _sampling(0.8, eng.SAMPLE_MAX_TOP_K + 1, 0.9, 1.0),
               _sampling(0.8, 40, 0.9, 1.1, last_n=-1),                     # penalty over the whole history
               _sampling(0.8, 40, 0.9, 1.1, last_n=CL_W + 1),
               _sampling(0.0, 40, 0.9, 1.0)):                               # greedy rows are the step tail's
        with pytest.raises(eng.EngineError) as ei:
            eng.op_sample(x, [sp], [[]], [0])
        assert ei.value.status == eng.CL_ERR_INVALID_ARG


def _mixed_samplings(B, vocab):
    out = []
    for b in range(B):
        if b % 3 == 0:
            out.append(eng.greedy(0))
        elif b % 3 == 1:
            out.append(eng.ollama_default_sampling(seed=b))
        else:
            out.append(_sampling(1.5, min(eng.SAMPLE_MAX_TOP_K, vocab - 1), 0.5, 0.8, last_n=16, seed=1000 + b))
    return out


def _device_loop_vs_replay(e, B, n_steps):
    V = e.cfg["vocab_size"]
    sps = _mixed_samplings(B, V)
    prompts = [np.array([(i * 7919 + 13 * b + 5) % V for i in range(5 + b % 7)], np.int32) for b in range(B)]

    def admit():
        seqs, first, hists = [], [], []
        for b in range(B):
            s = e.seq_create()
            lg = e.prefill(s, prompts[b])
            t = eng.sample_token(lg, sps[b], prompts[b], 0)
            seqs.append(s); first.append(t); hists.append(list(prompts[b]) + [t])
        return seqs, first, hists

    seqs, first, _ = admit()
    dev, _ = e.decode_sample_batch(seqs, first, sps, [1] * B, n_steps)
    for s in seqs:
        e.seq_free(s)
    seqs, toks, hists = admit()
    for i in range(n_steps):
        lg, _ = e.decode_step_batch(seqs, toks)
        toks = [eng.sample_token(lg[b], sps[b], hists[b], 1 + i) for b in range(B)]
        for b in range(B):
            hists[b].append(toks[b])
        np.testing.assert_array_equal(dev[i], toks, err_msg=f"step {i}")
    for s in seqs:
        e.seq_free(s)
    assert e.stats()["kv_pages_used"] == 0


def test_decode_sample_batch_matches_host_replay_tiny():
    with eng.Engine(preset="tiny-test", seed=5, max_batch=128) as e:
        for B in (1, 3, 40, 128):
            _device_loop_vs_replay(e, B, 24)


def test_decode_sample_batch_matches_host_replay_llama3_layers():
    model = dict(eng.model_preset("llama3-8b"))
    model.update(n_layers=2, max_seq_len=512)
    with eng.Engine(model=model, model_name="llama3-8b-2l", seed=9, max_batch=128) as e:
        for B in (1, 3, 40, 128):
            _device_loop_vs_replay(e, B, 12)


def test_decode_sample_batch_rejects_options_outside_the_limits():
    with eng.Engine(preset="tiny-test", seed=5, max_batch=4) as e:
        s = e.seq_create()
        e.prefill(s, np.arange(1, 9, dtype=np.int32), want_logits=False)
        with pytest.raises(eng.EngineError) as ei:
            e.decode_sample_batch([s], [3], [_sampling(0.8, 0, 0.9, 1.0)], [1], 4)
        assert ei.value.status == eng.CL_ERR_INVALID_ARG


def _requests(V):
    reqs = [eng.ollama_default_sampling(seed=sd, max_new_tokens=40) for sd in (1, 2, 77)]
    reqs.append(_sampling(1.2, 128, 0.95, 0.9, last_n=8, seed=5, max_new=40))
    reqs.append(_sampling(0.7, 0, 0.9, 1.1, last_n=64, seed=6, max_new=40))          # outside the limits: host path
    reqs.append(eng.greedy(40))
    for s in reqs:
        s.ignore_eos = 1
    return reqs


def _engine(dev, scheduler, monkeypatch, **kw):
    monkeypatch.setenv("CL_SCHED_DEVICE_SAMPLE", "1" if dev else "0")
    return eng.Engine(preset="tiny-test", seed=21, start_scheduler=scheduler, **kw)


@pytest.mark.parametrize("scheduler", [False, True])
def test_generate_ids_same_with_device_sampler_on_and_off(scheduler, monkeypatch):
    out = {}
    for dev in (True, False):
        with _engine(dev, scheduler, monkeypatch) as e:
            V = e.cfg["vocab_size"]
            out[dev] = [e.generate_ids(np.array([(i * 31 + 7 * j) % V for i in range(9 + j)], np.int32), sp).token_ids
                        for j, sp in enumerate(_requests(V))]
    for a, b in zip(out[True], out[False]):
        assert len(a) == 40
        np.testing.assert_array_equal(a, b)


def test_sampled_request_runs_the_device_sampler(monkeypatch):
    N = 20
    with _engine(True, False, monkeypatch) as e:
        p = np.arange(3, 15, dtype=np.int32)
        g, s = eng.greedy(N, ignore_eos=True), eng.ollama_default_sampling(seed=3, max_new_tokens=N)
        s.ignore_eos = 1
        e.generate_ids(p, g)                             # warm-up: graphs and lazy set-up
        k0 = e.stats()["kernel_launches"]
        e.generate_ids(p, g)
        k1 = e.stats()["kernel_launches"]
        r = e.generate_ids(p, s)
        k2 = e.stats()["kernel_launches"]
        assert r.n_generated == N
        assert (k2 - k1) - (k1 - k0) == N                 # one sampler launch per drawn token, no other difference


def test_mixed_burst_through_the_scheduler(monkeypatch):
    with _engine(True, True, monkeypatch, max_batch=8, max_seqs=10) as e:
        V = e.cfg["vocab_size"]
        kinds = _requests(V)
        results = {}

        def one(i):
            sp = kinds[i % len(kinds)]
            n = 8 + (i * 7) % 25
            sp2 = eng.Sampling.from_buffer_copy(sp)
            sp2.max_new_tokens = n
            sp2.seed = sp.seed + i
            r = e.generate_ids(np.array([(j * 13 + i) % V for j in range(4 + i % 30)], np.int32), sp2)
            results[i] = (r.n_generated, n)

        th = [threading.Thread(target=one, args=(i,)) for i in range(36)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        assert len(results) == 36
        for i, (got, want) in results.items():
            assert got == want, (i, got, want)
        st = e.stats()
        assert st["kv_pages_used"] == 0 and st["active_seqs"] == 0
