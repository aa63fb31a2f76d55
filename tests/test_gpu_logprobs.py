"""Token log-probabilities (logprobs_kernel) on the GPU: the single-op entry point against numpy float64 log_softmax,
the token ids with logprobs on and off, the records' internal consistency, a B = 1 replay of the step logits, and the
wire end to end."""
import re
import threading
import zlib

import numpy as np
import pytest

from crowdllama_b200 import engine as eng
from crowdllama_b200 import pb

pytestmark = pytest.mark.gpu

K = eng.MAX_TOP_LOGPROBS


def _rows(rng, n, vocab, top_n):
    """Random rows plus the awkward cases: ties across the top_n-th place, a constant row, -inf entries, |x| up to 1e3."""
    x = (rng.standard_normal((n, vocab)) * 3.0).astype(np.float32)
    for r in range(n):
        kind = r % 6
        if kind == 1:                                   # a run of equal values across the N-th place
            order = np.argsort(-x[r], kind="stable")
            lo, hi = max(0, top_n - 3), min(vocab, top_n + 3)
            x[r, order[lo:hi]] = x[r, order[lo]]
        elif kind == 2:                                 # constant row
            x[r] = np.float32(0.25)
        elif kind == 3:                                 # -inf entries (some finite ones stay)
            mask = rng.random(vocab) < 0.4
            mask[rng.permutation(vocab)[:4]] = False
            x[r, mask] = -np.inf
        elif kind == 4:                                 # large magnitudes
            x[r] = (rng.standard_normal(vocab) * 300.0).clip(-1e3, 1e3).astype(np.float32)
        elif kind == 5:                                 # a large offset on a narrow spread
            x[r] = x[r] * 0.01 + np.float32(900.0)
    return x


def _ref(x, chosen, top_n):
    """numpy float64 log_softmax; top_n ids by fp32 value descending, then id ascending."""
    xd = x.astype(np.float64)
    m = np.max(xd, axis=1, keepdims=True)
    lse = m[:, 0] + np.log(np.sum(np.exp(xd - m), axis=1))
    lp = xd - lse[:, None]
    ids = np.stack([np.lexsort((np.arange(x.shape[1]), -x[r]))[:top_n] for r in range(x.shape[0])]) if top_n else \
        np.zeros((x.shape[0], 0), np.int64)
    return lp[np.arange(x.shape[0]), chosen], ids, np.take_along_axis(lp, ids, axis=1), np.max(np.abs(np.where(np.isfinite(x), x, 0)), axis=1)


def _close(got, want, mx):
    """values within 1e-5 (1 + |logprob| + |max logit|); -inf must be exactly -inf"""
    inf = np.isneginf(want)
    assert np.array_equal(np.isneginf(got), inf)
    tol = 1e-5 * (1.0 + np.abs(want[~inf]) + np.broadcast_to(mx, want.shape)[~inf])
    err = np.abs(got[~inf].astype(np.float64) - want[~inf])
    assert np.all(err <= tol), float(np.max(err - tol))


@pytest.mark.parametrize("vocab", [128256, 32003, 64])
@pytest.mark.parametrize("top_n", [0, 1, 5, 20])
def test_op_logprobs_matches_numpy(vocab, top_n):
    rng = np.random.default_rng(zlib.crc32(f"logprobs/{vocab}/{top_n}".encode()))
    n = 24
    x = _rows(rng, n, vocab, max(top_n, 1))
    chosen = np.array([rng.choice(np.flatnonzero(np.isfinite(x[r]))) for r in range(n)], np.int32)
    chosen[3] = np.flatnonzero(np.isneginf(x[3]))[0]          # an emitted id with probability 0 reports -inf
    lp, ids, tl, _ = eng.op_logprobs(x, chosen, top_n)
    want_lp, want_ids, want_tl, mx = _ref(x, chosen, top_n)
    _close(lp, want_lp, mx)
    np.testing.assert_array_equal(ids, want_ids)
    _close(tl, want_tl, mx[:, None])
    # the same row gives the same bits at any batch size and position
    perm = rng.permutation(n)
    lp2, ids2, tl2, _ = eng.op_logprobs(np.concatenate([x[perm], x[:5]]), np.concatenate([chosen[perm], chosen[:5]]), top_n)
    assert np.array_equal(lp2[:n].view(np.uint32), lp[perm].view(np.uint32))
    assert np.array_equal(lp2[n:].view(np.uint32), lp[:5].view(np.uint32))
    np.testing.assert_array_equal(ids2[:n], ids[perm])
    assert np.array_equal(tl2[:n].view(np.uint32), tl[perm].view(np.uint32))
    for r in (0, 3, 7):
        lp1, ids1, tl1, _ = eng.op_logprobs(x[r:r + 1], chosen[r:r + 1], top_n)
        assert lp1.view(np.uint32)[0] == lp.view(np.uint32)[r]
        np.testing.assert_array_equal(ids1[0], ids[r])
        assert np.array_equal(tl1[0].view(np.uint32), tl[r].view(np.uint32))


def test_op_logprobs_rejects_bad_top_n():
    x = np.zeros((1, 100), np.float32)
    for n in (-1, K + 1):
        with pytest.raises(eng.EngineError) as ei:
            eng.op_logprobs(x, [0], n)
        assert ei.value.status == eng.CL_ERR_INVALID_ARG


def _sampling(temperature, top_k, top_p, penalty, last_n=64, seed=0, max_new=-1):
    s = eng.Sampling()
    s.temperature, s.top_k, s.top_p, s.repeat_penalty, s.repeat_last_n = temperature, top_k, top_p, penalty, last_n
    s.seed, s.max_new_tokens = seed, max_new
    return s


def _kinds():
    """greedy, Ollama defaults (device sampler) and top_k 0 (host sampler)"""
    out = [eng.greedy(24), eng.ollama_default_sampling(seed=3, max_new_tokens=24), _sampling(0.7, 0, 0.9, 1.1, seed=6, max_new=24)]
    for s in out:
        s.ignore_eos = 1
    return out


def _prompt(i, V):
    return np.array([(j * 13 + 7 * i + 1) % V for j in range(4 + (i * 5) % 23)], np.int32)


def _burst(e, n, top):
    V = e.cfg["vocab_size"]
    kinds, res = _kinds(), {}

    def one(i):
        sp = eng.Sampling.from_buffer_copy(kinds[i % 3])
        sp.seed = sp.seed + i
        res[i] = e.generate_ids(_prompt(i, V), sp, top_logprobs=top)

    th = [threading.Thread(target=one, args=(i,)) for i in range(n)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert len(res) == n
    return [res[i] for i in range(n)]


def _check_records(r, greedy, top):
    n = r.n_generated
    assert r.logprob.shape == (n,) and r.top_ids.shape == (n, top) and r.top_logprobs.shape == (n, top)
    assert np.all(r.logprob <= 0.0)
    if top:
        assert np.all(np.diff(r.top_logprobs, axis=1) <= 0)
        assert np.all(np.sum(np.exp(r.top_logprobs.astype(np.float64)), axis=1) <= 1 + 1e-5)
        assert np.all(r.top_logprobs[:, 0] >= r.logprob)
    if greedy and top:
        np.testing.assert_array_equal(r.top_ids[:, 0], r.token_ids)
        assert np.array_equal(r.top_logprobs[:, 0].view(np.uint32), r.logprob.view(np.uint32))


@pytest.mark.parametrize("scheduler", [False, True])
def test_ids_unchanged_and_records_consistent(scheduler):
    with eng.Engine(preset="tiny-test", seed=21, max_batch=48, max_seqs=48, start_scheduler=scheduler) as e:
        for n in (1, 3, 40):
            off = _burst(e, n, None)
            on = _burst(e, n, 5)
            on20 = _burst(e, min(n, 3), 20)
            for i, (a, b) in enumerate(zip(off, on)):
                assert a.n_generated == 24 and a.logprob is None
                np.testing.assert_array_equal(a.token_ids, b.token_ids, err_msg=f"burst {n} request {i}")
                _check_records(b, i % 3 == 0, 5)
            for i, c in enumerate(on20):
                np.testing.assert_array_equal(c.token_ids, off[i].token_ids)
                _check_records(c, i % 3 == 0, 20)
                np.testing.assert_array_equal(c.top_ids[:, :5], on[i].top_ids)     # the top 5 of the top 20
        st = e.stats()
        assert st["kv_pages_used"] == 0 and st["active_seqs"] == 0


def _log_softmax(x):
    x = x.astype(np.float64)
    m = np.max(x)
    return x - (m + np.log(np.sum(np.exp(x - m))))


def _replay(e, prompt, ids):
    """log_softmax of the logits before every generated id: prefill, then one cl_decode_step per id (teacher forced)"""
    s = e.seq_create()
    rows = [e.prefill(s, prompt)]
    for t in ids[:-1]:
        rows.append(e.decode_step(s, int(t))[0])
    e.seq_free(s)
    return [(_log_softmax(r), r) for r in rows]


def _order(row, n):
    return np.lexsort((np.arange(row.size), -row))[:n]


def test_records_match_a_single_sequence_replay():
    """Synchronous path at B = 1 (the same single-sequence step graph as cl_decode_step): ids exact, values to 1e-5."""
    with eng.Engine(preset="tiny-test", seed=21, max_batch=8) as e:
        V = e.cfg["vocab_size"]
        for j, sp in enumerate(_kinds()):
            p = _prompt(j, V)
            r = e.generate_ids(p, sp, top_logprobs=K)
            for i, (ls, row) in enumerate(_replay(e, p, r.token_ids)):
                mx = np.max(np.abs(row))
                want_ids = _order(row, K)
                np.testing.assert_array_equal(r.top_ids[i], want_ids, err_msg=f"request {j} token {i}")
                _close(r.top_logprobs[i], ls[want_ids], mx)
                _close(r.logprob[i:i + 1], ls[r.token_ids[i]:r.token_ids[i] + 1], mx)


def test_batched_records_match_replay_within_the_logit_tolerance():
    """Scheduler bursts (batched steps, group admission): every value within twice the model logit tolerance of DESIGN.md
    §2 (0.125 for <= 3 layers; a log-probability moves with its logit and the log-sum-exp); the top ids may differ only
    where the replay's values are that close."""
    tol = 2 * 0.125
    with eng.Engine(preset="tiny-test", seed=21, max_batch=48, max_seqs=48, start_scheduler=True) as e:
        res = _burst(e, 40, 5)
    with eng.Engine(preset="tiny-test", seed=21, max_batch=8) as ref:
        V = ref.cfg["vocab_size"]
        for j in range(0, 40, 7):
            r = res[j]
            for i, (ls, row) in enumerate(_replay(ref, _prompt(j, V), r.token_ids)):
                assert abs(r.logprob[i] - ls[r.token_ids[i]]) <= tol, (j, i)
                assert np.all(np.abs(r.top_logprobs[i] - ls[r.top_ids[i]]) <= tol), (j, i)
                kth = ls[_order(row, 5)[-1]]
                assert np.all(ls[r.top_ids[i]] >= kth - tol), (j, i)             # the reported ids are the top 5 up to near-ties


def _wire(e, top, stream, n=24):
    opt = pb.GenerateOptions(temperature=0.0, num_predict=n, raw=True, logprobs=True, top_logprobs=top)
    req = pb.BaseMessage(generate_request=pb.GenerateRequest(model=e.model_name, prompt="Hello wire", stream=stream, options=opt))
    s = eng.greedy(n, ignore_eos=True)
    frames = []
    e.handle_message_stream(req.encode(), s, lambda f: frames.append(pb.BaseMessage.decode(f).generate_response) and False)
    return frames


def _byte_ids(recs):
    """token bytes -> ids of the byte-level tokenizer: byte b is id b + 3, ids past the byte range read "<id>", the
    specials 0..2 have no surface bytes (and no text)"""
    out = []
    for t in recs:
        if len(t.token) == 1:
            out.append(t.token[0] + 3)
        elif t.token:
            m = re.fullmatch(rb"<(\d+)>", t.token)
            assert m, t.token
            out.append(int(m.group(1)))
    return out


def test_wire_carries_one_record_per_streamed_id():
    with eng.Engine(preset="tiny-test", seed=21, max_batch=8, start_scheduler=True) as e:
        for stream in (True, False):
            frames = _wire(e, 3, stream)
            assert frames[-1].done and all(not f.done for f in frames[:-1])
            recs = [t for f in frames for t in f.logprobs]
            assert len(recs) == 24
            text = "".join(f.response for f in frames)
            ids = _byte_ids(recs)
            assert text == e.detokenize(np.array(ids, np.int32))      # the tokens' bytes make up the response text
            for t in recs:
                assert len(t.top_logprobs) == 3 and t.logprob <= 0.0
                assert t.top_logprobs[0].token == t.token and t.top_logprobs[0].logprob == t.logprob      # greedy
            if stream:                                      # each frame carries the records of the ids its text covers
                seen, so_far = [], ""
                for f in frames[:-1]:
                    assert f.logprobs and f.response
                    seen += _byte_ids(f.logprobs)
                    so_far += f.response
                    assert e.detokenize(np.array(seen, np.int32)).startswith(so_far)
        bad = pb.BaseMessage(generate_request=pb.GenerateRequest(model=e.model_name, prompt="x", options=pb.GenerateOptions(
            logprobs=True, top_logprobs=K + 1)))
        with pytest.raises(eng.EngineError) as ei:
            e.handle_message(bad.encode(), eng.greedy(4))
        assert ei.value.status == eng.CL_ERR_INVALID_ARG
        plain = pb.BaseMessage(generate_request=pb.GenerateRequest(model=e.model_name, prompt="x", options=pb.GenerateOptions(
            top_logprobs=5)))
        assert pb.BaseMessage.decode(e.handle_message(plain.encode(), eng.greedy(4))).generate_response.logprobs == []


def test_requests_without_logprobs_add_no_launch():
    with eng.Engine(preset="tiny-test", seed=21, max_batch=8) as e:
        p, g = np.arange(3, 15, dtype=np.int32), eng.greedy(20, ignore_eos=True)
        e.generate_ids(p, g)
        k0 = e.stats()["kernel_launches"]
        e.generate_ids(p, g)
        k1 = e.stats()["kernel_launches"]
        e.generate_ids(p, g, top_logprobs=5)
        k2 = e.stats()["kernel_launches"]
        e.generate_ids(p, g)
        k3 = e.stats()["kernel_launches"]
        assert k3 - k2 == k1 - k0                          # a request that does not ask costs nothing, even after one that did
        assert (k2 - k1) - (k1 - k0) == 20                 # one logprobs launch per generated token
