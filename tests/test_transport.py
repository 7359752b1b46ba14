"""Shared-memory transport (SURVEY 8f F1): the queue contracts of ProcessAgent / ThreadPredictor / ThreadTrainer kept over
shared memory.  CPU only; multi-process cases fork real agent processes."""
import multiprocessing as mp
import os
import queue
import sys
import threading
import time

import numpy as np
import pytest

from ga3c_b200.transport import SlabPredictionQueue, SlabTrainingQueue
from ga3c_b200 import ThreadPredictor, ThreadTrainer
from conftest import REFERENCE

S, A = 24, 3
CTX = mp.get_context("fork")


class FakeModel:
    """p depends on the state so that a reply delivered to the wrong agent is caught."""
    def __init__(self):
        self.batches = []

    def predict_p_and_v(self, x):
        x = np.asarray(x, dtype=np.float32)
        self.batches.append(x.shape[0])
        s = x.sum(axis=1)
        return np.stack([s, s + 1, s + 2], axis=1).astype(np.float32), (2 * s).astype(np.float32)


class FakeServer:
    def __init__(self, training_q=None):
        self.model = FakeModel()
        self.agents = []
        self.training_q = training_q
        self.trained = []

    def train_model(self, x, r, a, x2, done, tid):
        self.trained.append((x.copy(), np.asarray(r).copy(), a.copy(), x2.shape, done.copy()))


def test_prediction_queue_contract_single_process():
    q = SlabPredictionQueue(8, S, A, ctx=CTX)
    try:
        assert q.empty() and q.qsize() == 0
        with pytest.raises(queue.Empty):
            q.get(block=False)
        st = {i: np.full(S, i + 0.5, np.float32) for i in (5, 2, 7)}
        for i, s in st.items():
            q.put((i, s))
        assert not q.empty() and q.qsize() == 3
        got = dict(q.get() for _ in range(3))
        assert set(got) == {5, 2, 7} and all(np.array_equal(got[i], st[i]) for i in st)
        assert q.empty()
        # batch path + replies
        for i, s in st.items():
            q.put((i, s))
        buf = np.zeros((4, S), np.float32)
        ids = q.get_batch(4, buf)
        assert sorted(ids.tolist()) == [2, 5, 7] and all(np.array_equal(buf[k], st[int(i)]) for k, i in enumerate(ids))
        q.reply_batch(ids, np.arange(9, dtype=np.float32).reshape(3, 3), np.array([10, 11, 12], np.float32))
        for k, i in enumerate(ids):
            p, v = q.wait_q(int(i)).get(timeout=1)
            assert np.array_equal(p, np.arange(3 * k, 3 * k + 3)) and v == 10 + k
        assert q.get_batch(4, buf, timeout=0.01) is None
        # cap smaller than what is pending: the rest stays queued, nobody is starved
        for i in range(8):
            q.put((i, np.full(S, i, np.float32)))
        a = q.get_batch(3, buf); b = q.get_batch(3, buf); c = q.get_batch(3, buf)
        assert sorted(a.tolist() + b.tolist() + c.tolist()) == list(range(8))
    finally:
        q.close()


def test_vector_posts_and_waits():
    """post_many / wait_many: a process hosting several agents posts and collects for all of them in one call each."""
    q = SlabPredictionQueue(6, S, A, ctx=CTX)
    try:
        aids = np.array([4, 1, 5])
        states = np.stack([np.full(S, i, np.float32) for i in aids])
        q.post_many(aids, states)
        buf = np.zeros((6, S), np.float32)
        ids = q.get_batch(6, buf)
        assert sorted(ids.tolist()) == [1, 4, 5] and all(buf[k, 0] == i for k, i in enumerate(ids))
        p_out, v_out = np.zeros((3, A), np.float32), np.zeros(3, np.float32)
        assert q.wait_many(aids, p_out, v_out, timeout=0.01) == 0         # nothing replied yet
        q.reply_batch(np.array([4]), np.full((1, A), 4, np.float32), np.array([40], np.float32))
        got = q.wait_many(aids, p_out, v_out, timeout=0.01)               # agent 4 collected, agent 1 still out: resumable
        assert got == 1
        rest = np.array([1, 5])
        q.reply_batch(rest, np.stack([np.full(A, i, np.float32) for i in rest]), rest.astype(np.float32) * 10)
        assert q.wait_many(aids, p_out, v_out, timeout=1, start=got) == 3
        assert np.array_equal(p_out[:, 0], aids) and np.array_equal(v_out, aids * 10.0)
        assert q.get_batch(6, buf, timeout=0.01) is None
    finally:
        q.close()


def test_prediction_queue_random_traffic_against_a_model():
    """Random interleavings of put / post_many / get / get_batch / replies (hypothesis): every request is delivered exactly
    once with the state that was posted, nothing is invented, and the queue ends empty."""
    from hypothesis import given, settings, strategies as st

    ops = st.lists(st.one_of(st.tuples(st.just("put"), st.integers(0, 11)),
                             st.tuples(st.just("many"), st.lists(st.integers(0, 11), min_size=1, max_size=5, unique=True)),
                             st.tuples(st.just("get"), st.just(0)),
                             st.tuples(st.just("batch"), st.integers(1, 6))), max_size=40)

    @settings(max_examples=60, deadline=None)
    @given(ops)
    def run(seq):
        q = SlabPredictionQueue(12, S, A, ctx=CTX)
        q._POLL = 0.0                                   # single-threaded model run: never wait for a producer
        try:
            outstanding, stamp = {}, 0
            buf = np.zeros((6, S), np.float32)

            def deliver(aid, state):
                assert aid in outstanding and state[0] == outstanding.pop(aid)
                q.reply_batch(np.array([aid]), np.zeros((1, A), np.float32), np.array([state[0]], np.float32))
                p, v = q.wait_q(aid).get(timeout=1)
                assert v == state[0]

            for op, arg in seq:
                if op == "put" and arg not in outstanding:
                    stamp += 1
                    outstanding[arg] = float(stamp)
                    q.put((arg, np.full(S, stamp, np.float32)))
                elif op == "many":
                    free = [a for a in arg if a not in outstanding]
                    if free:
                        vals = []
                        for a in free:
                            stamp += 1
                            outstanding[a] = float(stamp)
                            vals.append(np.full(S, stamp, np.float32))
                        q.post_many(np.array(free), np.stack(vals))
                elif op == "get":
                    try:
                        aid, state = q.get(block=False)
                    except queue.Empty:
                        assert not outstanding
                    else:
                        deliver(aid, state)
                elif op == "batch":
                    ids = q.get_batch(arg, buf, timeout=0.0)
                    if ids is None:
                        assert not outstanding
                    else:
                        assert 1 <= ids.size <= arg and len(set(ids.tolist())) == ids.size
                        for k, aid in enumerate(ids):
                            deliver(int(aid), buf[k].copy())
            while outstanding:
                aid, state = q.get(block=False)
                deliver(aid, state)
            assert q.empty() and q.get_batch(6, buf, timeout=0.0) is None
        finally:
            q.close()

    run()


def test_training_queue_contract_and_backpressure():
    tq = SlabTrainingQueue(2, max_rows=6, state_dim=S, num_actions=A, blocks_per_agent=2, ctx=CTX)
    try:
        mine = tq.for_agent(1)
        items = []
        for k in range(2):
            n = 3 + k
            item = (np.random.rand(n, S).astype(np.float32), np.random.rand(n), np.eye(A, dtype=np.float32)[np.arange(n) % A],
                    np.random.rand(n, S).astype(np.float32), np.arange(n) % 2 == 0)
            items.append(item)
            mine.put(item)
        with pytest.raises(queue.Full):                       # ring of 2 blocks is full: Queue(maxsize) behaviour
            mine.put(items[0], timeout=0.05)
        with pytest.raises(ValueError):
            tq.for_agent(0).put((np.zeros((7, S), np.float32), np.zeros(7), np.zeros((7, A), np.float32), None, np.zeros(7, bool)))
        for item in items:
            x, r, a, x2, done = tq.get(timeout=1)
            assert np.array_equal(x, item[0]) and np.array_equal(r, item[1]) and r.dtype == np.float64
            assert np.array_equal(a, item[2]) and np.array_equal(done, item[4]) and x2.shape == (x.shape[0], 0)
        assert tq.empty()
        mine.put(items[0])                                    # blocks were released
        assert tq.qsize() == 1
    finally:
        tq.close()


def test_training_queue_get_batch_follows_the_reference_stop_rule():
    """get_batch: rows are gathered until the count EXCEEDS min_rows (ThreadTrainer.py:49), never beyond the buffer."""
    tq = SlabTrainingQueue(4, max_rows=5, state_dim=S, num_actions=A, blocks_per_agent=2, ctx=CTX)
    try:
        x = np.zeros((12, S), np.float32); r = np.zeros(12); a = np.zeros((12, A), np.float32); d = np.zeros(12, bool)
        assert tq.get_batch(6, x, r, a, d, timeout=0.02) is None
        for aid in range(4):
            n = 3
            tq.for_agent(aid).put((np.full((n, S), aid, np.float32), np.full(n, aid, np.float64),
                                   np.eye(A, dtype=np.float32)[[aid % A] * n], None, np.zeros(n, bool)))
        n = tq.get_batch(6, x, r, a, d, timeout=1)
        assert n == 9 and sorted(set(r[:n].tolist())) == [0.0, 1.0, 2.0]      # 3 + 3 = 6 does not exceed 6: a third block is taken
        assert np.array_equal(x[:n, 0], r[:n]) and np.all(a[:n].sum(axis=1) == 1)
        t0 = time.time()                                                      # one block left: the call keeps waiting for more rows,
        n = tq.get_batch(6, x, r, a, d, timeout=1, stop=lambda: time.time() - t0 > 0.2)   # as the reference would, until told to stop
        assert n == 3 and r[0] == 3.0 and tq.empty()
        for aid in range(4):                                                  # blocks were handed back to their owners
            tq.for_agent(aid).put((np.zeros((5, S), np.float32), np.zeros(5), np.zeros((5, A), np.float32), None, np.zeros(5, bool)), timeout=1)
        small = np.zeros((7, S), np.float32)
        assert tq.get_batch(100, small, r, a, d, timeout=1) == 5              # the second block would not fit 7 rows
    finally:
        tq.close()


def test_training_queue_loses_no_item_when_the_consumer_wraps_past_a_producer():
    """The consumer's cursor runs over the whole slab, so it can take a producer's newer block before an older one; the
    producer's next put must then go to the block that was freed, not overwrite the older item that is still posted."""
    tq = SlabTrainingQueue(2, max_rows=1, state_dim=S, num_actions=A, blocks_per_agent=2, ctx=CTX)
    try:
        x = np.zeros((1, S), np.float32); r = np.zeros(1); a = np.zeros((1, A), np.float32); d = np.zeros(1, bool)

        def put(aid, v):
            tq.for_agent(aid).put((np.full((1, S), v, np.float32), np.full(1, v, np.float64), np.zeros((1, A), np.float32),
                                   None, np.zeros(1, bool)), timeout=1)

        def take():
            n = tq.get_batch(0, x, r, a, d, timeout=0.05)
            return None if n is None else float(r[0])

        put(0, 1.0); assert take() == 1.0              # agent 0's block 0; the cursor moves to block 1
        put(1, 10.0); assert take() == 10.0            # agent 1's block 2; the cursor moves to block 3
        put(0, 2.0); put(0, 3.0)                       # agent 0: item 2 in block 1, item 3 in block 0
        assert take() == 3.0                           # the cursor wraps to block 0 first
        put(0, 4.0)                                    # must not land on block 1, which still holds item 2
        rest = []
        while (v := take()) is not None:
            rest.append(v)
        assert sorted(rest) == [2.0, 4.0]
        assert np.array_equal(x[0], np.full(S, rest[-1], np.float32))
    finally:
        tq.close()


def _agent_proc(aid, pq, tq, n_steps, t_max, out):
    """A ProcessAgent-shaped loop (ProcessAgent.py:102-107, :117-176): predict every step, ship experiences every t_max."""
    rng = np.random.default_rng(aid)
    wait_q = pq.wait_q(aid)
    train_q = tq.for_agent(aid)
    bad = 0
    xs = []
    for t in range(n_steps):
        state = rng.random(S, dtype=np.float32)
        pq.put((aid, state))
        p, v = wait_q.get()
        s = np.float32(state.sum())
        if not (np.allclose(p, [s, s + 1, s + 2], rtol=1e-6) and np.isclose(v, 2 * s, rtol=1e-6)):
            bad += 1
        xs.append(state)
        if len(xs) == t_max:
            x = np.array(xs)
            train_q.put((x, np.full(t_max, aid, np.float64), np.eye(A, dtype=np.float32)[np.arange(t_max) % A], x, np.zeros(t_max, bool)))
            xs = []
    out.put((aid, bad))


def test_agents_in_processes_through_predictor_and_trainer_threads():
    n_agents, n_steps, t_max = 6, 40, 5
    pq = SlabPredictionQueue(n_agents, S, A, ctx=CTX)
    tq = SlabTrainingQueue(n_agents, max_rows=t_max, state_dim=S, num_actions=A, ctx=CTX)
    server = FakeServer(tq)
    out = CTX.Queue()
    pred = ThreadPredictor(server, 0, S, pq)
    trainer = ThreadTrainer(server, 0)
    pred.start(); trainer.start()
    procs = [CTX.Process(target=_agent_proc, args=(i, pq, tq, n_steps, t_max, out)) for i in range(n_agents)]
    try:
        for p in procs:
            p.start()
        res = dict(out.get(timeout=180) for _ in procs)
        for p in procs:
            p.join(timeout=30)
        assert res == {i: 0 for i in range(n_agents)}                    # every reply reached the agent that asked
        # (how many requests share a predictor batch depends on the scheduler, so batch sizes are not asserted here;
        #  test_prediction_queue_contract_single_process pins the batching rule deterministically)
        assert pred.rows == n_agents * n_steps and sum(server.model.batches) == pred.rows
        deadline = time.time() + 60
        while len(server.trained) < n_agents * n_steps // t_max and time.time() < deadline:
            time.sleep(0.01)
        assert len(server.trained) == n_agents * n_steps // t_max
        assert sorted(int(t[1][0]) for t in server.trained) == sorted(list(range(n_agents)) * (n_steps // t_max))
        assert all(t[0].shape == (t_max, S) and t[3] == (t_max, 0) for t in server.trained)
    finally:
        pred.exit_flag = True; trainer.exit_flag = True
        for p in procs:
            if p.is_alive():
                p.terminate()
        time.sleep(0.1)
        pq.close(); tq.close()


def test_trainer_batches_equal_over_queue_and_slab():
    """The slab batch path of ThreadTrainer forms the same batches as the queue path (= the reference rule: concatenate until
    the row count exceeds TRAINING_MIN_BATCH_SIZE) from the same item stream."""
    from ga3c_b200 import Config

    class Cfg(Config):
        TRAINING_MIN_BATCH_SIZE = 7
    rng = np.random.default_rng(4)
    items = []
    for i in range(9):
        n = int(rng.integers(1, 5))
        items.append((rng.random((n, S), dtype=np.float32), rng.random(n), np.eye(A, dtype=np.float32)[rng.integers(0, A, n)],
                      np.zeros((n, 0), np.float32), rng.random(n) < 0.5))
    results = {}
    for mode in ("queue", "slab"):
        tq = queue.Queue() if mode == "queue" else SlabTrainingQueue(1, max_rows=4, state_dim=S, num_actions=A, blocks_per_agent=16, ctx=CTX)
        server = FakeServer(tq)
        th = ThreadTrainer(server, 0, config=Cfg)
        th.start()
        put = tq.put if mode == "queue" else tq.for_agent(0).put
        for it in items:                       # one producer, in order: the slab ring keeps the order of a single agent
            put(it)
        deadline = time.time() + 5
        while sum(t[0].shape[0] for t in server.trained) < sum(it[0].shape[0] for it in items) - 7 and time.time() < deadline:
            time.sleep(0.01)
        th.exit_flag = True
        time.sleep(0.15)
        results[mode] = server.trained
        if mode == "slab":
            tq.close()
    q, s_ = results["queue"], results["slab"]
    assert len(q) >= 2 and len(s_) >= len(q)
    for bq, bs in zip(q, s_):                  # full batches are identical; only a trailing partial batch may differ (stop flag)
        assert bq[0].shape[0] > 7
        assert np.array_equal(bq[0], bs[0]) and np.array_equal(bq[1], bs[1]) and np.array_equal(bq[2], bs[2]) and np.array_equal(bq[4], bs[4])


@pytest.mark.reference
def test_reference_threads_run_unmodified_over_the_slab_queues():
    """The reference's own ThreadPredictor / ThreadTrainer (imported from $GA3C_REFERENCE) over the slab objects."""
    sys.dont_write_bytecode = True
    sys.path.insert(0, REFERENCE)
    try:
        from ThreadPredictor import ThreadPredictor as RefPredictor
        from ThreadTrainer import ThreadTrainer as RefTrainer
        from Config import Config as RefConfig
    finally:
        sys.path.remove(REFERENCE)
    n_agents = 5
    pq = SlabPredictionQueue(n_agents, S, A, ctx=CTX)
    tq = SlabTrainingQueue(n_agents, max_rows=4, state_dim=S, num_actions=A, ctx=CTX)
    server = FakeServer(tq)

    class Agent:
        def __init__(self, i):
            self.wait_q = pq.wait_q(i)
    server.agents = [Agent(i) for i in range(n_agents)]
    old = (RefConfig.USE_REPLAY_MEMORY, RefConfig.TRAIN_MODELS, RefConfig.TRAINING_MIN_BATCH_SIZE, getattr(RefConfig, "USE_NETWORK_TESTER", False))
    RefConfig.USE_REPLAY_MEMORY, RefConfig.TRAIN_MODELS, RefConfig.TRAINING_MIN_BATCH_SIZE, RefConfig.USE_NETWORK_TESTER = False, True, 0, False
    pred, trainer = RefPredictor(server, 0, S, pq), RefTrainer(server, 0)
    pred.daemon = trainer.daemon = True
    try:
        pred.start(); trainer.start()
        states = {i: np.full(S, 0.25 * (i + 1), np.float32) for i in range(n_agents)}
        for i, s in states.items():
            pq.put((i, s))
        for i, s in states.items():
            p, v = server.agents[i].wait_q.get(timeout=5)
            assert np.allclose(p, [s.sum(), s.sum() + 1, s.sum() + 2]) and np.isclose(v, 2 * s.sum())
        x = np.random.rand(4, S).astype(np.float32)
        tq.for_agent(3).put((x, np.ones(4), np.eye(A, dtype=np.float32)[[0, 1, 2, 0]], x, np.zeros(4, bool)))
        deadline = time.time() + 5
        while not server.trained and time.time() < deadline:
            time.sleep(0.01)
        assert len(server.trained) == 1 and np.array_equal(server.trained[0][0], x)
    finally:
        pred.exit_flag = True; trainer.exit_flag = True
        RefConfig.USE_REPLAY_MEMORY, RefConfig.TRAIN_MODELS, RefConfig.TRAINING_MIN_BATCH_SIZE, RefConfig.USE_NETWORK_TESTER = old
        pq.put((0, states[0]))           # unblock the reference predictor so its loop sees exit_flag
        tq.for_agent(0).put((x, np.ones(4), np.eye(A, dtype=np.float32)[[0, 1, 2, 0]], x, np.zeros(4, bool)))
        time.sleep(0.2)
        pq.close(); tq.close()
