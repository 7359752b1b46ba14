"""Shared-memory transport under the predictor / trainer queue contracts (SURVEY.md 8f F1).

The reference moves every state through `multiprocessing.Queue`s: one pickle + pipe write + unpickle per item
(`ProcessAgent.py:102-107`, `ThreadPredictor.py:46-66`, `Server.py:73-75`), which caps the loop at a few thousand
predictions per second whatever the network costs (SURVEY 0.5).  These classes keep the contracts -- items `(id, state)` in,
`(p_row, v)` back on the agent's own one-slot `wait_q`, items `(x_, r_, a_, x2_, done_)` to the trainer, `put` / `get` /
`empty` / bounded capacity -- but the payload never leaves shared memory:

    SlabPredictionQueue   one state row per agent + a `pending` byte per agent.  `put((id, state))` copies the state into
                          row `id` and raises the byte; the consumer scans the bytes.  One outstanding request per agent
                          (that is what wait_q's maxsize = 1 enforces in the reference, ProcessAgent.py:64), so every byte
                          has one writer per transition and no lock or atomic is needed across processes.
    SlabReplySlot         `wait_q` of one agent: `put((p, v))` writes the agent's reply row and wakes it.
    SlabTrainingQueue     each agent owns a small ring of experience blocks; `put` copies the arrays into the next free
                          block (blocking while the ring is full = Queue(maxsize) back-pressure) and posts it.

The reference's own `ThreadPredictor` / `ThreadTrainer` / `ProcessAgent` run unmodified over these objects (duck-typed
queues; tests/test_transport.py does exactly that when GA3C_REFERENCE is set).  `ga3c_b200.ThreadPredictor` also uses
the batch calls (`get_batch`, `reply_batch`): one gather into a pinned buffer and one reply scatter per batch instead of
128 queue operations.  Blocking uses OS semaphores (no busy-waiting: 256 agents share the host's cores).

Memory ordering: a producer writes the payload, then the flag byte; x86-64 keeps stores in order (TSO) and numpy's copies
are plain stores, so a consumer that sees the flag sees the payload.  That is an x86-64 property: on a weakly ordered host
(aarch64, e.g. Grace-based Blackwell nodes) a consumer on the flag-polling path could see `pending = 1` before the row.  The
module refuses to import there rather than hand over stale frames (a port needs a release fence after the payload copy and
an acquire fence after the flag read: take the semaphore permit before touching the row).
"""
from __future__ import annotations

import mmap
import multiprocessing as mp
import platform
import threading
from multiprocessing import shared_memory

import numpy as np

if platform.machine().lower() not in ("x86_64", "amd64", "i686", "i386"):      # see "Memory ordering" above
    raise ImportError(f"ga3c_b200.transport relies on x86-64 store ordering; this host is {platform.machine()!r}")


class _Shm:
    """A shared block viewed as one numpy array.  Default: an anonymous MAP_SHARED mapping, inherited by forked children
    (how the reference starts its agents on Linux) and not subject to the size of /dev/shm (64 MB in a default container,
    far less than a training slab of fp32 frames).  named=True uses multiprocessing.shared_memory instead, which
    re-attaches by name when the object is pickled into a spawned process."""

    def __init__(self, shape, dtype, named=False):
        self.shape, self.dtype = tuple(shape), np.dtype(dtype)
        nbytes = max(1, int(np.prod(self.shape)) * self.dtype.itemsize)
        self._named = bool(named)
        if named:
            self._shm = shared_memory.SharedMemory(create=True, size=nbytes)
            buf = self._shm.buf
        else:
            self._shm = mmap.mmap(-1, nbytes)               # MAP_SHARED | MAP_ANONYMOUS, zero-filled
            buf = self._shm
        self._owner = True
        self.array = np.ndarray(self.shape, dtype=self.dtype, buffer=buf)

    def __getstate__(self):
        if not self._named:
            raise TypeError("anonymous shared mapping: pass the transport objects to forked children (or build them with "
                            "named=True to pickle them into spawned processes)")
        return {"name": self._shm.name, "shape": self.shape, "dtype": self.dtype.str}

    def __setstate__(self, st):
        self.shape, self.dtype = st["shape"], np.dtype(st["dtype"])
        self._named = True
        self._shm = shared_memory.SharedMemory(name=st["name"])
        self._owner = False
        self.array = np.ndarray(self.shape, dtype=self.dtype, buffer=self._shm.buf)

    def close(self):
        self.array = None
        try:
            self._shm.close()
            if self._named and self._owner:
                self._shm.unlink()
        except Exception:
            pass


class SlabPredictionQueue:
    """`prediction_q` (Server.py:74): items `(agent_id, state)`; ids 0 .. num_agents-1."""

    def __init__(self, num_agents, state_dim, num_actions, dtype=np.float32, ctx=None, named=False):
        ctx = ctx or mp.get_context()
        self.num_agents, self.state_dim, self.num_actions = int(num_agents), int(state_dim), int(num_actions)
        self._states = _Shm((num_agents, state_dim), dtype, named)
        self._pending = _Shm((num_agents,), np.uint8, named)
        self._reply_p = _Shm((num_agents, num_actions), np.float32, named)
        self._reply_v = _Shm((num_agents,), np.float32, named)
        self._work = ctx.Semaphore(0)                       # one release per posted request
        self._wake = [ctx.Semaphore(0) for _ in range(num_agents)]
        self._lock = threading.Lock()                       # consumers are threads of one process
        self._cursor = 0

    def __getstate__(self):
        d = self.__dict__.copy()
        d["_lock"] = None
        return d

    def __setstate__(self, d):
        self.__dict__.update(d)
        self._lock = threading.Lock()

    # ---- producer side (agent processes) ----
    def _check_id(self, aid):
        # ids are rows of the slab: an id outside 0 .. num_agents-1 (e.g. the reference's NETWORK_TESTER_ID = 100 with fewer
        # agents, ThreadPredictor.py:64-66) must not alias another agent's row through negative / wrapped indexing
        if not 0 <= int(aid) < self.num_agents:
            raise IndexError(f"agent id {aid} outside 0..{self.num_agents - 1}: size the slab queue for every producer id")

    def put(self, item, block=True, timeout=None):
        """One outstanding request per agent (wait_q has maxsize 1, ProcessAgent.py:64), so a row is always free when its
        agent puts: `block` / `timeout` are accepted for Queue compatibility and never needed."""
        aid, state = item
        self._check_id(aid)
        self._states.array[aid] = np.asarray(state).reshape(-1)
        self._pending.array[aid] = 1
        self._work.release()

    def state_row(self, aid):
        """The agent's own row, for environments that render straight into shared memory (then call `post`)."""
        self._check_id(aid)
        return self._states.array[aid]

    def post(self, aid):
        self._check_id(aid)
        self._pending.array[aid] = 1
        self._work.release()

    def post_many(self, aids, states):
        """A process that hosts several agents posts one request per agent in one go: rows states[i] -> agent aids[i].
        One wake-up for the whole group (the consumer takes every pending row it sees)."""
        self._states.array[aids] = states
        self._pending.array[aids] = 1
        for _ in range(len(aids)):          # one permit per request, as put() does: consumers return one permit per row taken
            self._work.release()

    def wait_many(self, aids, p_out, v_out, timeout=None, start=0):
        """Waits for the replies of aids[start:], in order.  Returns how many of `aids` have been collected so far: len(aids)
        when all replies are in (p_out[i], v_out[i] filled), less after a time-out -- call again with start = that number."""
        for i in range(start, len(aids)):
            if not self._wake[int(aids[i])].acquire(True, timeout):
                return i
        p_out[...] = self._reply_p.array[aids]
        v_out[...] = self._reply_v.array[aids]
        return len(aids)

    def wait_q(self, aid):
        return SlabReplySlot(self, aid)

    # ---- consumer side (predictor threads) ----
    def empty(self):
        return not self._pending.array.any()

    def qsize(self):
        return int(self._pending.array.sum())

    def _take(self, max_n):
        """Indices of up to max_n pending requests, oldest-cursor-first; caller holds the lock."""
        idx = np.flatnonzero(self._pending.array.copy())    # snapshot: producers keep raising bytes while we look
        if idx.size == 0:
            return idx
        if idx.size > max_n:
            k = int(np.searchsorted(idx, self._cursor))
            idx = np.concatenate((idx[k:], idx[:k]))[:max_n]
        self._cursor = (int(idx[-1]) + 1) % self.num_agents
        return idx

    _POLL = 0.05       # the semaphore is a wake-up hint: a consumer also looks at the bytes every _POLL seconds, so a lost or
                       # stolen permit costs latency, never a request

    def get(self, block=True, timeout=None):
        """-> (agent_id, state copy).  Blocks like Queue.get()."""
        import queue
        import time
        deadline = None if timeout is None else time.monotonic() + timeout
        while True:
            if block:
                left = self._POLL if deadline is None else max(0.0, min(self._POLL, deadline - time.monotonic()))
                self._work.acquire(True, left)
            else:
                self._work.acquire(False)
            with self._lock:
                idx = self._take(1)
                if idx.size:
                    aid = int(idx[0])
                    state = self._states.array[aid].copy()
                    self._pending.array[aid] = 0
                    return aid, state
            if not block or (deadline is not None and time.monotonic() >= deadline):
                raise queue.Empty

    def get_batch(self, max_n, out_states, timeout=None):
        """Blocks for the first request, then takes whatever is pending (at most max_n, ThreadPredictor.py:50-55): gathers
        the rows into out_states[:n] and returns the agent ids (int array of length n >= 1), or None on timeout."""
        import time
        deadline = None if timeout is None else time.monotonic() + timeout
        while True:
            left = self._POLL if deadline is None else max(0.0, min(self._POLL, deadline - time.monotonic()))
            got = self._work.acquire(True, left)
            with self._lock:
                idx = self._take(max_n)
                if idx.size:
                    np.take(self._states.array, idx, axis=0, out=out_states[:idx.size])
                    self._pending.array[idx] = 0
            if idx.size:
                for _ in range(idx.size - (1 if got else 0)):       # one permit per row taken (best effort)
                    self._work.acquire(False)
                return idx
            if deadline is not None and time.monotonic() >= deadline:
                return None

    def reply_batch(self, ids, p, v):
        """(p[i], v[i]) to agent ids[i]'s wait_q, for a whole batch."""
        self._reply_p.array[ids] = p
        self._reply_v.array[ids] = v
        wake = self._wake
        for aid in ids:
            wake[int(aid)].release()

    def close(self):
        for s in (self._states, self._pending, self._reply_p, self._reply_v):
            s.close()


class SlabReplySlot:
    """`agent.wait_q` (ProcessAgent.py:64, Queue(maxsize=1)): the predictor `put`s `(p_row, v)`, the agent `get`s it."""

    def __init__(self, q: SlabPredictionQueue, aid: int):
        self._q, self._aid = q, int(aid)

    def put(self, item, block=True, timeout=None):
        p, v = item
        self._q._reply_p.array[self._aid] = p
        self._q._reply_v.array[self._aid] = v
        self._q._wake[self._aid].release()

    def get(self, block=True, timeout=None):
        if not self._q._wake[self._aid].acquire(block, timeout):
            import queue
            raise queue.Empty
        return self._q._reply_p.array[self._aid].copy(), self._q._reply_v.array[self._aid].copy()[()]


class SlabTrainingQueue:
    """`training_q` (Server.py:73): items `(x_, r_, a_, x2_, done_)` from ProcessAgent.run (ProcessAgent.py:175).

    Every producer (agent id) owns `blocks_per_agent` blocks of `max_rows` rows.  `put` needs the producer's id: bind it once
    with `for_agent(id)` (what an agent process holds as its `training_q`).  x2_ is shipped only with ship_next_state=True
    (the A3C networks ignore it, NetworkVP.py:254-257); otherwise the consumer gets a zero-width array, which the
    reference ThreadTrainer concatenates without complaint."""

    def __init__(self, num_agents, max_rows, state_dim, num_actions, blocks_per_agent=2, dtype=np.float32,
                 ship_next_state=False, ctx=None, named=False):
        ctx = ctx or mp.get_context()
        self.num_agents, self.max_rows, self.state_dim, self.num_actions = num_agents, max_rows, state_dim, num_actions
        self.blocks = int(blocks_per_agent)
        nb = num_agents * self.blocks
        self._x = _Shm((nb, max_rows, state_dim), dtype, named)
        self._x2 = _Shm((nb, max_rows, state_dim if ship_next_state else 0), dtype, named)
        self._r = _Shm((nb, max_rows), np.float64, named)   # r_ arrives as float64 (ProcessAgent.py:99)
        self._a = _Shm((nb, max_rows, num_actions), np.float32, named)
        self._done = _Shm((nb, max_rows), np.bool_, named)
        self._rows = _Shm((nb,), np.int32, named)
        self._posted = _Shm((nb,), np.uint8, named)
        self._work = ctx.Semaphore(0)
        self._free = [ctx.Semaphore(self.blocks) for _ in range(num_agents)]
        self._next = [0] * num_agents                       # per-producer cursor (each producer only touches its own)
        self._lock = threading.Lock()
        self._cursor = 0
        self.ship_next_state = bool(ship_next_state)

    def __getstate__(self):
        d = self.__dict__.copy()
        d["_lock"] = None
        return d

    def __setstate__(self, d):
        self.__dict__.update(d)
        self._lock = threading.Lock()

    def for_agent(self, aid):
        return _AgentTrainingQueue(self, aid)

    def put_from(self, aid, item, block=True, timeout=None):
        x, r, a, x2, done = item
        if not 0 <= int(aid) < self.num_agents:
            raise IndexError(f"agent id {aid} outside 0..{self.num_agents - 1}")
        n = int(np.asarray(x).shape[0])
        if n > self.max_rows:
            raise ValueError(f"training item of {n} rows exceeds max_rows={self.max_rows} (Config.TIME_MAX + 1)")
        if not self._free[aid].acquire(block, timeout):     # ring full: Queue(maxsize) back-pressure
            import queue
            raise queue.Full
        # the consumer takes blocks in slab order from its cursor, not in this producer's order: the block after the last one
        # written may still be posted while an earlier one was taken (the permit guarantees that one block is free)
        k = self._next[aid]
        while self._posted.array[aid * self.blocks + k]:
            k = (k + 1) % self.blocks
        b = aid * self.blocks + k
        self._next[aid] = (k + 1) % self.blocks
        self._x.array[b, :n] = np.asarray(x).reshape(n, -1)
        if self.ship_next_state:
            self._x2.array[b, :n] = np.asarray(x2).reshape(n, -1)
        self._r.array[b, :n] = r
        self._a.array[b, :n] = np.asarray(a).reshape(n, -1)
        self._done.array[b, :n] = done
        self._rows.array[b] = n
        self._posted.array[b] = 1
        self._work.release()

    def empty(self):
        return not self._posted.array.any()

    def qsize(self):
        return int(self._posted.array.sum())

    def get(self, block=True, timeout=None):
        """-> (x_, r_, a_, x2_, done_) copies, like Queue.get()."""
        import queue
        import time
        deadline = None if timeout is None else time.monotonic() + timeout
        while True:
            if block:
                self._work.acquire(True, 0.05 if deadline is None else max(0.0, min(0.05, deadline - time.monotonic())))
            else:
                self._work.acquire(False)
            item = None
            with self._lock:
                idx = np.flatnonzero(self._posted.array.copy())     # snapshot (see SlabPredictionQueue._take)
                if idx.size:
                    k = int(np.searchsorted(idx, self._cursor)) % idx.size
                    b = int(idx[k])
                    self._cursor = (b + 1) % self._posted.array.size
                    n = int(self._rows.array[b])
                    item = (self._x.array[b, :n].copy(), self._r.array[b, :n].copy(), self._a.array[b, :n].copy(),
                            self._x2.array[b, :n].copy(), self._done.array[b, :n].copy())
                    self._posted.array[b] = 0
            if item is not None:
                self._free[b // self.blocks].release()
                return item
            if not block or (deadline is not None and time.monotonic() >= deadline):
                raise queue.Empty

    def get_batch(self, min_rows, x_out, r_out, a_out, done_out, timeout=None, stop=None):
        """ThreadTrainer.py:48-59 in one call: blocks for the first item, then keeps taking posted blocks until the row count
        EXCEEDS min_rows (the reference loops `while batch_size <= TRAINING_MIN_BATCH_SIZE`, however long that takes), copying
        the rows straight into the caller's (pinned) arrays -- one copy per row instead of get() + np.concatenate + staging.
        Stops early when the next block would not fit x_out.  `timeout` bounds the wait for the FIRST item only (None is
        returned when nothing arrived); `stop()` is polled every 50 ms and ends the call with the rows gathered so far."""
        import time
        deadline = None if timeout is None else time.monotonic() + timeout
        cap, n = x_out.shape[0], 0
        while True:
            left = 0.05 if deadline is None else max(0.0, min(0.05, deadline - time.monotonic()))
            got = self._work.acquire(True, left)
            taken = 0
            with self._lock:
                idx = np.flatnonzero(self._posted.array.copy())
                if idx.size:
                    k = int(np.searchsorted(idx, self._cursor)) % idx.size
                    for b in np.concatenate((idx[k:], idx[:k])):
                        b = int(b)
                        rows = int(self._rows.array[b])
                        if n + rows > cap:
                            break
                        x_out[n:n + rows] = self._x.array[b, :rows]
                        r_out[n:n + rows] = self._r.array[b, :rows]
                        a_out[n:n + rows] = self._a.array[b, :rows]
                        done_out[n:n + rows] = self._done.array[b, :rows]
                        self._posted.array[b] = 0
                        self._free[b // self.blocks].release()
                        self._cursor = (b + 1) % self._posted.array.size
                        n += rows
                        taken += 1
                        if n > min_rows:
                            break
            for _ in range(taken - (1 if got else 0)):          # one permit per block taken (best effort, see get_batch above)
                self._work.acquire(False)
            if n > min_rows or (n > 0 and taken == 0 and idx.size > 0):    # enough rows, or the next block does not fit
                return n
            if n == 0 and deadline is not None and time.monotonic() >= deadline:
                return None
            if stop is not None and stop():
                return n if n else None

    def close(self):
        for s in (self._x, self._x2, self._r, self._a, self._done, self._rows, self._posted):
            s.close()


class _AgentTrainingQueue:
    """What one agent holds as `training_q`: `put(item)` with the agent's id bound."""

    def __init__(self, q: SlabTrainingQueue, aid: int):
        self._q, self._aid = q, int(aid)

    def put(self, item, block=True, timeout=None):
        self._q.put_from(self._aid, item, block, timeout)
