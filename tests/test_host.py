"""CPU tests (`-m "not gpu"`) of the boundary and the host logic: the C-ABI library loads and exports
every symbol include/ga3c_b200.h declares (no compute calls), the batching threads keep the
reference's queue contracts, and -- where $GA3C_REFERENCE is set -- behave like the reference's
own ThreadPredictor / ThreadTrainer on the same queue traffic."""
import ctypes
import os
import queue
import re
import sys
import time

import numpy as np
import pytest

from conftest import ROOT, REFERENCE


# ---------------------------------------------------------------- C ABI
def _header_symbols():
    src = open(os.path.join(ROOT, "include", "ga3c_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ga3c_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_header_symbol():
    from ga3c_b200 import _capi
    lib = ctypes.CDLL(_capi.LIB_PATH)
    syms = _header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/ga3c_b200.h but not exported"
    assert sorted(_capi.SIGNATURES) == syms               # the ctypes table covers the header exactly
    assert _capi.load().ga3c_abi_version() >= 1


def test_header_compiles_as_plain_c(tmp_path):
    """The boundary is plain C: no C++ / torch types in the signatures."""
    import subprocess
    c = tmp_path / "t.c"
    c.write_text('#include "ga3c_b200.h"\nint main(void){ga3c_config c; (void)c; return sizeof(ga3c_config)==32?0:1;}\n')
    exe = tmp_path / "t"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(c), "-c", "-o",
                    str(exe)], check=True)


def test_config_struct_layouts_match_the_ctypes_binding(tmp_path):
    """The C structs of include/ga3c_b200.h and their ctypes mirrors (ga3c_b200/_capi.py) must agree field by field: a
    silent mismatch would hand the library shifted knobs.  A gcc-compiled probe prints sizeof / offsetof."""
    import ctypes as C
    import subprocess
    from ga3c_b200 import _capi
    fields = {"ga3c_config": [f for f, _ in _capi.ga3c_config._fields_],
              "ga3c_mlp_config": [f for f, _ in _capi.ga3c_mlp_config._fields_]}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "ga3c_b200.h"', 'int main(void){']
    for st, fs in fields.items():
        lines.append(f'printf("{st} %zu\\n", sizeof({st}));')
        for f in fs:
            lines.append(f'printf("{st}.{f} %zu\\n", offsetof({st}, {f}));')
    lines.append('return 0;}')
    c = tmp_path / "probe.c"
    c.write_text("\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(c), "-o", str(exe)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for st, fs in fields.items():
        cls = getattr(_capi, st)
        assert int(out[st]) == C.sizeof(cls), (st, out[st], C.sizeof(cls))
        for f in fs:
            assert int(out[f"{st}.{f}"]) == getattr(cls, f).offset, (st, f)


def test_no_cpu_fallback_without_gpu():
    """On a box without a GPU constructing a Network must fail loudly, not fall back."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import ga3c_b200
    from ga3c_b200 import _capi
    with pytest.raises(_capi.Ga3cError):
        ga3c_b200.Network("gpu:0", "t", 6)


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "ga3c_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                assert "oracle" not in open(os.path.join(dirpath, f)).read(), f


def test_parse_device():
    from ga3c_b200.network import _parse_device
    assert _parse_device("gpu:0") == 0 and _parse_device("/gpu:3") == 3 and _parse_device("cuda:1") == 1
    assert _parse_device("GPU") == 0 and _parse_device(2) == 2
    with pytest.raises(ValueError):
        _parse_device("cpu:0")


def test_annealing_matches_server_loop():
    """Server.py:168-175: linear in the episode count, clamped at ANNEALING_EPISODE_COUNT - 1."""
    from ga3c_b200 import Config
    from ga3c_b200.config import annealed

    class Cfg(Config):
        LEARNING_RATE_START, LEARNING_RATE_END = 3e-4, 1e-4
        BETA_START, BETA_END = 0.01, 0.002
        ANNEALING_EPISODE_COUNT = 1000
    for ep in (0, 1, 500, 999, 1000, 50000):
        lr_mult = (Cfg.LEARNING_RATE_END - Cfg.LEARNING_RATE_START) / Cfg.ANNEALING_EPISODE_COUNT
        beta_mult = (Cfg.BETA_END - Cfg.BETA_START) / Cfg.ANNEALING_EPISODE_COUNT
        step = min(ep, Cfg.ANNEALING_EPISODE_COUNT - 1)
        assert annealed(Cfg, ep) == (Cfg.LEARNING_RATE_START + lr_mult * step, Cfg.BETA_START + beta_mult * step)
    assert annealed(Config, 12345) == (Config.LEARNING_RATE_START, Config.BETA_START)     # START == END by default


def test_config_matches_reference_defaults():
    """Every knob the path reads has the reference's default (Config.py)."""
    from ga3c_b200 import Config
    if not os.path.isdir(REFERENCE):
        pytest.skip("reference not present")
    sys.dont_write_bytecode = True
    sys.path.insert(0, REFERENCE)
    try:
        import Config as RC
    finally:
        sys.path.remove(REFERENCE)
    ref = RC.Config
    skip = {"PREDICTORS", "TRAINERS", "AGENTS"}            # machine-dependent in the fork
    for k, v in vars(Config).items():
        if k.startswith("_") or k in skip or not hasattr(ref, k):
            continue
        assert getattr(ref, k) == v, k


# ---------------------------------------------------------------- batching threads with a fake model
class FakeModel:
    """Deterministic stand-in so the thread logic is testable without a GPU: p row = softmax-free
    function of the state, v = state mean."""
    def __init__(self, a=6):
        self.a = a
        self.calls = []
        self.trained = []

    def predict_p_and_v(self, x):
        self.calls.append(x.shape[0])
        p = np.tile(np.arange(self.a, dtype=np.float32), (x.shape[0], 1)) + x[:, :1]
        return [p, x.mean(axis=1)]

    def train(self, x, r, a, x2, done, tid):
        self.trained.append((x.copy(), np.asarray(r).copy(), a.copy(), tid))


class Agent:
    def __init__(self):
        self.wait_q = queue.Queue(maxsize=1)


class Server:
    def __init__(self, n):
        self.model = FakeModel()
        self.agents = [Agent() for _ in range(n)]
        self.training_q = queue.Queue(maxsize=100)

    def train_model(self, x_, r_, a_, x2_, done_, trainer_id):
        self.model.train(x_, r_, a_, x2_, done_, trainer_id)


def _drive_predictor(cls, **kw):
    srv = Server(50)
    pq = queue.Queue(maxsize=100)
    rng = np.random.default_rng(0)
    states = rng.standard_normal((50, 12)).astype(np.float32)
    for i in range(50):
        pq.put((i, states[i]))
    th = cls(srv, 0, 12, pq, **kw) if kw else cls(srv, 0, 12, pq)
    th.daemon = True
    th.start()
    out = [srv.agents[i].wait_q.get(timeout=20) for i in range(50)]
    th.exit_flag = True
    return states, out, srv.model.calls


def test_thread_predictor_contract():
    from ga3c_b200 import ThreadPredictor
    states, out, calls = _drive_predictor(ThreadPredictor)
    assert sum(calls) == 50 and max(calls) <= 128
    for i, (p, v) in enumerate(out):
        assert np.array_equal(p, np.arange(6, dtype=np.float32) + states[i, 0]) and v == states[i].mean()


def test_thread_predictor_respects_batch_cap():
    from ga3c_b200 import ThreadPredictor, Config

    class Cfg(Config):
        PREDICTION_BATCH_SIZE = 16
    _, _, calls = _drive_predictor(ThreadPredictor, config=Cfg)
    assert max(calls) <= 16 and sum(calls) == 50


@pytest.mark.reference
def test_thread_predictor_matches_reference_class():
    """The reference's own ThreadPredictor (ThreadPredictor.py:34-66), unmodified, on the same traffic."""
    sys.dont_write_bytecode = True
    sys.path.insert(0, REFERENCE)
    try:
        import ThreadPredictor as RTP
    finally:
        sys.path.remove(REFERENCE)
    from ga3c_b200 import ThreadPredictor
    s1, o1, _ = _drive_predictor(RTP.ThreadPredictor)
    s2, o2, _ = _drive_predictor(ThreadPredictor)
    for (p1, v1), (p2, v2) in zip(o1, o2):
        assert np.array_equal(p1, p2) and v1 == v2


def _drive_trainer(cls, min_batch, **kw):
    srv = Server(1)
    rng = np.random.default_rng(1)
    items = []
    for n in (5, 3, 7, 2, 9, 4):
        items.append((rng.standard_normal((n, 12)).astype(np.float32), rng.standard_normal(n),
                      np.eye(6, dtype=np.float32)[rng.integers(0, 6, n)], rng.standard_normal((n, 12)).astype(np.float32),
                      np.zeros(n, bool)))
    for it in items:
        srv.training_q.put(it)
    th = cls(srv, 3, **kw) if kw else cls(srv, 3)
    th.daemon = True
    th.start()
    t0 = time.time()
    while not srv.training_q.empty() and time.time() - t0 < 20:
        time.sleep(0.01)
    time.sleep(0.2)
    th.exit_flag = True
    return items, srv.model.trained


def test_thread_trainer_contract_min_batch_zero():
    from ga3c_b200 import ThreadTrainer
    items, trained = _drive_trainer(ThreadTrainer, 0)
    assert [t[0].shape[0] for t in trained] == [5, 3, 7, 2, 9, 4]           # one agent batch per step
    assert all(t[3] == 3 for t in trained)
    assert np.array_equal(trained[2][0], items[2][0]) and trained[2][1].dtype == np.float64


def test_thread_trainer_concatenates_until_exceeding_min():
    from ga3c_b200 import ThreadTrainer, Config

    class Cfg(Config):
        TRAINING_MIN_BATCH_SIZE = 8
    items, trained = _drive_trainer(ThreadTrainer, 8, config=Cfg)
    assert [t[0].shape[0] for t in trained] == [15, 11]                     # 5+3+7 > 8 ; 2+9 > 8 ; 4 waits
    assert np.array_equal(trained[0][0], np.concatenate([items[0][0], items[1][0], items[2][0]]))
    assert np.array_equal(trained[1][2], np.concatenate([items[3][2], items[4][2]]))


@pytest.mark.reference
def test_thread_trainer_matches_reference_class():
    sys.dont_write_bytecode = True
    sys.path.insert(0, REFERENCE)
    try:
        import ThreadTrainer as RTT
    finally:
        sys.path.remove(REFERENCE)
    from ga3c_b200 import ThreadTrainer
    _, t1 = _drive_trainer(RTT.ThreadTrainer, 0)
    _, t2 = _drive_trainer(ThreadTrainer, 0)
    assert len(t1) == len(t2)
    for a, b in zip(t1, t2):
        assert all(np.array_equal(a[k], b[k]) for k in range(3)) and a[3] == b[3]


def test_stage_h2d_host_copy_is_exact_for_ragged_sizes_and_thread_counts():
    """ga3c_stage_h2d (include/ga3c_b200.h) with dst_dev = NULL is the host half alone: the pageable -> staging copy by the
    library's worker threads in 512 KB pieces with streaming stores.  Byte-exact for sizes that are not multiples of the
    piece, the chunk or 64 bytes, for unaligned source and destination, for every thread count, and for concurrent callers
    (the two trainer threads of the reference's Server queue on one job at a time)."""
    import threading
    from ga3c_b200 import _capi
    lib = _capi.load()
    rng = np.random.default_rng(5)
    for nbytes, so, do, threads, chunk in ((0, 0, 0, 4, 0), (1, 0, 0, 4, 0), (63, 1, 3, 2, 0), (512 * 1024, 0, 0, 3, 0),
                                           (512 * 1024 + 1, 5, 0, 3, 1 << 20), (3 * 1024 * 1024 + 77, 0, 9, 8, 1 << 20),
                                           (9 * 1024 * 1024 + 13, 3, 1, 5, 0), (20 * 1024 * 1024, 0, 0, 1, 0),
                                           (20 * 1024 * 1024 + 5, 7, 64, 32, 2 << 20)):
        src = rng.integers(0, 256, size=nbytes + so + 64, dtype=np.uint8)
        dst = np.full(nbytes + do + 128, 0xAB, dtype=np.uint8)
        rc = lib.ga3c_stage_h2d(None, dst.ctypes.data + do, src.ctypes.data + so, nbytes, chunk, threads, None)
        assert rc == 0, lib.ga3c_last_error()
        assert np.array_equal(dst[do:do + nbytes], src[so:so + nbytes]), (nbytes, so, do, threads)
        assert (dst[:do] == 0xAB).all() and (dst[do + nbytes:] == 0xAB).all()       # nothing outside the range is touched
    assert lib.ga3c_stage_h2d(None, None, None, 16, 0, 2, None) != 0 and b"null buffer" in lib.ga3c_last_error()

    srcs = [rng.integers(0, 256, size=6 * 1024 * 1024 + 11 * i, dtype=np.uint8) for i in range(4)]
    dsts = [np.zeros_like(s) for s in srcs]
    def call(i):
        for _ in range(5):
            assert lib.ga3c_stage_h2d(None, dsts[i].ctypes.data, srcs[i].ctypes.data, srcs[i].nbytes, 1 << 20, 2 + i, None) == 0
    ts = [threading.Thread(target=call, args=(i,)) for i in range(4)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert all(np.array_equal(d, s) for d, s in zip(dsts, srcs))


def test_arena_mixin_named_tensors_slots_checkpoints_and_log(tmp_path, monkeypatch):
    """ga3c_b200/_arena.py -- the host plumbing the conv Network and the MLP networks share -- over an in-memory arena (no GPU):
    the arena as TF-named tensors (get / set, shape errors), both optimizers' slots, the checkpoint round trip with the
    reference's file naming (NetworkVP.py:267-282: latest checkpoint or Config.LOAD_EPISODE, episode number returned, slots of
    the second optimizer only with DUAL_RMSPROP) and the scalar log of NetworkVP.py:259-265."""
    from ga3c_b200._arena import ArenaNetworkMixin

    class Cfg:
        LOAD_EPISODE = 0

    class Fake(ArenaNetworkMixin):
        def __init__(self, name, dual=False):
            self.model_name, self.config, self._dual = name, Cfg, dual
            self.learning_rate, self.beta = 3e-4, 0.01
            self._table = {"dense1/w:0": (0, (3, 4)), "dense1/b:0": (64, (4,)), "logits_v/w:0": (128, (4, 1))}
            self._arenas = {w: np.zeros(192, np.float32) for w in (0, 1, 2, 3, 5, 6)}
            self._step, self.loaded = 0, 0
        def _download(self, which): return self._arenas[which].copy()
        def _upload(self, which, arena): self._arenas[which] = np.asarray(arena, np.float32).copy()
        def get_global_step(self): return self._step
        def _set_global_step(self, step): self._step = step
        def _after_load(self): self.loaded += 1
        def predict_p_and_v(self, x): return [np.full((len(x), 2), 0.5, np.float32), np.arange(len(x), dtype=np.float32)]
        def losses(self, x, y_r, a): return dict(cost_p_1=1.0, cost_p_2=2.0, cost_p=-3.0, cost_v=4.0, cost_all=1.0)

    monkeypatch.chdir(tmp_path)
    rng = np.random.default_rng(3)
    net = Fake("m", dual=True)
    assert net.get_variables_names() == ["dense1/w:0", "dense1/b:0", "logits_v/w:0"]
    w = {k: rng.standard_normal(s).astype(np.float32) for k, (o, s) in net._table.items()}
    net.set_variables(w)
    assert all(np.array_equal(net.get_variables()[k], w[k]) for k in w)
    assert np.array_equal(net.get_variable_value("dense1/b:0"), w["dense1/b:0"])
    assert net._arenas[0][12:64].sum() == 0 and net._arenas[0][68:128].sum() == 0          # alignment gaps stay untouched
    with pytest.raises(ValueError):
        net.set_variables({"dense1/b:0": np.zeros(5, np.float32)})
    net.set_variables({"dense1/b:0": np.ones(4)})                                           # a subset; float64 is converted
    assert np.array_equal(net.get_variables()["dense1/b:0"], np.ones(4, np.float32)) and np.array_equal(net.get_variables()["dense1/w:0"], w["dense1/w:0"])
    ms = {k: np.full(s, 2.0, np.float32) for k, (o, s) in net._table.items()}
    mom = {k: np.full(s, 3.0, np.float32) for k, (o, s) in net._table.items()}
    net.set_slots(ms, mom)
    net.set_slots({k: v * 10 for k, v in ms.items()}, None, optimizer=1)
    assert net.get_slots()[0]["dense1/w:0"][0, 0] == 2.0 and net.get_slots()[1]["dense1/w:0"][0, 0] == 3.0
    assert net.get_slots(1)[0]["dense1/w:0"][0, 0] == 20.0 and net.get_slots(1)[1]["dense1/w:0"][0, 0] == 0.0
    assert net.predict_v(np.zeros((3, 2)))[2] == 2.0 and net.predict_p(np.zeros((3, 2))).shape == (3, 2)
    assert net.predict_single(np.zeros(2)).shape == (2,)

    net._step = 77
    assert net.save(5) == "checkpoints/m_00000005.npz" and net._get_episode_from_filename("checkpoints/m_00000005") == 5
    net._step = 99
    net.set_variables({"dense1/b:0": np.full(4, 9.0)})
    net.save(12)
    z = np.load("checkpoints/m_00000012.npz")
    assert {"dense1/w:0", "dense1/w/RMSProp:0", "dense1/w/RMSProp_1:0", "dense1/w/RMSProp_2:0", "dense1/w/RMSProp_3:0", "step:0"} <= set(z.files)
    other = Fake("m", dual=True)
    assert other.load() == 12 and other._step == 99 and other.loaded == 1                  # the latest checkpoint
    assert other.get_variables()["dense1/b:0"][0] == 9.0 and other.get_slots(1)[0]["dense1/w:0"][0, 0] == 20.0
    Cfg.LOAD_EPISODE = 5
    try:
        single = Fake("m", dual=False)
        assert single.load() == 5 and single._step == 77 and single.get_variables()["dense1/b:0"][0] == 1.0
        assert single.get_slots(1)[0]["dense1/w:0"][0, 0] == 0.0                            # not DUAL_RMSPROP: second optimizer untouched
    finally:
        Cfg.LOAD_EPISODE = 0
    plain = Fake("p")
    plain.save(1)
    assert "dense1/w/RMSProp_2:0" not in np.load("checkpoints/p_00000001.npz").files

    net.log(None, None, None, 1234)
    net.log(None, None, None, 1235)
    rows = open("logs/m/scalars.csv").read().strip().splitlines()
    assert rows[0] == "1234,1.0,2.0,-3.0,4.0,0.0003,0.01" and rows[1].startswith("1235,") and len(rows) == 2


def test_copy_threads_for_pageable_staging(monkeypatch):
    """Network._copy_threads: GA3C_COPY_THREADS wins (0 = the interpreter-side copy); otherwise half of this rank's share of the
    cores the process may run on, between 2 and 8 (LOCAL_WORLD_SIZE ranks of a torchrun job share the host)."""
    import ga3c_b200
    f = ga3c_b200.Network._copy_threads
    monkeypatch.setenv("GA3C_COPY_THREADS", "0")
    assert f() == 0
    monkeypatch.setenv("GA3C_COPY_THREADS", "5")
    assert f() == 5
    monkeypatch.delenv("GA3C_COPY_THREADS")
    monkeypatch.setattr(os, "sched_getaffinity", lambda pid: set(range(32)), raising=False)
    monkeypatch.delenv("LOCAL_WORLD_SIZE", raising=False)
    assert f() == 8
    monkeypatch.setenv("LOCAL_WORLD_SIZE", "8")
    assert f() == 2
    monkeypatch.setenv("LOCAL_WORLD_SIZE", "2")
    assert f() == 8
    monkeypatch.setattr(os, "sched_getaffinity", lambda pid: set(range(3)), raising=False)
    assert f() == 2
