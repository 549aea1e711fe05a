"""Parity of the CUDA TRAIN step (through the C ABI) against the CPU oracle on identical injected tables, batches and
hyper-parameters.  Tolerance (north_star): per-step loss and updated embeddings within 1e-5 relative, fp32 -- judged
against the fp64 shadow of the oracle (see _assert_close)."""
import numpy as np
import pytest

from conftest import make_coo
from oracle import glove_oracle as o

pytestmark = pytest.mark.gpu

RTOL = 1e-5
SHADOW_C = 3.0          # the CUDA path may be at most this many times further from the fp64 shadow than the fp32 oracle is
MAXIMA = {}             # test id -> observed maxima (written to gpurun_out/parity_maxima.json at session end)


def _rel(a, b):
    """max |a-b| / max |b|: error relative to the scale of the tensor (an element-wise relative error is meaningless
    next to zero-crossing embeddings)."""
    return float(np.max(np.abs(np.asarray(a, np.float64) - b)) / max(float(np.max(np.abs(b))), 1e-30))


def _record(name, **kw):
    MAXIMA.setdefault(name, {}).update({k: float(v) for k, v in kw.items()})


@pytest.fixture(scope="module", autouse=True)
def _dump_maxima():
    yield
    import json, os
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "parity_maxima.json"), "w") as f:
        json.dump(MAXIMA, f, indent=1, sort_keys=True)


def _c_mode(adam_mode):
    return "lazy" if adam_mode == "lazy" else "keras_dense"


def _shadow(st, coo, batches, *, optimizer, head, lr, reg_scale, adam_mode, neg_factor=0.7, l2_reg=0.01, both=True):
    """fp32 C oracle and its fp64 shadow (same source, -DORACLE_F64) on the same injected problem."""
    from oracle import c_oracle
    out = []
    for dt in ((np.float32, np.float64) if both else (np.float64,)):
        c = c_oracle.COracle(st.R, st.C, st.rb, st.cb, g=float(st.g), optimizer=optimizer, dtype=dt)
        l = c.train(coo, batches, head=head, learning_rate=lr, l2_reg=l2_reg, reg_scale=reg_scale, neg_factor=neg_factor,
                    adam_mode=_c_mode(adam_mode))
        out.append((c, l))
    return out


def _run_pair(V, d, B, steps, *, optimizer="Adam", head="glove", adam_mode="replay", K=4, seed=0, hot=None, lr=0.01,
              reg_scale=2.0, n=None, zipf=True, numpy_oracle=True):
    from glove_tensorflow_b200.engine import GloveEngine
    n = n or max(4 * B, 1000)
    coo = make_coo(V, n, seed, zipf=zipf, hot=hot)
    rng = np.random.default_rng(seed + 1)
    batches = rng.integers(0, n, (steps, B))
    st = o.init_state(V, d, seed + 2)
    (c32, l32), (c64, l64) = _shadow(st, coo, batches, optimizer=optimizer, head=head, lr=lr, reg_scale=reg_scale,
                                     adam_mode=adam_mode)
    if numpy_oracle:        # the cited NumPy restatement (slow: small cases only); the C port is checked against it on the CPU
        ref = st.copy()
        ref_losses = np.array(o.train(ref, coo, batches, optimizer=optimizer, head=head, learning_rate=lr,
                                      reg_scale=reg_scale, adam_mode=_c_mode(adam_mode), neg_factor=0.7))
    else:
        ref, ref_losses = c32, l32
    eng = GloveEngine(V, d, optimizer=optimizer, head=head, adam_mode=adam_mode, learning_rate=lr, reg_scale=reg_scale,
                      neg_factor=0.7, batch_size=B, plan_steps=K, max_steps=steps + 8)
    eng.load_state(st.R, st.C, st.rb, st.cb, st.g)
    a, b = ("target", "weight") if head == "glove" else ("pos", "neg")
    eng.set_coo(coo["row"], coo["col"], coo[a], coo[b])
    eng.set_batches(batches)
    losses = eng.train(steps)
    got = eng.get_state()
    got["_o32"], got["_o64"], got["_l64"] = c32, c64, l64
    return ref, np.array(ref_losses), got, losses, eng


def _assert_close(ref, ref_losses, got, losses, name=None):
    """north_star: per-step loss and updated tables within 1e-5 relative (fp32).  The tables are compared with the fp64
    SHADOW of the oracle: the CUDA path must be within 1e-5 of it, or -- where fp32 rounding of the recurrence itself
    exceeds that (Adam's m / (sqrt(v) + eps) amplifies the rounding of near-cancelling gradient sums) -- no more than
    SHADOW_C times further from it than the fp32 oracle is.  Observed maxima go to gpurun_out/parity_maxima.json."""
    import os
    name = name or os.environ.get("PYTEST_CURRENT_TEST", "?").split("::")[-1].split(" ")[0]
    assert np.all(np.isfinite(losses))
    e_loss = float(np.max(np.abs(losses - ref_losses) / np.abs(ref_losses)))
    e_loss64 = float(np.max(np.abs(losses - got["_l64"]) / np.abs(got["_l64"])))
    _record(name, loss_vs_oracle32=e_loss, loss_vs_shadow64=e_loss64)
    assert e_loss < RTOL, (losses[:4], ref_losses[:4])
    c32, c64 = got["_o32"], got["_o64"]
    for k in ("R", "C", "rb", "cb"):
        e_gpu, e_o32 = _rel(got[k], getattr(c64, k)), _rel(getattr(c32, k), getattr(c64, k))
        _record(name, **{k + "_gpu_vs_shadow64": e_gpu, k + "_oracle32_vs_shadow64": e_o32,
                         k + "_gpu_vs_oracle32": _rel(got[k], getattr(ref, k))})
        assert e_gpu <= max(RTOL, SHADOW_C * e_o32), (k, e_gpu, e_o32)
    assert abs(float(got["g"]) - float(c64.g)) <= RTOL * max(abs(float(c64.g)), 1e-3)
    assert got["step"] == ref.step


@pytest.mark.parametrize("optimizer", ["Adam", "Adagrad", "SGD"])
@pytest.mark.parametrize("head", ["glove", "logistic"])
def test_small_parity(optimizer, head):
    ref, rl, got, l, _ = _run_pair(50, 8, 16, 30, optimizer=optimizer, head=head)
    _assert_close(ref, rl, got, l)


@pytest.mark.parametrize("d", [1, 5, 30, 64, 100, 126, 200, 300, 320])
def test_embedding_sizes(d):
    ref, rl, got, l, _ = _run_pair(200, d, 64, 12, K=5)
    _assert_close(ref, rl, got, l)


def test_text8_shape_100_steps():
    """cfg2-like: V ~ 10k, d = 64, Adam lr 1e-3, batch 1024, 100 injected steps."""
    ref, rl, got, l, _ = _run_pair(10001, 64, 1024, 100, lr=0.001, K=16, n=200000)
    _assert_close(ref, rl, got, l)


def test_d300_zipf():
    ref, rl, got, l, _ = _run_pair(5000, 300, 2048, 20, lr=0.001, K=8, n=100000)
    _assert_close(ref, rl, got, l)


def test_heavy_hitters_long_segments():
    """40 % of a 4096 batch on one row id and one col id: segments far longer than one work item."""
    ref, rl, got, l, eng = _run_pair(300, 64, 4096, 10, hot=0.4, K=3, lr=0.01)
    _assert_close(ref, rl, got, l)
    counts = eng.batch_counts(eng.host_step - 1)
    assert counts[2] > counts[0] and counts[3] > counts[1]  # more items than segments => split segments exist


def test_split_segment_protocol_stress():
    """compute-sanitizer is closed on the GPU pool (racecheck / memcheck cannot be run), so the hand-rolled synchronisation
    of the update kernel -- partial sums of split segments published with __threadfence + chunk / segment tickets, work
    items handed out by atomic counters in a timing-dependent order, fixed-point loss atomics, the last-CTA ticket -- is
    hammered instead: 60 steps at B = 16,384 with 60 % of every batch on one row id and one col id (~300 pieces, 20 chunks
    and a three-level combine per side and step, d = 300 so a row spans all three float4 chunks of a lane), three
    independent runs.  A lost update, a stale partial or a double count shows up as a difference between runs or against the
    oracle; every run must be bit-identical to the others and within tolerance of the C oracle."""
    from glove_tensorflow_b200.engine import GloveEngine
    from oracle import c_oracle
    V, d, B, steps = 2000, 300, 16384, 60
    coo = make_coo(V, 200_000, 91, hot=0.6)
    batches = np.random.default_rng(92).integers(0, 200_000, (steps, B))
    st = o.init_state(V, d, 93)
    runs = []
    for _ in range(3):
        eng = GloveEngine(V, d, learning_rate=0.01, batch_size=B, plan_steps=6, max_steps=steps + 8)
        eng.load_state(st.R, st.C, st.rb, st.cb, st.g)
        eng.set_coo(coo["row"], coo["col"], coo["target"], coo["weight"])
        eng.set_batches(batches)
        losses = eng.train(steps)
        runs.append((losses, eng.get_state(slots=True)))
        c = eng.batch_counts(steps - 1)
        assert c[2] - c[0] > 250 and c[3] - c[1] > 250        # hundreds of pieces per side
    for losses, state in runs[1:]:
        assert np.array_equal(losses, runs[0][0])
        for k in state:
            assert np.array_equal(np.asarray(state[k]), np.asarray(runs[0][1][k])), k
    c32 = c_oracle.COracle(st.R, st.C, st.rb, st.cb)
    l32 = c32.train(coo, batches, learning_rate=0.01)
    assert np.max(np.abs(runs[0][0] - l32) / np.abs(l32)) < RTOL
    for k in ("R", "C", "rb", "cb"):
        assert _rel(runs[0][1][k], getattr(c32, k)) < 3e-5, k


def test_lazy_mode_matches_lazy_oracle():
    ref, rl, got, l, _ = _run_pair(2000, 32, 256, 40, adam_mode="lazy", zipf=False)
    _assert_close(ref, rl, got, l)


def test_dense_mode_matches_oracle_and_exact_replay_bit_exact():
    """The step-by-step replay schedule and the literal dense sweep must give bit-identical tables on the GPU; the
    closed-form replay (the default) must match the oracle like they do."""
    ref, rl, got_r, l_r, _ = _run_pair(3000, 24, 128, 60, adam_mode="replay_exact", zipf=False, K=7)
    _, _, got_d, l_d, _ = _run_pair(3000, 24, 128, 60, adam_mode="dense", zipf=False, K=7)
    _, _, got_c, l_c, _ = _run_pair(3000, 24, 128, 60, adam_mode="replay", zipf=False, K=7)
    _assert_close(ref, rl, got_d, l_d, "dense_vs_exact/dense")
    _assert_close(ref, rl, got_r, l_r, "dense_vs_exact/replay_exact")
    _assert_close(ref, rl, got_c, l_c, "dense_vs_exact/replay_closed_form")
    for k in ("R", "C", "rb", "cb"):
        assert np.array_equal(got_r[k], got_d[k]), k
    assert np.array_equal(l_r, l_d)


def test_closed_form_replay_long_idle_gaps():
    """Rows idle for hundreds of steps between two touches (uniform ids over a vocabulary much larger than the batch):
    the closed-form replay must track the dense-sweep oracle through the whole drift of every row."""
    ref, rl, got, l, _ = _run_pair(20000, 16, 64, 400, zipf=False, K=16, lr=0.001, numpy_oracle=False, seed=11)
    _assert_close(ref, rl, got, l)


def test_error_is_at_the_oracles_own_rounding_noise():
    """The CUDA path must be no further from the fp64 shadow than the fp32 oracle is (x SHADOW_C), on a problem where
    Adam amplifies fp32 rounding visibly (lr 0.01, heavy duplicates)."""
    V, d, B, steps, lr = 400, 32, 256, 40, 0.01
    ref, rl, got, l, _ = _run_pair(V, d, B, steps, lr=lr, seed=5)
    rms = lambda a: float(np.sqrt(np.mean((np.asarray(a, np.float64) - got["_o64"].R) ** 2)))
    rms_gpu, rms_o32 = rms(got["R"]), rms(got["_o32"].R)          # RMS: the maximum of 12,800 heavy-tailed errors is noisy
    _record("rounding_noise_rms", gpu=rms_gpu, oracle32=rms_o32)
    assert rms_gpu <= 2.0 * rms_o32 + 1e-9, (rms_gpu, rms_o32)
    _assert_close(ref, rl, got, l)


def test_reg_scale_one():
    ref, rl, got, l, _ = _run_pair(100, 16, 32, 20, reg_scale=1.0)
    _assert_close(ref, rl, got, l)


def test_deterministic_rerun_bitwise():
    _, _, g1, l1, _ = _run_pair(1000, 64, 512, 25, hot=0.2)
    _, _, g2, l2, _ = _run_pair(1000, 64, 512, 25, hot=0.2)
    assert np.array_equal(l1, l2)
    for k in ("R", "C", "rb", "cb"):
        assert np.array_equal(g1[k], g2[k])


@pytest.mark.parametrize("optimizer", ["Adam", "Adagrad"])
def test_cuda_graph_replay_is_bit_identical(optimizer):
    """K steps captured once as a CUDA graph (glove_step_graph_*) and replayed for every later chunk of the same plan buffer
    give bit for bit the tables and losses of single glove_train_step launches: the step index and the batch are read
    from device memory, so nothing step-specific is baked into the graph.  27 steps, K = 4: six graph launches (three per
    plan buffer) and three single steps at the tail."""
    from glove_tensorflow_b200.engine import GloveEngine
    V, d, B, steps, K = 800, 48, 256, 27, 4
    coo = make_coo(V, 4000, 11, hot=0.1)
    batches = np.random.default_rng(12).integers(0, 4000, (steps, B))
    st = o.init_state(V, d, 13)
    out = []
    for use_graph in (False, True):
        eng = GloveEngine(V, d, optimizer=optimizer, learning_rate=0.01, batch_size=B, plan_steps=K, max_steps=steps + 8)
        eng.load_state(st.R, st.C, st.rb, st.cb, st.g)
        eng.set_coo(coo["row"], coo["col"], coo["target"], coo["weight"])
        eng.set_batches(batches)
        eng.use_graph = use_graph
        losses = eng.train(steps)
        assert (eng._graphs[0] is not None) == use_graph and (eng._graphs[1] is not None) == use_graph
        out.append((losses, eng.get_state(slots=True)))
    assert np.array_equal(out[0][0], out[1][0])
    for k in out[0][1]:
        assert np.array_equal(np.asarray(out[0][1][k]), np.asarray(out[1][1][k])), k


def test_batch_size_one_and_single_id():
    ref, rl, got, l, _ = _run_pair(3, 4, 1, 10, zipf=False)
    _assert_close(ref, rl, got, l)


def test_plan_counts_match_numpy():
    from glove_tensorflow_b200.engine import GloveEngine
    V, B = 500, 777
    coo = make_coo(V, 5000, 3)
    batches = np.random.default_rng(4).integers(0, 5000, (5, B))
    eng = GloveEngine(V, 16, batch_size=B, plan_steps=3, max_steps=16)
    eng.set_coo(coo["row"], coo["col"], coo["target"], coo["weight"])
    eng.set_batches(batches)
    for s in range(5):
        c = eng.batch_counts(s)
        assert c[0] == len(np.unique(coo["row"][batches[s]]))
        assert c[1] == len(np.unique(coo["col"][batches[s]]))


def test_unsupported_inputs_fail_loudly():
    from glove_tensorflow_b200.engine import GloveEngine
    with pytest.raises(ValueError):
        GloveEngine(10, 4, optimizer="RMSprop")
    with pytest.raises(ValueError):
        GloveEngine(10, 600)


@pytest.mark.parametrize("world,adam_mode,optimizer", [(2, "replay", "Adam"), (4, "lazy", "Adam"), (2, "replay", "Adagrad")])
def test_data_parallel_replicas_on_one_gpu(world, adam_mode, optimizer):
    """Emulates `world` data-parallel ranks as `world` replica engines on one GPU (the real thing differs only in the
    NCCL all-reduce, replaced here by summing the ranks' buffers in rank order): the replicas must stay bit-identical
    and match the single-process oracle step on the global batch."""
    import torch
    from glove_tensorflow_b200.engine import GloveEngine
    V, d, B, steps, n = 600, 48, 512, 12, 20000
    coo = make_coo(V, n, 31, hot=0.15)
    batches = np.random.default_rng(32).integers(0, n, (steps, B))
    st = o.init_state(V, d, 33)
    ref = st.copy()
    ref_losses = np.array(o.train(ref, coo, batches, optimizer=optimizer, learning_rate=0.01,
                                  adam_mode="lazy" if adam_mode == "lazy" else "keras_dense"))
    engs = []
    for r in range(world):
        e = GloveEngine(V, d, optimizer=optimizer, adam_mode=adam_mode, learning_rate=0.01, batch_size=B, plan_steps=5,
                        max_steps=steps + 8, dp_rank=r, dp_world=world)
        e.load_state(st.R, st.C, st.rb, st.cb, st.g)
        e.set_coo(coo["row"], coo["col"], coo["target"], coo["weight"])
        e.set_batches(batches)
        engs.append(e)
    losses = []
    for s in range(steps):
        bufs = [e.grad_step() for e in engs]
        total = [torch.stack([b[i] for b in bufs]).sum(0) for i in range(3)]
        for e, b in zip(engs, bufs):
            for i in range(3):
                b[i].copy_(total[i])
            e.apply_step()
        torch.cuda.synchronize()
        losses.append(float(engs[0].read_scalars()["loss"]))
    states = [e.get_state() for e in engs]
    for k in ("R", "C", "rb", "cb"):
        for stt in states[1:]:
            assert np.array_equal(states[0][k], stt[k]), k
        assert _rel(states[0][k], getattr(ref, k)) < 3e-5, (k, _rel(states[0][k], getattr(ref, k)))
    assert np.max(np.abs(np.array(losses) - ref_losses) / np.abs(ref_losses)) < RTOL


@pytest.mark.parametrize("adam_mode", ["replay", "replay_exact"])
def test_overlap_streams_do_not_change_results(adam_mode):
    """Plan prefetch (and, for the step-by-step replay, the catch-up on the side stream) vs everything on one stream:
    bit-identical tables and losses."""
    from glove_tensorflow_b200.engine import GloveEngine
    V, d, B, steps, n = 5000, 64, 1024, 70, 60000
    coo = make_coo(V, n, 41)
    st = o.init_state(V, d, 42)
    out = []
    for overlap in (True, False):
        eng = GloveEngine(V, d, learning_rate=0.01, batch_size=B, plan_steps=6, max_steps=steps + 8, adam_mode=adam_mode)
        eng.overlap = overlap
        eng.load_state(st.R, st.C, st.rb, st.cb, st.g)
        eng.set_coo(coo["row"], coo["col"], coo["target"], coo["weight"], shuffle_key=3)
        l = np.concatenate([eng.train(25), eng.train(45)])          # a flush-free pause in the middle
        s = eng.get_state(slots=True)
        out.append((l, s))
    assert np.array_equal(out[0][0], out[1][0])
    for k in ("R", "C", "rb", "cb", "R/s0", "R/s1", "C/s0", "cb/s1"):
        assert np.array_equal(out[0][1][k], out[1][1][k]), k


@pytest.mark.parametrize("exchange", ["alltoall", "allgather", "peer", "peer-direct", "peer-sync", "peer-push",
                                      "alltoall+shared-plans", "peer-sync+shared-plans", "peer-push+shared-plans"])
@pytest.mark.parametrize("world,adam_mode,optimizer,V", [(2, "replay", "Adam", 601), (4, "replay", "Adam", 1000),
                                                         (3, "lazy", "Adam", 333), (2, "replay", "Adagrad", 64),
                                                         (8, "replay", "Adam", 5000)])
def test_row_sharded_tables_on_one_gpu(world, adam_mode, optimizer, V, exchange):
    """cfg4 scheme (SURVEY 8e): tables split row-wise over `world` owners (id % world), emulated as `world` engines on one
    GPU with the two collectives (all-gather of the owners' snapshot blocks, all-reduce of the loss scalars) done by
    hand; every owner runs the fused update of its own segments.  The union of the shards must match the single-process oracle."""
    _run_row_sharded(world, adam_mode, optimizer, V, exchange)


def _run_row_sharded(world, adam_mode, optimizer, V, exchange, d=40):
    B, steps, n = 512 if world != 3 else 510, 14, 20000
    coo = make_coo(V, n, 51, hot=0.1)
    batches = np.random.default_rng(52).integers(0, n, (steps, B))
    st = o.init_state(V, d, 53)
    ref = st.copy()
    ref_losses = np.array(o.train(ref, coo, batches, optimizer=optimizer, learning_rate=0.01,
                                  adam_mode="lazy" if adam_mode == "lazy" else "keras_dense"))
    got, losses = _row_sharded_train(world, adam_mode, optimizer, V, exchange, d, st, coo, batches)
    for k in ("R", "C", "rb", "cb"):
        assert _rel(got[k], getattr(ref, k)) < 3e-5, (k, _rel(got[k], getattr(ref, k)))
    assert np.max(np.abs(np.array(losses) - ref_losses) / np.abs(ref_losses)) < RTOL


def _row_sharded_train(world, adam_mode, optimizer, V, exchange, d, st, coo, batches, K=5, lr=0.01):
    """Trains `st` on (coo, batches) with the tables split over `world` owner engines on one GPU; returns the union of the
    shards' tables (reference layout) and the per-step losses."""
    import torch
    from glove_tensorflow_b200.engine import GloveEngine
    # "+shared-plans": the plan of chunk c is built by engine c % world alone and every engine copies its slice out of the
    # builder's buffer (glove_plan_pull_slice) -- results must not change by a bit (compared with the oracle like the rest)
    shared = exchange.endswith("+shared-plans")
    exchange = exchange.split("+")[0]
    steps, B = batches.shape
    engs = []
    for r in range(world):
        e = GloveEngine(V, d, optimizer=optimizer, adam_mode=adam_mode, learning_rate=lr, batch_size=B, plan_steps=K,
                        max_steps=steps + 8, dp_rank=r, dp_world=world, dp_mode="sharded")
        if world in (3, 8):                                        # frequency-balanced owner map instead of id % world
            e.balance_owners(coo["row"], coo["col"], hot=64)       # (the balance itself is checked in tests/test_dp_gloo.py)
        e.load_state(st.R, st.C, st.rb, st.cb, st.g)
        if shared:                                                 # one GPU: the "barrier" is a device synchronisation
            e.enable_plan_sharing(_emulate=(None, torch.cuda.synchronize))
        e.set_coo(coo["row"], coo["col"], coo["target"], coo["weight"])
        e.set_batches(batches)
        engs.append(e)
    if shared:
        for e in engs:
            e._ring["ptrs"] = [x._ring["buf"].data_ptr() for x in engs]
            e.plans[0].fill_(0xAB); e.plans[1].fill_(0xAB)         # whatever is not pulled stays garbage
    if exchange.startswith("peer"):                                # on one GPU every "peer" workspace is plain device memory
        for e in engs:
            e.set_peer_workspaces([x.step_ws.data_ptr() for x in engs], direct=exchange == "peer-direct",
                                  sync=exchange in ("peer-sync", "peer-push"), push=exchange == "peer-push")
    side_streams = [torch.cuda.Stream() for _ in engs]
    losses = []
    for s in range(steps):
        if shared:
            # real ranks meet at a barrier before a round of chunks is pulled; engines called one after the other cannot, so
            # the builds of the rounds that this step (and its plan prefetch) may pull from are issued up front
            for c in (s // K, s // K + 1):
                for e in engs:
                    e._ring_build(c // world)
            torch.cuda.synchronize()
        upads = [e.shard_stage() for e in engs]
        assert all(u == upads[0] for u in upads)
        torch.cuda.synchronize()
        if exchange == "peer-direct":
            pass                                                   # the update kernels read each other's snapshots directly
        elif exchange in ("peer-sync", "peer-push"):
            for e in engs:
                e.shard_signal_staged()                            # every shard announces its block ...
            for e in engs:                                         # ... before any shard waits for the owners' announcements
                if e.shard_exchange == "peer-push":
                    e.shard_wait_staged()                          # (the stage kernels have pushed the rows already)
                else:
                    e.shard_pull()
        elif exchange == "peer":
            for e in engs:
                e.shard_pull()                                     # one kernel: requested rows, owner's snapshot -> mine
        elif exchange == "allgather":
            for side in (0, 1):
                u = upads[0][side]
                for dst in engs:                                   # all-gather of the owners' snapshot blocks
                    for q, src in enumerate(engs):
                        if src is not dst:
                            dst.snapshot_view(side)[q * u:(q + 1) * u].copy_(src.snapshot_view(side)[q * u:(q + 1) * u])
        else:                                                      # all-to-all of the requested rows only
            counts = [e.shard_pack() for e in engs]                # (send to each peer, receive from each owner)
            torch.cuda.synchronize()
            for r, dst in enumerate(engs):
                roff = 0
                for q, src in enumerate(engs):
                    n = counts[r][1][q]
                    assert n == counts[q][0][r]
                    soff = sum(counts[q][0][:r])
                    dst._xbuf[1][roff:roff + n].copy_(src._xbuf[0][soff:soff + n])
                    roff += n
            for e in engs:
                e.shard_unpack()
        for e in engs:
            e.shard_update()                                   # owner-computes: no gradient exchange
        torch.cuda.synchronize()
        if exchange in ("peer-sync", "peer-push"):
            # device-side all-reduce: every shard's finish kernel announces its sums, then waits for all the others --
            # the kernels must be able to run side by side, so each goes on its own stream (they are one warp each)
            for e, st_ in zip(engs, side_streams):
                with torch.cuda.stream(st_):
                    e.shard_finish_sync()
        else:
            tot = torch.stack([e._sscal for e in engs]).sum(0)     # all-reduce of the loss scalars
            for e in engs:
                e._sscal.copy_(tot)
                e.shard_finish()
        torch.cuda.synchronize()
        losses.append(float(engs[0].read_scalars()["loss"]))
    got = {k: np.zeros_like(np.asarray(getattr(st, k), np.float32)) for k in ("R", "C", "rb", "cb")}
    for r, e in enumerate(engs):
        stt = e.get_state()
        ids = e.owned_ids()
        assert len(ids) == len(got["rb"][r::world]) and (world in (3, 8) or np.array_equal(ids, np.arange(r, V, world)))
        for k in got:
            got[k][ids] = stt[k][: len(ids)]
    got["g"], got["step"] = np.float32(engs[0].read_scalars()["g"]), engs[0].read_scalars()["step"]
    return got, np.array(losses)
