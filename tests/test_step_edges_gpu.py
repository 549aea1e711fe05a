"""TRAIN step edge tests: batches built so that segments have prescribed lengths at every boundary of the split-segment
protocol of update_kernel, run through every step path and compared with the fp64 shadow of the C oracle.

A work item holds at most kItemMax = 32 triples of one segment; a longer segment is split into ceil(L / 32) pieces whose
partial sums are combined per chunk of kChunk = 16 pieces and then chunk by chunk.  The lengths below sit on each side of
those boundaries: one piece (31, 32), two (33), one whole chunk with the second level skipped (512), a last chunk of one
piece (513), and 256 / 257 pieces (8192, 8193).  Random (Zipf, heavy-hitter) batches only land on them by chance."""
import functools

import numpy as np
import pytest

from conftest import make_coo
from oracle import glove_oracle as o
from test_train_gpu import RTOL, _assert_close, _dump_maxima, _record, _rel, _row_sharded_train, _shadow  # noqa: F401

pytestmark = pytest.mark.gpu

ITEM_MAX = 32             # kItemMax: triples per work item
LENGTHS = (1, 2, 31, 32, 33, 63, 64, 65, 511, 512, 513, 543, 544, 545, 1023, 1024, 1025, 8191, 8192, 8193)
B_STD = 32768             # sum(LENGTHS) = 31,107 long-segment triples + 1,661 fillers per side


def _batches_with_lengths(V, B, steps, row_lengths, col_lengths, seed, keep_out=()):
    """COO (the columns make_coo gives) and explicit batches[steps, B] in which row id i occurs exactly row_lengths[s][i]
    times in batch s and col id j exactly col_lengths[s][j] times (one dict stands for every step).  Every other slot of
    a side holds a filler id that occurs once in the batch.  Fillers never take an id that is long on that side in any
    step, nor one of `keep_out`: an id that is long in some steps is absent from the others.  Positions are shuffled, so
    the triples of a long segment arrive scattered over the batch (and over the data-parallel rank blocks)."""
    rng = np.random.default_rng(seed)
    sides = []
    for lens in (row_lengths, col_lengths):
        lens = list(lens) if isinstance(lens, (list, tuple)) else [lens] * steps
        reserved = np.array(sorted(set(keep_out).union(*lens)), np.int64)
        pool = np.setdiff1d(np.arange(V), reserved)
        ids = []
        for s in range(steps):
            long_ids = np.repeat(np.array(list(lens[s]), np.int64), np.array(list(lens[s].values()), np.int64))
            assert len(long_ids) <= B
            ids.append(rng.permutation(np.concatenate([long_ids, rng.choice(pool, B - len(long_ids), replace=False)])))
        sides.append(np.concatenate(ids).astype(np.int32))
    n = steps * B
    count = 10 + np.floor(rng.pareto(1.0, n)).clip(0, 1e6)
    value = count * rng.uniform(0.3, 0.6, n)
    coo = {"row": sides[0], "col": sides[1], "target": np.log(value).astype(np.float32),
           "weight": np.clip((count / 100.0) ** 0.75, 0, 1).astype(np.float32), "pos": value.astype(np.float32),
           "neg": (count * rng.uniform(0.0, 0.5, n)).astype(np.float32)}
    batches = np.stack([s * B + rng.permutation(B) for s in range(steps)])
    return coo, batches


def _cycling_lengths(V, steps, seed):
    """{id: length} per step for one side: 30 candidate ids drawn above V / 4 (so the long ids are not the lowest ids, and
    the work list is not longest-first); id k is long in step s unless (k + s) % 3 == 0, so ids go long -> long (the
    previous batch has them) and long -> absent -> long (Adam gaps read in the combine path); the 20 lengths are dealt
    afresh to each step's 20 long ids."""
    rng = np.random.default_rng(seed)
    cand = rng.choice(np.arange(V // 4, V), 30, replace=False)
    out = []
    for s in range(steps):
        live = [int(cand[k]) for k in range(30) if (k + s) % 3]
        out.append(dict(zip(live, rng.permutation(LENGTHS).tolist())))
    return out


@functools.lru_cache(maxsize=None)
def _problem(V, B, steps, seed=0):
    """The standard problem: every batch holds one segment of each of LENGTHS on each side, with different id <-> length
    assignments on the two sides and from step to step."""
    rl, cl = _cycling_lengths(V, steps, seed), _cycling_lengths(V, steps, seed + 1)
    coo, batches = _batches_with_lengths(V, B, steps, rl, cl, seed + 2)
    return coo, batches, rl, cl


def _expected_counts(B, row_len, col_len):
    """(segments row, segments col, work items row, work items col) of a batch: ceil(L / 32) items per segment."""
    fr, fc = B - sum(row_len.values()), B - sum(col_len.values())
    items = lambda lens: sum(-(-L // ITEM_MAX) for L in lens.values())
    return (len(row_len) + fr, len(col_len) + fc, items(row_len) + fr, items(col_len) + fc)


def _engine(V, d, B, K, steps, st, coo, batches, *, optimizer="Adam", head="glove", adam_mode="replay", lr=0.01, **kw):
    from glove_tensorflow_b200.engine import GloveEngine
    eng = GloveEngine(V, d, optimizer=optimizer, head=head, adam_mode=adam_mode, learning_rate=lr, reg_scale=2.0,
                      neg_factor=0.7, batch_size=B, plan_steps=K, max_steps=steps + 8, **kw)
    eng.load_state(st.R, st.C, st.rb, st.cb, st.g)
    a, b = ("target", "weight") if head == "glove" else ("pos", "neg")
    eng.set_coo(coo["row"], coo["col"], coo[a], coo[b])
    eng.set_batches(batches)
    return eng


def _with_shadow(got, st, coo, batches, *, optimizer="Adam", head="glove", adam_mode="replay", lr=0.01):
    """The fp32 C oracle and its fp64 shadow on the same problem, attached to `got` the way _assert_close expects."""
    (c32, l32), (c64, l64) = _shadow(st, coo, batches, optimizer=optimizer, head=head, lr=lr, reg_scale=2.0,
                                     adam_mode=adam_mode)
    got["_o32"], got["_o64"], got["_l64"] = c32, c64, l64
    return c32, l32


def _same_bits(a, b):
    la, sa = a
    lb, sb = b
    assert np.array_equal(la, lb)
    for k in sa:
        assert np.array_equal(np.asarray(sa[k]), np.asarray(sb[k])), k


# ---- 1 + 2: the plan at the boundaries --------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [B_STD, 65536])
def test_plan_counts_at_split_boundaries(B):
    """Segments and work items per batch are exactly (segments, sum ceil(L / 32)) of the prescribed lengths: pins
    itemflags / items / itemrec / longrec at every piece boundary before any arithmetic is compared."""
    V, steps = (4096, 6) if B == B_STD else (40000, 3)
    coo, batches, rl, cl = _problem(V, B, steps)
    for lens in (rl, cl):                              # the builder itself: exact multiplicities in every batch
        side = coo["row"] if lens is rl else coo["col"]
        for s in range(steps):
            ids, cnt = np.unique(side[batches[s]], return_counts=True)
            got = dict(zip(ids.tolist(), cnt.tolist()))
            assert all(got[i] == L for i, L in lens[s].items())
            assert sum(cnt > 1) == sum(L > 1 for L in lens[s].values()) and len(ids) == B - sum(lens[s].values()) + 20
    eng = _engine(V, 16, B, 4, steps, o.init_state(V, 16, 1), coo, batches)
    for s in range(steps):
        assert eng.batch_counts(s) == _expected_counts(B, rl[s], cl[s]), s


# ---- 3: single-GPU TRAIN parity ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", [64, 300])
@pytest.mark.parametrize("optimizer,head,adam_mode", [("Adam", "glove", "replay"), ("Adam", "glove", "replay_exact"),
                                                      ("Adam", "glove", "lazy"), ("Adagrad", "glove", "replay"),
                                                      ("SGD", "glove", "replay"), ("Adam", "logistic", "replay")])
def test_parity_at_split_boundaries(optimizer, head, adam_mode, d):
    V, B = 4096, B_STD
    steps, K = (6, 4) if d == 64 else (3, 2)           # d = 300: a few steps keep the oracle cheap
    coo, batches, _, _ = _problem(V, B, steps)
    st = o.init_state(V, d, 3)
    cfg = dict(optimizer=optimizer, head=head, adam_mode=adam_mode)
    eng = _engine(V, d, B, K, steps, st, coo, batches, **cfg)
    losses = eng.train(steps)
    got = eng.get_state()
    c32, l32 = _with_shadow(got, st, coo, batches, **cfg)
    _assert_close(c32, l32, got, losses)


def test_parity_at_split_boundaries_production_batch():
    """B = 65,536 (the production batch): 34,429 fillers per side next to the 20 prescribed segments."""
    V, B, d, steps = 40000, 65536, 64, 3
    coo, batches, _, _ = _problem(V, B, steps)
    st = o.init_state(V, d, 4)
    eng = _engine(V, d, B, 2, steps, st, coo, batches)
    losses = eng.train(steps)
    got = eng.get_state()
    c32, l32 = _with_shadow(got, st, coo, batches)
    _assert_close(c32, l32, got, losses)


def test_split_segments_bit_identical_reruns_and_graph():
    """Three independent runs give the same bits (tables, optimizer slots, losses), whichever warp wins the chunk and
    segment tickets; K steps captured as one CUDA graph give the bits of single launches."""
    V, d, B, steps, K = 4096, 64, B_STD, 8, 4
    coo, batches, _, _ = _problem(V, B, steps)
    st = o.init_state(V, d, 5)
    out = []
    for use_graph in (False, False, False, True):
        eng = _engine(V, d, B, K, steps, st, coo, batches)
        eng.use_graph = use_graph
        losses = eng.train(steps)
        assert (eng._graphs[0] is not None) == use_graph and (eng._graphs[1] is not None) == use_graph
        out.append((losses, eng.get_state(slots=True)))
    for r in out[1:]:
        _same_bits(out[0], r)


# ---- 4: the other step paths ---------------------------------------------------------------------------------------------
def _pin_to_rank(batch, mask, rank, world, seed):
    """`batch` reordered so that the entries selected by `mask` have their arrival index inside `rank`'s block."""
    rng = np.random.default_rng(seed)
    B = len(batch)
    blk = B // world
    out = np.full(B, -1, np.int64)
    pos = rng.choice(np.arange(rank * blk, (rank + 1) * blk), int(mask.sum()), replace=False)
    out[pos] = batch[mask]
    out[out < 0] = batch[~mask]
    return out


@pytest.mark.parametrize("world,adam_mode", [(2, "replay"), (3, "replay"), (2, "lazy")])
def test_data_parallel_replicas_at_split_boundaries(world, adam_mode):
    """Replicated data parallelism emulated on one GPU (as test_data_parallel_replicas_on_one_gpu): every replica masks the
    terms whose arrival index is outside its block.  In batch 1 every triple of the 513-long row segment and of the
    513-long col segment arrives inside rank 1's block, so the other ranks see both with n_eff = 0 in every piece (and a
    zero activity-L2 factor).  Replicas stay bit-identical and match the oracle on the global batch."""
    import torch
    V, d, steps, K = 4096, 64, 4, 3
    B = B_STD if world == 2 else 32769                 # grad / apply steps need B % world == 0 (B / world per rank)
    coo, batches, rl, cl = _problem(V, B, steps, seed=20)
    batches = batches.copy()
    rid = next(i for i, L in rl[1].items() if L == 513)
    cid = next(i for i, L in cl[1].items() if L == 513)
    mask = (coo["row"][batches[1]] == rid) | (coo["col"][batches[1]] == cid)
    batches[1] = _pin_to_rank(batches[1], mask, 1, world, 21)
    st = o.init_state(V, d, 22)
    engs = [_engine(V, d, B, K, steps, st, coo, batches, adam_mode=adam_mode, dp_rank=r, dp_world=world)
            for r in range(world)]
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
    for stt in states[1:]:
        for k in ("R", "C", "rb", "cb"):
            assert np.array_equal(states[0][k], stt[k]), k
    got = states[0]
    c32, l32 = _with_shadow(got, st, coo, batches, adam_mode=adam_mode)
    _assert_close(c32, l32, got, np.array(losses, np.float32))


def test_data_parallel_refuses_uneven_rank_blocks():
    """A batch that does not split into equal rank blocks is refused by the grad step rather than trained on with a
    remainder that no rank owns."""
    from glove_tensorflow_b200._lib import GloveError
    V, d, B = 4096, 16, B_STD
    coo, batches, _, _ = _problem(V, B, 6)
    eng = _engine(V, d, B, 4, 6, o.init_state(V, d, 1), coo, batches, dp_rank=0, dp_world=3)
    with pytest.raises(GloveError, match="bad dp split"):
        eng.grad_step()


def _owner_edge_lengths(V, world, steps, seed, shift=0):
    """{id: length} per step for one side of a row-sharded problem (owner = id % world, local row = id // world).  The
    first and the last local id of every owner (2 * world "edge" ids; in the plan's owner-major order the last id of
    owner r and the first of owner r + 1 are neighbours) carry, in rotation, 33, 513, 8193 and other lengths of LENGTHS, so
    that each of 33, 513 and 8193 lands on the first and on the last local id of an owner block; the rest of LENGTHS sits
    on fixed interior ids."""
    assert V % world == 0
    v_loc = V // world
    edges = [r + world * (v_loc - 1) * last for r in range(world) for last in (0, 1)]
    edge_len = (33, 513, 8193, 1, 32, 512, 8192, 65)[: len(edges)]
    rest = list(LENGTHS)
    for L in edge_len:
        rest.remove(L)
    rng = np.random.default_rng(seed)
    inner = rng.choice(np.arange(world, V - world), len(rest), replace=False)
    out = []
    for s in range(steps):
        lens = {int(e): edge_len[(j + s + shift) % len(edges)] for j, e in enumerate(edges)}
        lens.update(zip(inner.tolist(), rng.permutation(rest).tolist()))
        out.append(lens)
    return out, edges


@pytest.mark.parametrize("exchange", ["peer-push", "alltoall"])
@pytest.mark.parametrize("world", [2, 4])
def test_row_sharded_split_segments_at_owner_block_edges(world, exchange):
    """Row-sharded tables: b_own_item must cut the work list exactly at the first segment of every owner, also when a split
    segment is the first or the last segment of an owner's block."""
    V, d, B, steps, K = 4096, 64, B_STD, 4, 3
    rl, edges = _owner_edge_lengths(V, world, steps, 30)
    cl, _ = _owner_edge_lengths(V, world, steps, 31, shift=1)      # another id <-> length assignment on the col side
    coo, batches = _batches_with_lengths(V, B, steps, rl, cl, 32, keep_out=edges)
    st = o.init_state(V, d, 33)
    got, losses = _row_sharded_train(world, "replay", "Adam", V, exchange, d, st, coo, batches, K=K)
    c32, l32 = _with_shadow(got, st, coo, batches)
    _assert_close(c32, l32, got, losses)


# ---- 5: plan-chunk invariance --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("problem", ["split", "idle"])
@pytest.mark.parametrize("adam_mode", ["replay", "replay_exact"])
def test_plan_chunk_size_does_not_change_results(adam_mode, problem):
    """The same 24 steps planned K = 1, 5 or 24 at a time: only the plan buffers and the seg_prev hint (1, "unknown", for
    the first batch of every plan) differ, so tables, slots and losses must be the same bits.  'split': the prescribed
    segment lengths; 'idle': uniform ids, rows idle for many steps between touches (closed-form / step-by-step replay)."""
    steps, d = 24, 64
    if problem == "split":
        V, B = 4096, B_STD
        coo, batches, _, _ = _problem(V, B, steps)
        lr = 0.01
    else:
        V, B, n = 1000, 64, 4000
        coo = make_coo(V, n, 11, zipf=False)
        batches = np.random.default_rng(12).integers(0, n, (steps, B))
        lr = 0.001
    st = o.init_state(V, d, 40)
    out = []
    for K in (1, 5, 24):
        eng = _engine(V, d, B, K, steps, st, coo, batches, adam_mode=adam_mode, lr=lr)
        losses = eng.train(steps)
        out.append((losses, eng.get_state(slots=True)))
    for r in out[1:]:
        _same_bits(out[0], r)


# ---- 6: the fixed-point loss accumulator and the error flag ---------------------------------------------------------------
def test_loss_accumulator_large_terms():
    """Targets of about +-3,000 with weight 1: a 32-triple item's loss is ~2.9e8 > 2^24 (no fraction limb, the integer limb
    carries); the sign follows the row id, so the per-item sum_e * B terms are large and of both signs.  The per-step loss
    and the global bias g stay within 1e-5 of the fp64 shadow, and reruns are bit-identical."""
    V, d, B, steps, K = 4096, 64, B_STD, 4, 3
    coo, batches, _, _ = _problem(V, B, steps)
    coo = dict(coo)
    rng = np.random.default_rng(50)
    sign = np.where(coo["row"] % 2 == 0, 1.0, -1.0)
    coo["target"] = (sign * rng.uniform(2900.0, 3100.0, len(sign))).astype(np.float32)
    coo["weight"] = np.ones(len(sign), np.float32)
    st = o.init_state(V, d, 51)
    runs = []
    for _ in range(2):
        eng = _engine(V, d, B, K, steps, st, coo, batches)
        losses = eng.train(steps)
        runs.append((losses, eng.get_state(slots=True)))
    _same_bits(runs[0], runs[1])
    losses, got = runs[0]
    c32, l32 = _with_shadow(got, st, coo, batches)
    e64 = float(np.max(np.abs(losses - got["_l64"]) / np.abs(got["_l64"])))
    _record("test_loss_accumulator_large_terms", loss_min=float(np.min(losses)), loss_vs_shadow64_direct=e64,
            g_vs_shadow64=abs(float(got["g"]) - float(got["_o64"].g)) / abs(float(got["_o64"].g)))
    assert np.min(losses) > 2.0 ** 24 / ITEM_MAX          # mean loss per triple: a full 32-triple item is above 2^24
    assert e64 < RTOL, e64
    _assert_close(c32, l32, got, losses)


def _error_run(coo, batches, V):
    from glove_tensorflow_b200._lib import GloveError
    eng = _engine(V, 16, batches.shape[1], 1, 1, o.init_state(V, 16, 60), coo, batches)
    with pytest.raises(GloveError, match="non-finite loss"):
        eng.train(1)


@pytest.mark.parametrize("what", ["nan_target", "inf_weight", "finite_above_4e18"])
def test_non_finite_loss_raises(what):
    """A per-item loss term that is NaN, infinite or >= 4e18 (where the int64 limbs of the fixed-point accumulator would
    overflow) sets the device error flag; eng.train surfaces it as GloveError('... non-finite loss ...') instead of
    returning a loss.  One step on its own engine each; the flag is an expected result, not a fault."""
    V, B = 2000, 1024
    coo, batches = _batches_with_lengths(V, B, 1, {123: ITEM_MAX}, {45: 40}, 61)
    coo = dict(coo)
    coo["target"], coo["weight"] = coo["target"].copy(), coo["weight"].copy()
    if what == "nan_target":
        coo["target"][batches[0][17]] = np.nan
    elif what == "inf_weight":
        coo["weight"][batches[0][17]] = np.inf
    else:                                          # 32 triples of one item: 32 * 0.1 * (1e10)^2 ~ 3e20, finite in fp32
        m = coo["row"] == 123
        coo["target"][m], coo["weight"][m] = 1e10, 0.1
    _error_run(coo, batches, V)
