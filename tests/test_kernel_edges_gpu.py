"""Kernels at the edges the other GPU tests do not reach, each against a plain fp64 NumPy reference (or the C oracle and
its fp64 shadow for TRAIN):
  A. the tensor-core top-k on a table built to defeat its bf16 error bound (see tests/test_topk_bound.py);
  B. the top-k over a sample of shapes: both K-chunk counts of the tensor-core pass and the scan-only sizes, k across the
     tensor-core cut at 24, V around the 1024 floor and the 256-row padding, query counts around the 256-row query tile,
     one, three and the default number of table slices, with tied rows on tile and slice boundaries;
  C. TRAIN at the embedding sizes where the float4-per-lane count NV changes (126/127, 254/255, 382/383) and at NV = 4
     (d up to 510, the largest size the engine accepts);
  D. EVAL at several sizes, both heads, batch sizes that are not multiples of the 32-triple tile, and sub-windows."""
import numpy as np
import pytest

from conftest import make_coo
from oracle import glove_oracle as o
from test_topk_bound import adversarial_table
from test_train_gpu import _assert_close, _dump_maxima, _run_pair, _run_row_sharded  # noqa: F401 (fixture)

pytestmark = pytest.mark.gpu

SIM_ATOL = 3e-6         # fp32 cosine (normalisation + <= 510-term dot) against fp64


def _engine(T, **kw):
    from glove_tensorflow_b200.engine import GloveEngine
    V, d = T.shape
    eng = GloveEngine(V, d, batch_size=64, plan_steps=1, max_steps=4, **kw)
    eng.load_state(T, T[::-1].copy(), np.zeros(V, np.float32), np.zeros(V, np.float32))
    return eng


def _ref_sims(T, q):
    """fp64 cosine of every query row against every table row (tf.math.l2_normalize's 1e-12 floor)."""
    t = T.astype(np.float64)
    t /= np.sqrt(np.maximum(np.sum(t * t, axis=1, keepdims=True), 1e-12))
    return t[q] @ t.T


def _check64(sim, idx, T, q, k):
    """Each returned similarity is the fp64 cosine of its id to within fp32 noise; position by position the list is the
    fp64 top-k (so ids may differ from the reference only between entries tied to within that noise); exact ties --
    identical rows -- are listed by increasing id."""
    full = _ref_sims(T, q)
    want_idx = np.argsort(-full, axis=1, kind="stable")[:, :k]
    want = np.take_along_axis(full, want_idx, 1)
    assert idx.shape == (len(q), k) and np.all((idx >= 0) & (idx < len(T)))
    assert all(len(set(r)) == k for r in idx.tolist())
    assert np.all(np.diff(sim, axis=1) <= 0)
    got = np.take_along_axis(full, idx.astype(np.int64), 1)
    np.testing.assert_allclose(sim, got, rtol=0, atol=SIM_ATOL)
    np.testing.assert_allclose(got, want, rtol=0, atol=2 * SIM_ATOL)
    same = np.diff(got, axis=1) == 0
    assert np.all(np.diff(idx, axis=1)[same] > 0), "exact ties must come in id order"


# ---- A. adversarial bf16 rounding ----------------------------------------------------------------------------------
@pytest.mark.parametrize("k,start,slices", [(1, 0, None), (5, 0, None), (1, 120, "3"), (5, 120, "3"), (1, 0, "1"),
                                            (5, 0, "1")])
def test_adversarial_bf16_rounding_goes_to_the_exact_scan(monkeypatch, k, start, slices):
    """The query (and its k - 1 copies) loses ~2^-7 of its self-similarity to bf16 rounding and is left out of its own
    candidate list; the candidates' k-th exact score is 4e-3..8e-3 above the cut-off.  The guarantee check must send
    exactly these queries to the exact scan.  start = 120: the block straddles the 128-row tile boundary inside one of
    three slices, so one candidate list is carried across accumulator tiles."""
    if slices is None:
        monkeypatch.delenv("GLOVE_TOPK_SLICES", raising=False)
    else:
        monkeypatch.setenv("GLOVE_TOPK_SLICES", slices)
    T, queries, near, fill = adversarial_table(k=k, start=start)
    eng = _engine(T)
    assert eng.tc_path_covers(k)
    controls = np.arange(400, 440)                              # ordinary rows: never flagged on this table
    q = np.concatenate([queries, controls]).astype(np.int32)
    sim, idx = eng.topk(q, k)
    fallbacks = eng.last_topk_fallbacks
    _check64(sim, idx, T, q, k)
    n = len(queries)
    assert np.array_equal(idx[:n], np.tile(queries, (n, 1)))    # the query and its copies, in id order
    assert np.array_equal(idx[n:, 0], controls)
    assert fallbacks == n, fallbacks
    s2, i2 = eng.topk(q, k, exact_fp32=True)
    assert np.array_equal(i2, idx) and np.array_equal(s2, sim)


def test_adversarial_bf16_rounding_row_sharded():
    """The same table spread over two row shards (owner = id % 2): the block sits on the even ids, so shard 0 alone meets
    the adversarial candidate list and must flag every query; the merged answer is the query itself."""
    import torch
    from glove_tensorflow_b200.engine import GloveEngine
    world, k = 2, 1
    T, queries, near, fill = adversarial_table(V=4096, k=k, stride=2)
    V, d = T.shape
    engs = []
    for r in range(world):
        e = GloveEngine(V, d, batch_size=64, plan_steps=1, max_steps=4, dp_rank=r, dp_world=world, dp_mode="sharded")
        e.load_state(T, T[::-1].copy(), np.zeros(V, np.float32), np.zeros(V, np.float32))
        engs.append(e)
    assert engs[0].tc_path_covers(k)
    q = np.concatenate([queries, np.arange(1001, 1041)]).astype(np.int32)
    qrows = sum(e.topk_shard_query_rows(q) for e in engs)     # == dist.all_reduce
    parts = [e.topk_shard_local(qrows, k) for e in engs]
    assert engs[0].last_topk_fallbacks == len(queries), engs[0].last_topk_fallbacks
    assert engs[1].last_topk_fallbacks == 0, engs[1].last_topk_fallbacks
    sim, idx = engs[0].topk_shard_merge(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]), k)
    _check64(sim, idx, T, q, k)
    assert np.array_equal(idx[:, 0], q)


# ---- B. top-k shape sweep -------------------------------------------------------------------------------------------
def _slice_edges(V, slices):
    """Table rows at which a new slice of the tensor-core pass starts (tc_ws_view; the default slice count gives one
    128-row tile per slice at these sizes, so every tile boundary is a slice boundary)."""
    tiles = (V + 255) // 256 * 2
    per = 1 if slices is None else -(-tiles // int(slices))
    return [t * 128 for t in range(per, tiles, per)]


# (d, k, V, n_queries, GLOVE_TOPK_SLICES): a pairwise-style sample.  d <= 320 runs the tensor-core pass (Kp = 64..320, one
# to five K chunks) when k <= 24 and V >= 1024; d >= 321, k >= 25 or V = 1023 run the exact scan alone (d >= 383: NV = 4)
SWEEP = [(64, 24, 1024, 257, "3"), (64, 1, 1023, 1, None), (100, 1, 5249, 600, None), (100, 25, 1024, 1, "3"),
         (128, 25, 1025, 256, "1"), (128, 24, 1023, 256, None), (192, 32, 5249, 1, "3"), (192, 24, 1024, 255, "1"),
         (256, 24, 1025, 255, None), (256, 24, 5249, 600, "1"), (300, 1, 1024, 600, "1"), (300, 24, 5249, 257, None),
         (320, 24, 5249, 256, "3"), (320, 1, 1025, 600, None), (321, 24, 1025, 257, None), (383, 1, 5249, 255, "1"),
         (448, 32, 1023, 600, "3"), (510, 25, 5249, 257, None), (510, 1, 1024, 256, "3")]


@pytest.mark.parametrize("d,k,V,nq,slices", SWEEP)
def test_topk_shape_sweep(monkeypatch, d, k, V, nq, slices):
    if slices is None:
        monkeypatch.delenv("GLOVE_TOPK_SLICES", raising=False)
    else:
        monkeypatch.setenv("GLOVE_TOPK_SLICES", slices)
    rng = np.random.default_rng(d * 7 + V)
    T = rng.uniform(-0.05, 0.05, (V, d)).astype(np.float32)
    edges = _slice_edges(V, slices)
    ties = sorted({e + o for e in [128, 256] + edges[:2] + edges[-1:] for o in (-1, 0)} | {V - 1})
    ties = [t for t in ties if 12 <= t < V]
    T[ties] = T[7]                                              # exact duplicates on both sides of tile / slice edges
    T[11] = 0.0                                                 # zero row: every similarity 0, ties everywhere
    head = [7, 11] + ties[:4]
    q = np.concatenate([head, rng.integers(0, V, max(nq - len(head), 0))])[:nq].astype(np.int32)
    eng = _engine(T)
    s_tc, i_tc = eng.topk(q, k)
    _check64(s_tc, i_tc, T, q, k)
    m = min(k, len(ties) + 1)
    assert list(i_tc[0, :m]) == ([7] + ties)[:m]                # row 7 and its copies lead its own list, in id order
    s_ex, i_ex = eng.topk(q, k, exact_fp32=True)
    _check64(s_ex, i_ex, T, q, k)
    if eng.tc_path_covers(k):
        assert np.array_equal(i_tc, i_ex) and np.array_equal(s_tc, s_ex)   # same fp32 re-score routine: bit-identical
        # with the default slicing (one 128-row tile per slice here) the cut-off is far below the k-th score; a forced
        # single slice at k = 24 leaves the 24th and the 32nd best of ~1000 random rows ~0.01 apart, within the 8e-3 bound,
        # so there most queries rightly go to the exact scan
        if slices is None:
            assert eng.last_topk_fallbacks <= max(2, nq // 8), eng.last_topk_fallbacks
    else:
        assert d > 320 or k > 24 or V < 1024


# ---- C. TRAIN at the NV boundaries and at NV = 4 ---------------------------------------------------------------------
@pytest.mark.parametrize("d", [127, 254, 255, 382, 383, 448, 510])
def test_train_embedding_sizes_nv_edges(d):
    """NV = ceil(S / 128) float4 per lane, S = (d + 9) & ~7: 127 -> 1 vs 2 ... 383 -> 4; the masked last float4 moves."""
    ref, rl, got, l, _ = _run_pair(200, d, 64, 12, K=5, numpy_oracle=d <= 128)
    _assert_close(ref, rl, got, l)


@pytest.mark.parametrize("optimizer,head", [("Adagrad", "glove"), ("SGD", "glove"), ("Adam", "logistic"),
                                            ("Adagrad", "logistic")])
def test_train_d510_optimizers_and_heads(optimizer, head):
    ref, rl, got, l, _ = _run_pair(200, 510, 64, 12, optimizer=optimizer, head=head, K=5, numpy_oracle=False)
    _assert_close(ref, rl, got, l)


def test_train_d510_lazy():
    ref, rl, got, l, _ = _run_pair(800, 510, 128, 20, adam_mode="lazy", zipf=False, numpy_oracle=False)
    _assert_close(ref, rl, got, l)


def test_train_d510_dense_and_exact_replay_bit_identical():
    ref, rl, got_r, l_r, _ = _run_pair(600, 510, 128, 24, adam_mode="replay_exact", zipf=False, K=7, numpy_oracle=False)
    _, _, got_d, l_d, _ = _run_pair(600, 510, 128, 24, adam_mode="dense", zipf=False, K=7, numpy_oracle=False)
    _assert_close(ref, rl, got_r, l_r, "d510_dense_vs_exact/replay_exact")
    _assert_close(ref, rl, got_d, l_d, "d510_dense_vs_exact/dense")
    for k in ("R", "C", "rb", "cb"):
        assert np.array_equal(got_r[k], got_d[k]), k
    assert np.array_equal(l_r, l_d)


def test_train_d510_heavy_hitters():
    """40 % of a 4096 batch on one row id and one col id: split segments, partial sums of four float4 per lane."""
    ref, rl, got, l, eng = _run_pair(300, 510, 4096, 6, hot=0.4, K=3, numpy_oracle=False)
    _assert_close(ref, rl, got, l)
    counts = eng.batch_counts(eng.host_step - 1)
    assert counts[2] > counts[0] and counts[3] > counts[1]     # more items than segments => split segments exist


def test_train_d448_row_sharded_peer_push_shared_plans():
    _run_row_sharded(2, "replay", "Adam", 601, "peer-push+shared-plans", d=448)


def test_embedding_size_511_is_refused():
    from glove_tensorflow_b200.engine import GloveEngine
    GloveEngine(10, 510, batch_size=8, plan_steps=1, max_steps=2)
    with pytest.raises(ValueError):
        GloveEngine(10, 511, batch_size=8, plan_steps=1, max_steps=2)


# ---- D. EVAL --------------------------------------------------------------------------------------------------------
EVAL_N = 2017           # = 2 * 1000 + 17, 61 * 33 + 4, 65 * 31 + 2: a short last batch at every batch size below
NEG_FACTOR = 0.7


def _softplus64(x):
    return np.maximum(x, 0.0) + np.log1p(np.exp(-np.abs(x)))


def _eval_terms(st, coo, head):
    """fp64 per-triple terms of the 8 EVAL sums, and an fp32 error scale for each: |term| + |d term / d z| * sum of the
    magnitudes that make up z (the logit is formed in fp32 by the kernel)."""
    R, C = st.R.astype(np.float64), st.C.astype(np.float64)
    rb, cb, g = st.rb.astype(np.float64), st.cb.astype(np.float64), float(st.g)
    i, j = coo["row"], coo["col"]
    prod = R[i] * C[j]
    z = prod.sum(1) + rb[i] + cb[j] + g
    mz = np.abs(prod).sum(1) + np.abs(rb[i]) + np.abs(cb[j]) + abs(g)
    sig = lambda x: 1.0 / (1.0 + np.exp(-x))
    if head == "glove":
        y, w = coo["target"].astype(np.float64), coo["weight"].astype(np.float64)
        t = [w * (z - y) ** 2, w, w * y, w * z]
        dz = [2 * w * np.abs(z - y), 0 * w, 0 * w, w]
    else:
        p, n = coo["pos"].astype(np.float64), coo["neg"].astype(np.float64)
        t = [p * _softplus64(-z), p, n * _softplus64(z), n]
        dz = [p * sig(-z), 0 * p, n * sig(z), 0 * n]
    t += [(R[i] ** 2).sum(1), (C[j] ** 2).sum(1), rb[i] ** 2, cb[j] ** 2]
    dz += [0 * z] * 4
    terms = np.stack(t, 1)
    scale = np.abs(terms) + np.stack(dz, 1) * mz[:, None]
    return terms, scale


def _batch_sums(x, first, count, B):
    x = x[first:first + count]
    return np.add.reduceat(x, np.arange(0, count, B), axis=0)


def _metrics64(sums, sizes, head, g, d, lam=0.01, reg_scale=2.0, neg_factor=NEG_FACTOR):
    """EVAL metrics from per-batch fp64 sums: RegressionHead / MultiHead(BinaryClassHead x 2) over batches of `sizes`
    triples, with the activity-L2 term of each batch (reg_loss)."""
    s = sums
    reg = reg_scale * ((lam / d) * s[:, 4] / sizes + (lam / d) * s[:, 5] / sizes + lam * s[:, 6] / sizes
                       + lam * s[:, 7] / sizes + lam * g * g)
    if head == "glove":
        return {"average_loss": s[:, 0].sum() / s[:, 1].sum(), "loss": np.mean(s[:, 0] / sizes + reg),
                "label/mean": s[:, 2].sum() / s[:, 1].sum(), "prediction/mean": s[:, 3].sum() / s[:, 1].sum(),
                "regularization_loss": np.mean(reg)}
    return {"loss": np.mean(s[:, 0] / sizes + neg_factor * s[:, 2] / sizes + reg), "regularization_loss": np.mean(reg),
            "pos/average_loss": s[:, 0].sum() / s[:, 1].sum(), "neg/average_loss": s[:, 2].sum() / s[:, 3].sum()}


@pytest.mark.parametrize("head", ["glove", "logistic"])
@pytest.mark.parametrize("d", [20, 200, 300, 510])
def test_eval_sums_and_metrics(d, head):
    from glove_tensorflow_b200.engine import GloveEngine
    V = 300
    coo = make_coo(V, EVAL_N, 21 + d)
    st = o.init_state(V, d, 22 + d)
    st.g = np.float32(0.3)
    eng = GloveEngine(V, d, head=head, neg_factor=NEG_FACTOR, batch_size=64, plan_steps=2, max_steps=8)
    eng.load_state(st.R, st.C, st.rb, st.cb, st.g)
    a, b = ("target", "weight") if head == "glove" else ("pos", "neg")
    eng.set_coo(coo["row"], coo["col"], coo[a], coo[b])
    terms, scale = _eval_terms(st, coo, head)
    # whole passes at batch sizes on both sides of the 32-triple tile, then windows that start mid-batch, a window
    # shorter than one batch and the single last triple
    windows = [(B, 0, EVAL_N) for B in (1, 31, 33, 1000)] + [(31, 45, 1500), (33, 17, 33 * 5 + 7), (1000, 5, 700),
                                                              (1, EVAL_N - 1, 1)]
    for B, first, count in windows:
        got = eng.eval_sums(B, first=first, count=count)
        want = _batch_sums(terms, first, count, B)
        tol = 1e-5 * _batch_sums(scale, first, count, B) + 1e-12
        assert got.shape == want.shape == ((count + B - 1) // B, 8)
        err = np.abs(got - want) / tol
        assert np.all(err <= 1), (B, first, count, np.unravel_index(np.argmax(err), err.shape), float(err.max()))
    g = float(np.float32(0.3))
    for B in (1, 31, 33, 1000):
        sums = _batch_sums(terms, 0, EVAL_N, B)
        sizes = np.minimum(B, EVAL_N - B * np.arange(len(sums))).astype(np.float64)
        want = _metrics64(sums, sizes, head, g, d)
        got = eng.eval_metrics(B)
        assert set(got) == set(want)
        for k, v in want.items():
            assert abs(got[k] - v) <= 1e-5 * max(abs(v), 1e-3), (B, k, got[k], v)
