"""The analogy and pair-cosine kernels (glove_analogy.cu) at their edges, against the float64 oracle
(oracle/analogy_oracle.py) with the id rule of test_analogy_gpu._check:
  A. live columns past d: random non-zero row and column biases on every table of this file, random values in the padding
     of one-plane tables, and NaN / inf there too, at the float4 tails d % 4 = 1, 2, 3, 0 and at NV = 3 / 4;
  B. a pairwise-style shape sweep (d, V, questions, k, restricted vocabulary, forced top-k slicing), with the tensor-core
     and exact fp32 3CosAdd paths bit-identical wherever the tensor-core pass runs;
  C. exact ties planted on the warp, 256-row tile and 3CosMul slice edges, copies of a, b and c that must not be excluded,
     and repeated words;
  D. batch independence of 3CosMul and exact 3CosAdd, pair cosines equal to the top-k similarity at the NV edges;
  E. tables as training leaves them (replay and lazy Adam), retraining, replaced tables at the same step, one-plane tables;
  F. the adversarial bf16 table of test_topk_bound.py through the tensor-core 3CosAdd path;
  G. zero rows and rows below the 1e-12 floor of the sum of squares.
Rows large enough to overflow the fp32 sum of squares are out of scope: fp32 tf.math.l2_normalize overflows there too."""
import numpy as np
import pytest

from conftest import make_coo
from oracle import analogy_oracle as ao
from test_analogy_gpu import _check
from test_topk_bound import adversarial_table

pytestmark = pytest.mark.gpu

METHODS = (("add", False), ("add", True), ("mul", False))    # 3CosAdd tensor-core path, 3CosAdd exact fp32, 3CosMul
PAIR_ATOL = 1e-6                                              # as test_pair_cosine_is_the_topk_similarity_bit_for_bit


def _biases(rng, V):
    return (rng.uniform(0.5, 3.0, V) * rng.choice([-1.0, 1.0], V)).astype(np.float32)


def _engine(W, optimizer="SGD", seed=0, **kw):
    """Engine whose row table holds W, with random non-zero row and column biases (the row bias is column d of the
    packed row) and random column vectors; on a one-plane table the columns d+1..S-1 get random values as well."""
    import torch
    from glove_tensorflow_b200.engine import GloveEngine
    V, d = W.shape
    rng = np.random.default_rng(seed + 12345)
    eng = GloveEngine(V, d, optimizer=optimizer, batch_size=64, plan_steps=1, max_steps=64, **kw)
    eng.load_state(W, rng.normal(size=W.shape).astype(np.float32), _biases(rng, V), _biases(rng, V))
    if eng.P == 1:
        eng.row_plane()[:, d + 1:] = torch.from_numpy(rng.uniform(-3.0, 3.0, (V, eng.S - d - 1)).astype(np.float32)).cuda()
    return eng


def _table(rng, V, d):
    """Random rows.  For d <= 4 every entry is positive: with a handful of dimensions, rows nearly opposite to a lie within
    fp32 noise of 1 + cos(a, x) = 0, where 3CosMul's 1 / (pa + 1e-3) amplifies that noise past the tolerance."""
    if d <= 4:
        return rng.uniform(0.05, 1.0, (V, d)).astype(np.float32)
    return rng.normal(size=(V, d)).astype(np.float32)


def _questions(rng, R, n):
    abc = rng.integers(0, R, (n, 3))
    for i, (x, y) in enumerate([(0, 1), (0, 2), (1, 2)][: n]):   # a = b, a = c, b = c
        abc[i, y] = abc[i, x]
    if n > 3:
        abc[3, 1:] = abc[3, 0]                                    # a = b = c
    return abc


def _tc_runs(eng, k, restrict):
    """Whether glove_topk_cosine_queries takes the tensor-core pass for the k + 3 list of 3CosAdd."""
    return eng.tc_path_covers(k + 3) and (restrict is None or restrict >= 1024)


def _run(eng, abc, k, restrict=None):
    """{(method, exact): (score, idx)} for every method and path."""
    return {(m, ex): eng.analogy(abc, k, m, restrict=restrict, exact_fp32=ex) for m, ex in METHODS}


def _verify(eng, W, abc, k, res, restrict=None):
    """Every result against the oracle; the two 3CosAdd paths bit-identical where the tensor-core pass runs."""
    for (method, exact), (s, i) in res.items():
        assert s.shape == i.shape == (len(abc), k)
        _check(W, abc, k, method, restrict, s, i)
    if _tc_runs(eng, k, restrict):
        (s_tc, i_tc), (s_ex, i_ex) = res["add", False], res["add", True]
        np.testing.assert_array_equal(i_tc, i_ex)
        np.testing.assert_array_equal(s_tc.view(np.uint32), s_ex.view(np.uint32))
    return res


def _analogies(eng, W, abc, k, restrict=None):
    return _verify(eng, W, abc, k, _run(eng, abc, k, restrict), restrict)


def _bits_equal(x, y):
    np.testing.assert_array_equal(np.asarray(x, np.float32).view(np.uint32), np.asarray(y, np.float32).view(np.uint32))


# ---- A. live columns past d ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", [29, 30, 31, 32, 381, 382, 383])
def test_live_bias_and_padding_columns(d):
    """d % 4 = 1, 2, 3, 0 put the bias into the last float4 of the 3CosMul column chunk at each offset; 381..383 are the
    last NV = 3 size and the first NV = 4 ones (S = 384, 384, 392)."""
    rng = np.random.default_rng(100 + d)
    V = 3000
    W = _table(rng, V, d)
    eng = _engine(W, seed=d)
    abc = _questions(rng, V, 40)
    for k in (1, 21, 29):
        _analogies(eng, W, abc, k)
    pairs = rng.integers(0, V, (600, 2))
    np.testing.assert_allclose(eng.pair_cosine(pairs), ao.pair_cosine(W, pairs), rtol=0, atol=PAIR_ATOL)


@pytest.mark.parametrize("d", [29, 30, 31, 32, 383])
def test_non_finite_columns_past_d_are_ignored(d):
    """NaN, inf and -inf in the bias, last_step and padding columns of every row: nothing past column d may reach a score,
    a similarity or a norm (a diverged bias must not poison the evaluation of the embedding)."""
    rng = np.random.default_rng(200 + d)
    V = 1500
    W = _table(rng, V, d)
    eng = _engine(W, seed=d)
    junk = np.array([np.nan, np.inf, -np.inf], np.float32)[np.arange(eng.S - d) % 3]
    import torch
    eng.row_plane()[:, d:] = torch.from_numpy(np.tile(junk, (V, 1))).cuda()
    abc = _questions(rng, V, 24)
    for k in (1, 8):
        _analogies(eng, W, abc, k)
    pairs = rng.integers(0, V, (300, 2))
    got = eng.pair_cosine(pairs)
    np.testing.assert_allclose(got, ao.pair_cosine(W, pairs), rtol=0, atol=PAIR_ATOL)
    q = rng.integers(0, V, 16)
    for exact in (False, True):
        sim, idx = eng.topk(q, 8, exact_fp32=exact)
        assert np.all(np.isfinite(sim))
        _bits_equal(eng.pair_cosine(np.stack([np.repeat(q, 8), idx.reshape(-1)], 1)), sim.reshape(-1))


# ---- B. shape sweep -------------------------------------------------------------------------------------------------
# (d, V, n questions, k, restrict, GLOVE_TOPK_SLICES).  d = 1..4: one float4; 33 / 129: one column past a 32-column chunk;
# 383..510: NV = 4 (exact scan only).  V = k + 3 is the smallest legal table, 255..257 the first 3CosMul tile, 1023 / 1024
# the tensor-core floor, >= 16,384 the 64-slice cap of mul_plan at few questions; n >= 2,369 drops mul_plan to one slice.
SWEEP = [(1, 4, 1, 1, None, None), (1, 16384, 9, 8, None, "3"), (3, 31, 7, 8, None, None), (3, 257, 1, 29, 32, None),
         (4, 255, 8, 21, None, "3"), (4, 1023, 2369, 1, 255, None), (33, 256, 9, 29, None, None),
         (33, 5249, 1, 21, 257, "1"), (64, 5249, 9, 8, 1500, "3"), (128, 257, 2369, 8, None, None),
         (128, 1024, 2400, 29, 255, None), (129, 1023, 1, 21, 24, None), (129, 5249, 2369, 1, None, None),
         (300, 1024, 7, 1, None, "1"), (300, 16400, 8, 21, None, "3"), (300, 24, 8, 21, None, None),
         (383, 5249, 8, 8, 257, None), (383, 1024, 1, 29, None, "1"), (448, 16411, 9, 29, None, None),
         (448, 31, 8, 21, None, None), (510, 20000, 1, 1, 255, None), (510, 256, 7, 8, None, None),
         (510, 1024, 2369, 21, 1024, "3")]


@pytest.mark.parametrize("d,V,n,k,restrict,slices", SWEEP)
def test_analogy_shape_sweep(monkeypatch, d, V, n, k, restrict, slices):
    if slices is None:
        monkeypatch.delenv("GLOVE_TOPK_SLICES", raising=False)
    else:
        monkeypatch.setenv("GLOVE_TOPK_SLICES", slices)
    assert k + 3 <= (V if restrict is None else restrict)
    rng = np.random.default_rng(d * 1009 + V + n)
    W = _table(rng, V, d)
    R = V if restrict is None else restrict
    abc = _questions(rng, R, n)
    if d > 4:                                                 # the last candidate row answers the last question
        abc[-1] = rng.choice(R - 1, 3, replace=False)
        Wn = ao.normalise(W)
        W[R - 1] = Wn[abc[-1, 1]] - Wn[abc[-1, 0]] + Wn[abc[-1, 2]]
    eng = _engine(W, seed=d + V)
    res = _analogies(eng, W, abc, k, restrict)
    if d > 4:
        for method in METHODS:
            assert res[method][1][-1, 0] == R - 1, (method, res[method][1][-1])


# ---- C. exact ties and exclusion ------------------------------------------------------------------------------------
def _tie_positions(V, ns):
    """Rows where the order of exact ties is decided by separate code: two rows of one warp, the last row of a warp and the
    first of the next, both sides of a 256-row tile edge in the first two 3CosMul slices, both sides of the first two slice
    edges (for each batch size in ns), and the last row."""
    pos = {40, 45, 63, 64, 255, 256, V - 1}
    for n in ns:
        _, slices, rps = ao.mul_plan(V, n)
        for s in (1, 2):
            if s < slices:
                pos |= {s * rps - 1, s * rps}
        pos |= {rps + 255, rps + 256}
    return sorted(p for p in pos if p < V)


def test_exact_ties_exclusion_and_repeated_words():
    rng = np.random.default_rng(31)
    V, d, k = 20000, 64, 21
    W = _table(rng, V, d)
    pad = 300                                                 # a second batch size: 8 slices of 2,500 rows, not 64 of 313
    ties = _tie_positions(V, (8, pad))
    x = 7000                                                  # the answer row; its copies sit on every edge
    W[ties] = W[x]
    e = lambda: rng.normal(size=d).astype(np.float32) * 0.05
    W[9100], W[9200], W[9300] = W[x] + e(), W[x] + e(), W[x] + e()
    y = rng.normal(size=d).astype(np.float32)                 # a second cluster: a, b, c near y, copies of each elsewhere
    a2, b2, c2 = 12000, 12001, 12002
    W[a2], W[b2], W[c2] = y + e(), y + e(), y + e()
    copies = {a2: [300, 15000], b2: [11999], c2: [19998]}
    for src, dst in copies.items():
        W[dst] = W[src]
    eng = _engine(W, seed=3)
    copy_ids = sorted(i for v in copies.values() for i in v)
    abc = np.array([[9100, 9200, 9300],                       # the answer: x and its copies, exactly tied
                    [a2, b2, c2],                             # a, b, c excluded, their copies under other ids are not
                    [a2, a2, c2], [a2, b2, a2], [a2, b2, b2], [a2, a2, a2],    # repeated words
                    [9100, 9100, 9300], [9300, 9200, 9300]])
    answer = sorted(ties + [x])
    for n_batch in (len(abc), pad):
        q = np.concatenate([abc, rng.integers(0, V, (n_batch - len(abc), 3))]) if n_batch > len(abc) else abc
        for (method, exact), (s, i) in _analogies(eng, W, q, k).items():
            m = min(k, len(answer))
            assert i[0, :m].tolist() == answer[:m], (method, exact, i[0])
            assert np.all(s[0, :m] == s[0, 0]), (method, exact)
            assert set(i[1, :len(copy_ids)].tolist()) == set(copy_ids), (method, exact, i[1])
            for r in range(1, 6):
                assert not set(i[r].tolist()) & set(q[r].tolist())
                for src, dst in copies.items():                   # a copy of an excluded word is still a candidate
                    if src in q[r]:
                        assert set(dst) <= set(i[r].tolist()), (method, exact, r, src)
                    same = [j for j in np.nonzero(np.isin(i[r], [src] + dst))[0]]
                    assert [i[r, j] for j in same] == sorted(i[r, j] for j in same)   # tied copies in id order


# ---- D. batch independence and pair cosines ---------------------------------------------------------------------------
def test_results_do_not_depend_on_the_batch():
    """A question's 3CosMul and exact 3CosAdd answers depend on that question only: asked alone, in batches of 9, 300 and
    2,500 at several offsets (64, 64, 8 and 1 3CosMul slices) and in reverse order, scores and ids are bit-identical."""
    rng = np.random.default_rng(41)
    V, d, k = 20000, 96, 10
    W = _table(rng, V, d)
    eng = _engine(W, seed=4)
    Q = _questions(rng, V, 9)
    for method, exact in (("mul", False), ("add", True)):
        ref_s, ref_i = eng.analogy(Q, k, method, exact_fp32=exact)
        _check(W, Q, k, method, None, ref_s, ref_i)
        for j in range(len(Q)):
            s, i = eng.analogy(Q[j:j + 1], k, method, exact_fp32=exact)
            _bits_equal(s[0], ref_s[j])
            assert i[0].tolist() == ref_i[j].tolist()
        s, i = eng.analogy(Q[::-1], k, method, exact_fp32=exact)
        _bits_equal(s[::-1], ref_s)
        np.testing.assert_array_equal(i[::-1], ref_i)
        for n, off in ((300, 0), (300, 291), (2500, 5), (2500, 1234), (2500, 2491)):
            big = rng.integers(0, V, (n, 3))
            big[off:off + len(Q)] = Q
            s, i = eng.analogy(big, k, method, exact_fp32=exact)
            _bits_equal(s[off:off + len(Q)], ref_s)
            np.testing.assert_array_equal(i[off:off + len(Q)], ref_i)


# the self-cosine is a sum of d rounded squares of rounded normalised entries: emulating the kernel's operation order
# in NumPy gives at most 4 units of 2^-24 below 1 and 2 units of 2^-23 above at d = 1..510, so 1 ulp is not attainable
SELF_COS_TOL = 2.0 ** -21


@pytest.mark.parametrize("d", [1, 127, 128, 383, 510])
def test_pair_cosine_is_the_topk_similarity_at_the_nv_edges(d):
    rng = np.random.default_rng(50 + d)
    V = 3000
    W = _table(rng, V, d)
    eng = _engine(W, seed=d)
    q = rng.integers(0, V, 40)
    for exact in (False, True):
        sim, idx = eng.topk(q, 8, exact_fp32=exact)
        pairs = np.stack([np.repeat(q, 8), idx.reshape(-1)], 1)
        got = eng.pair_cosine(pairs)
        _bits_equal(got, sim.reshape(-1))
    np.testing.assert_allclose(got, ao.pair_cosine(W, pairs), rtol=0, atol=PAIR_ATOL)
    ids = np.arange(0, V, 7)
    self_cos = eng.pair_cosine(np.stack([ids, ids], 1)).astype(np.float64)
    assert np.max(np.abs(self_cos - 1.0)) <= SELF_COS_TOL, float(np.max(np.abs(self_cos - 1.0)))


# ---- E. tables as training leaves them --------------------------------------------------------------------------------
def _trained_engine(adam_mode, V, d, seed):
    from glove_tensorflow_b200.engine import GloveEngine
    rng = np.random.default_rng(seed)
    eng = GloveEngine(V, d, optimizer="Adam", adam_mode=adam_mode, learning_rate=0.05, batch_size=256, plan_steps=4,
                      max_steps=256)
    eng.load_state(rng.normal(size=(V, d)).astype(np.float32), rng.normal(size=(V, d)).astype(np.float32),
                   _biases(rng, V), _biases(rng, V))
    coo = make_coo(V, 60000, seed)
    eng.set_coo(coo["row"], coo["col"], coo["target"], coo["weight"])
    return eng


@pytest.mark.parametrize("adam_mode", ["replay", "lazy"])
def test_trained_tables(adam_mode):
    """Analogies straight after training (the lazy-Adam flush and the normalised table come from the analogy call itself),
    again after more training, and after a new table at the same step; the three-plane table has live Adam state and
    live biases.  The oracle sees get_state()["R"]."""
    rng = np.random.default_rng(61)
    V, d, k = 1200, 31, 8
    eng = _trained_engine(adam_mode, V, d, 7)
    eng.train(24)
    abc = _questions(rng, V, 40)
    first = _run(eng, abc, k)                                 # no get_state before: the analogy flushes by itself
    pc_pairs = rng.integers(0, V, (200, 2))
    pc = eng.pair_cosine(pc_pairs)
    st = eng.get_state(slots=True)
    assert np.abs(st["R/s0"]).max() > 0 and np.abs(st["R/s1"]).max() > 0 and np.all(st["rb"] != 0)
    W1 = st["R"]
    _verify(eng, W1, abc, k, first)
    np.testing.assert_allclose(pc, ao.pair_cosine(W1, pc_pairs), rtol=0, atol=PAIR_ATOL)
    # more training: the second answer is that of the new rows
    eng.train(24)
    second = _run(eng, abc, k)
    W2 = eng.get_state()["R"]
    _verify(eng, W2, abc, k, second)
    assert np.abs(W2 - W1).max() > 1e-3
    assert any(not np.array_equal(second[m][0], first[m][0]) for m in METHODS)
    # a new table at the same step: the normalised copy keyed on the step must not be reused
    step = eng.host_step
    eng.load_state(rng.normal(size=(V, d)).astype(np.float32), rng.normal(size=(V, d)).astype(np.float32),
                   _biases(rng, V), _biases(rng, V))
    third = _run(eng, abc, k)
    assert eng.host_step == step
    _verify(eng, eng.get_state()["R"], abc, k, third)
    # and one from init_uniform, again at the same step
    eng.init_uniform(seed=5)
    fourth = _run(eng, abc, k)
    _verify(eng, eng.get_state()["R"], abc, k, fourth)


def test_one_plane_tables_row_plane_and_vectors_file(tmp_path):
    """The one-plane table of an evaluation-only engine: rows rewritten in place through row_plane() after a first
    analogy (the cached normalised table must go), and the engine vectors_engine builds from a GloVe text file."""
    import torch
    from glove_tensorflow_b200 import vectors
    rng = np.random.default_rng(71)
    V, d, k = 1500, 50, 5
    W = _table(rng, V, d)
    eng = _engine(W, seed=7)
    abc = _questions(rng, V, 30)
    _analogies(eng, W, abc, k)
    W2 = _table(rng, V, d)
    eng.row_plane()[:, :d] = torch.from_numpy(W2).cuda()
    _analogies(eng, W2, abc, k)
    path = str(tmp_path / "vectors.txt")
    vectors.write_vectors(path, ["w%d" % i for i in range(V)], W2, header=True)
    veng, words = vectors.vectors_engine(path)
    assert len(words) == V and veng.P == 1
    res = _analogies(veng, W2, abc, k)
    for m in METHODS:                                         # the same rows, whatever else the packed row holds
        np.testing.assert_array_equal(res[m][1], eng.analogy(abc, k, m[0], exact_fp32=m[1])[1])


# ---- F. adversarial bf16 rounding through 3CosAdd ----------------------------------------------------------------------
@pytest.mark.parametrize("table_k,k", [(1, 1), (1, 5), (5, 1), (5, 5)])
def test_adversarial_bf16_table_through_3cosadd(table_k, k):
    """(a, b, a) asks for the rows nearest b^ (up to rounding) outside {a, b}.  b is an adversarial query row of
    test_topk_bound.py: it loses ~2^-7 of its self-similarity to bf16 rounding and 32 other rows outrank it there.  b'
    (and the table's other copies of b) carry the same loss, and they are the true answers: the tensor-core path must
    find them, as the exact path and the oracle do."""
    T, queries, near, fill = adversarial_table(k=table_k)
    V0 = len(T)
    extra = np.tile(T[queries[:1]], (len(queries), 1))        # one more copy b' per query row, under new ids
    T = np.concatenate([T, extra])
    V = len(T)
    copies = sorted(list(queries) + list(range(V0, V)))
    eng = _engine(T, seed=table_k)
    assert _tc_runs(eng, k, None)
    unrelated = [500, 700, 900, 1100, 1300][: len(queries)]
    abc = np.array([[a, b, a] for a, b in zip(unrelated, queries)])
    res = _analogies(eng, T, abc, k)
    for r, b in enumerate(queries):
        want = [c for c in copies if c != b][:k]
        m = len(want)
        for method in (("add", False), ("add", True)):
            s, i = res[method]
            assert i[r, :m].tolist() == want, (method, r, i[r])
        if table_k == 1:
            assert res["add", False][1][r, 0] == V0               # b' comes first


# ---- G. degenerate rows -----------------------------------------------------------------------------------------------
def test_zero_and_tiny_rows():
    """Zero rows and rows at 1e-20 (sum of squares ~1e-38, under the 1e-12 floor) as candidates and as a, b or c, held to
    the oracle's normalise with the same floor.  All three words zero: every candidate scores exactly the same, so the
    answer is the k lowest ids outside the question."""
    rng = np.random.default_rng(81)
    V, d, k = 2000, 64, 8
    W = _table(rng, V, d)
    zero, tiny = [3, 700, 1999], [5, 800, 1500]
    W[zero] = 0.0
    W[tiny] = (rng.normal(size=(len(tiny), d)) * 1e-20).astype(np.float32)
    eng = _engine(W, seed=8)
    a, b, c = 10, 20, 30
    abc = np.array([[3, b, c], [a, 3, c], [a, b, 3], [3, 700, 1999], [3, 3, 3],
                    [5, b, c], [a, 800, c], [a, b, 1500], [5, 800, 1500], [5, 3, 800], [a, b, c]])
    res = _analogies(eng, W, abc, k)
    for (method, exact), (s, i) in res.items():
        for r in (3, 4):
            want = [v for v in range(V) if v not in abc[r]][:k]
            assert i[r].tolist() == want, (method, exact, r, i[r])
            assert np.all(s[r] == s[r, 0])
    pairs = np.array([[3, 4], [3, 3], [5, 800], [5, 5], [6, 1500], [1999, 700]])
    np.testing.assert_allclose(eng.pair_cosine(pairs), ao.pair_cosine(W, pairs), rtol=0, atol=PAIR_ATOL)
