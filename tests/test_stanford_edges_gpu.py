"""Edge tests of Stanford GloVe's trainer and co-occurrence finish on the GPU, compared bit for bit with
oracle/stanford_glove_oracle in the kernel's order (order=1), on the GPU's own parsed records:

  A  every branch of sgd_epoch_kernel (clip, diff skip, update gate, check_nan on the bias step) with injected W and
     gradsq: the oracle's CASES, clip 0 / -1 / inf, eta 0 / -0.05 / inf, gradsq and W at 0, subnormal, negative,
     infinite, NaN, huge and -0.0, and a table that diverges by itself
  B  every lane template K = 1..16 of sgd_epoch_kernel, at d = 1, 32k and 32k + 1, and 511
  C  log(val) and f at the edges of val, x_max and alpha against 60-digit decimal references, then one epoch on them
  D  record structure (V at 1..3 and around 2^16, one record, one repeated record, alternating and self pairs): links
     and epochs, and the same bits for grids of 1, 2, 3, 37, the default and 20,000 CTAs
  E  the epoch cost's fixed-shape sum at one, two and three reduction levels
  F  the rows of the vectors file around FLT_MAX, subnormal, infinite and NaN values, V around the <unk> row's 100
  G  glove_cooc_finish_stanford / glove_cooc_finish_sorted: value = numer / lcm(1..window) correctly rounded for every
     numerator below 2^63

Bits are compared through integer views; the one exception is NaN, which equals any NaN (CUDA produces a canonical
NaN and x86 its default -NaN, so payloads may differ)."""
import ctypes
import math
from decimal import Decimal, localcontext

import numpy as np
import pytest

from oracle import stanford_glove_oracle as sgo
from test_stanford_glove import CASES, _start, table

pytestmark = pytest.mark.gpu

REC = np.dtype([("w1", "<i4"), ("w2", "<i4"), ("val", "<f8")])
SKIP, CLIP, GATE, CHECK_NAN = range(4)         # oracle branch counters (sgo.epoch's hits)


def assert_bits(got, want, what="values"):
    """got and want hold the same bits (NaN equals any NaN)."""
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, want.shape, got.dtype, want.dtype)
    iv = {8: np.int64, 4: np.uint32}[got.dtype.itemsize]
    bad = (got.view(iv) != want.view(iv)) & ~(np.isnan(got) & np.isnan(want))
    if bad.any():
        i = np.argwhere(bad)[0]
        raise AssertionError("%s: %d of %d differ in their bits, first at %s: %r != %r"
                             % (what, int(bad.sum()), bad.size, tuple(i.tolist()), got[tuple(i)], want[tuple(i)]))


def write_bin(path, w1, w2, val):
    rec = np.zeros(len(w1), REC)
    rec["w1"], rec["w2"], rec["val"] = w1, w2, val
    rec.tofile(path)
    return str(path)


def trainer(path, w1, w2, val, V, d, x_max=100.0, alpha=0.75):
    from glove_tensorflow_b200.stanford_glove import StanfordGlove
    return StanfordGlove(write_bin(path, w1, w2, val), V, d, alpha=alpha, x_max=x_max, seed=1)


def run(sg, epochs, eta=0.05, clip=100.0, W=None, G=None, grid=0):
    """Sets W / G (if given), runs `epochs` epochs on the GPU and in the kernel-order oracle on the GPU's records, and
    checks W, gradsq and every epoch cost bit for bit.  Returns the oracle's (W0, W, G, branch counts, record costs)."""
    import torch
    if W is not None:
        sg.W.copy_(torch.from_numpy(W))
    if G is not None:
        sg.gradsq.copy_(torch.from_numpy(G))
    W0 = sg.W.cpu().numpy().copy()
    Wo, Go = W0.copy(), sg.gradsq.cpu().numpy().copy()
    words, lf = sg.words.cpu().numpy(), sg.lf.cpu().numpy()
    hits, costs = np.zeros(4, np.int64), []
    for e in range(epochs):
        costs.append(sgo.epoch(Wo, Go, words, lf, eta, clip, order=1, hits=hits))
        got = sg.epoch(eta, clip, grid)
        assert_bits(np.float64(got), np.float64(sgo.kernel_cost(costs[-1])), "cost of epoch %d" % (e + 1))
    assert_bits(sg.W.cpu().numpy(), Wo, "W")
    assert_bits(sg.gradsq.cpu().numpy(), Go, "gradsq")
    return W0, Wo, Go, hits, costs


def zipf_words(rng, V, n):
    p = 1.0 / np.arange(1, V + 1)
    return rng.choice(V, n, p=p / p.sum()) + 1, rng.choice(V, n, p=p / p.sum()) + 1


# ---------------------------------------------------------------------------------------------------------------- A

@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_branches_oracle_cases(tmp_path, case):
    name, seed, V, d, n, kind, eta, clip, tweak = case
    words, lf = table(seed, V, n, kind)
    sg = trainer(tmp_path / "c.bin", words[:, 0] + 1, words[:, 1] + 1, np.exp(lf[:, 0]), V, d)
    W, G = _start(V, d, tweak, seed)
    _, _, Go, hits, _ = run(sg, 2, eta, clip, W, G)
    assert hits[SKIP] < 2 * n
    want = {"clipping": hits[CLIP] > 0, "diff_skip": hits[SKIP] > 0, "update_skip": hits[GATE] > 0 and np.isinf(Go).any(),
            "one_word": (words == 2).any(axis=1).all(),
            "self_and_repeats": (words[:, 0] == words[:, 1]).any() and (words[1:] == words[:-1]).all(axis=1).any()}
    assert want.get(name, True), (name, hits)


def _table_a(tmp_path, d=5):
    rng = np.random.default_rng(21)
    w1, w2 = zipf_words(rng, 12, 400)
    return trainer(tmp_path / "a.bin", w1, w2, np.exp(rng.uniform(-3, 6, 400)), 12, d)


def _set(G, rows, cols, v):
    G = G.copy()
    G[rows, cols] = v
    return G


# name: (eta, clip, W tweak, gradsq tweak, evidence on the oracle's run)
_VEC, _BIAS = (slice(0, None, 2), slice(0, 5)), (slice(None), 5)
STATES = {
    "clip_0": (0.05, 0.0, None, None, lambda h, W0, W, G: h[CLIP] > 0),
    "clip_-1": (0.05, -1.0, None, None, lambda h, W0, W, G: h[CLIP] > 0),
    "clip_inf": (0.05, math.inf, None, None, lambda h, W0, W, G: h[CLIP] == 0 and (W != W0).any()),
    "eta_0": (0.0, 100.0, None, None, lambda h, W0, W, G: (W[:, :5] == W0[:, :5]).all() and (W[:, 5] != W0[:, 5]).any()),
    "eta_-0.05": (-0.05, 100.0, None, None, lambda h, W0, W, G: (W[:, :5] != W0[:, :5]).any()),
    "eta_inf": (math.inf, 100.0, None, None, lambda h, W0, W, G: h[GATE] > 0 and np.isinf(G).any()),
    "gradsq_vec_0": (0.05, 100.0, None, (_VEC, 0.0), lambda h, W0, W, G: h[GATE] > 0),
    "gradsq_vec_min_subnormal": (0.05, 100.0, None, (_VEC, 5e-324), lambda h, W0, W, G: np.abs(W).max() > 1e100),
    "gradsq_vec_-1": (0.05, 100.0, None, (_VEC, -1.0), lambda h, W0, W, G: h[GATE] > 0),
    "gradsq_vec_inf": (0.05, 100.0, None, (_VEC, math.inf), lambda h, W0, W, G: (W[::2, :5] == W0[::2, :5]).all()),
    "gradsq_vec_nan": (0.05, 100.0, None, (_VEC, math.nan), lambda h, W0, W, G: h[GATE] > 0),
    "gradsq_bias_0": (0.05, 100.0, None, (_BIAS, 0.0), lambda h, W0, W, G: h[CHECK_NAN] > 0),
    "gradsq_bias_min_subnormal": (0.05, 100.0, None, (_BIAS, 5e-324), lambda h, W0, W, G: np.abs(W[:, 5]).max() > 1e100),
    "gradsq_bias_-1": (0.05, 100.0, None, (_BIAS, -1.0), lambda h, W0, W, G: h[CHECK_NAN] > 0),
    "gradsq_bias_inf": (0.05, 100.0, None, (_BIAS, math.inf), lambda h, W0, W, G: (W[:, 5] == W0[:, 5]).all()),
    "gradsq_bias_nan": (0.05, 100.0, None, (_BIAS, math.nan), lambda h, W0, W, G: h[CHECK_NAN] > 0),
    "W_inf": (0.05, 100.0, ((0, 1), math.inf), None, lambda h, W0, W, G: h[SKIP] > 0),
    "W_-inf": (0.05, 100.0, ((12, 3), -math.inf), None, lambda h, W0, W, G: h[SKIP] > 0),
    "W_nan": (0.05, 100.0, ((1, 5), math.nan), None, lambda h, W0, W, G: h[SKIP] > 0),
    "W_1e200": (0.05, 100.0, ((13, 2), 1e200), None, lambda h, W0, W, G: h[CLIP] > 0 and np.isinf(G[:, 5]).any()),
    "W_-0": (0.05, 100.0, ((slice(0, 24, 3), slice(0, 5)), -0.0), None,
             lambda h, W0, W, G: (np.signbit(W0) & (W0 == 0)).sum() == 40 and (W[0:24:3, :5] != 0).all()),
}


@pytest.mark.parametrize("state", list(STATES))
def test_branches_injected_state(tmp_path, state):
    eta, clip, wt, gt, evidence = STATES[state]
    sg = _table_a(tmp_path)
    W, G = sg.W.cpu().numpy(), sg.gradsq.cpu().numpy()
    if wt is not None:
        W = _set(W, *wt[0], wt[1])
    if gt is not None:
        G = _set(G, *gt[0], gt[1])
    if clip == 0.0:   # C leaves the sign of fmin / fmax at +-0 unspecified: a -0.0 in W could decide a result
        assert not (np.signbit(W) & (W == 0)).any()
    W0, Wo, Go, hits, _ = run(sg, 2, eta, clip, W, G)
    assert hits[SKIP] < 2 * sg.n, hits
    assert evidence(hits, W0, Wo, Go), (state, hits)


def test_branches_divergent_zipf(tmp_path):
    rng = np.random.default_rng(22)
    V, n = 300, 20_000
    w1, w2 = zipf_words(rng, V, n)
    sg = trainer(tmp_path / "z.bin", w1, w2, np.exp(rng.uniform(-3, 9, n)), V, 20)
    _, Wo, Go, hits, costs = run(sg, 3, eta=10.0)
    assert hits[CLIP] > 0 and min(sgo.kernel_cost(c) for c in costs) > 1e9 and np.abs(Wo).max() > 1e6, hits


# ---------------------------------------------------------------------------------------------------------------- B

LANE_DIMS = [1] + [32 * k for k in range(1, 17)] + [32 * k + 1 for k in range(1, 16)] + [511]


@pytest.fixture(scope="module")
def lane_table(tmp_path_factory):
    rng = np.random.default_rng(31)
    V, n = 700, 30_000
    w1, w2 = zipf_words(rng, V, n)
    return write_bin(tmp_path_factory.mktemp("lanes") / "c.bin", w1, w2, np.exp(rng.uniform(-2, 7, n))), V


@pytest.mark.parametrize("d", LANE_DIMS)
def test_lane_templates(lane_table, d):
    from glove_tensorflow_b200.stanford_glove import StanfordGlove
    path, V = lane_table
    sg = StanfordGlove(path, V, d, seed=5)
    assert_bits(sg.W.cpu().numpy(), sgo.init_params(V, d, 5), "init")
    run(sg, 2)


# ---------------------------------------------------------------------------------------------------------------- C

DBL_MAX, DBL_MIN = np.finfo(np.float64).max, np.finfo(np.float64).tiny


def _edge_vals(x_maxes):
    """(special values, 10^5 log-uniform values over the positive finite doubles)."""
    v = [5e-324, DBL_MIN, 1e-300, 1.0, np.nextafter(1.0, 0), np.nextafter(1.0, 2), 1e300, DBL_MAX]
    for x in x_maxes:
        v += [x, np.nextafter(x, 0), np.nextafter(x, np.inf), np.nextafter(np.nextafter(x, 0), 0)]
    rng = np.random.default_rng(41)
    logu = np.exp2(rng.uniform(-1074, 1024, 100_000))
    return np.array(v, np.float64), np.clip(logu, 5e-324, DBL_MAX)


def _ordered(x):
    i = np.ascontiguousarray(x, np.float64).view(np.int64)
    m = i & np.int64(0x7FFFFFFFFFFFFFFF)
    return np.where(i < 0, -m, m)


def _ulps(got, want):
    g, w = np.asarray(got, np.float64), np.asarray(want, np.float64)
    same_inf = np.isinf(g) & np.isinf(w) & (g == w)
    return np.where(same_inf, 0, np.abs(_ordered(g) - _ordered(w)))


def _dec_ln(x):
    return Decimal(float(x)).ln()


def _ref_pow(q, alpha, ln_q):
    """q ** alpha for a double q >= 0, at 60 digits, rounded once."""
    if q == 0:
        return 1.0 if alpha == 0 else (0.0 if alpha > 0 else math.inf)
    if alpha == 0:
        return 1.0
    if alpha in (1.0, 2.0):
        return float(Decimal(float(q)) ** int(alpha))
    if alpha == 0.5:
        return float(Decimal(float(q)).sqrt())
    return float((Decimal(alpha) * ln_q).exp())


X_MAXES = [1e-300, 1.0, 100.0, 1e300]
ALPHAS = [0.0, 0.5, 0.75, 1.0, 2.0, 8.5, -0.75]
_C_MAX = {"log": 0, "pow": 0}


@pytest.fixture(scope="module")
def edge_records(tmp_path_factory):
    """The values, their 60-digit log, and per x_max the sample of records whose pow is checked with ln(val / x_max)."""
    special, logu = _edge_vals(X_MAXES)
    vals, n_special = np.concatenate([special, logu]), len(special)
    with localcontext() as ctx:
        ctx.prec = 60
        log_ref = np.array([float(_dec_ln(v)) for v in vals])
        rng = np.random.default_rng(42)
        sample = np.concatenate([np.arange(n_special), rng.choice(np.arange(n_special, len(vals)), 4000, replace=False)])
        ln_q = {}
        for x_max in X_MAXES:
            with np.errstate(over="ignore"):
                q = vals[sample] / x_max
            ln_q[x_max] = [None if (qq == 0 or v > x_max) else _dec_ln(qq) for qq, v in zip(q, vals[sample])]
    rng = np.random.default_rng(43)
    V = 50
    w1, w2 = rng.integers(1, V + 1, len(vals)), rng.integers(1, V + 1, len(vals))
    path = write_bin(tmp_path_factory.mktemp("edges") / "c.bin", w1, w2, vals)
    return path, V, vals, log_ref, sample, ln_q


@pytest.mark.parametrize("alpha", ALPHAS)
@pytest.mark.parametrize("x_max", X_MAXES)
def test_parse_edges_log_pow_and_epoch(edge_records, x_max, alpha):
    from glove_tensorflow_b200.stanford_glove import StanfordGlove
    path, V, vals, log_ref, sample, ln_q = edge_records
    sg = StanfordGlove(path, V, 3, alpha=alpha, x_max=x_max, seed=2)
    lf = sg.lf.cpu().numpy()
    lu = _ulps(lf[:, 0], log_ref)
    assert lu.max() <= 1, ("log", vals[np.argmax(lu)], lf[np.argmax(lu), 0], log_ref[np.argmax(lu)])
    f = lf[:, 1]
    above = vals > x_max
    assert_bits(f[above], np.ones(int(above.sum())), "f above x_max")
    with localcontext() as ctx:
        ctx.prec = 60
        want = np.array([1.0 if v > x_max else _ref_pow(v / x_max, alpha, lq)
                         for v, lq in zip(vals[sample], ln_q[x_max])])
    pu = _ulps(f[sample], want)
    assert pu.max() <= 2, ("pow", x_max, alpha, vals[sample][np.argmax(pu)], f[sample][np.argmax(pu)], want[np.argmax(pu)])
    _C_MAX["log"], _C_MAX["pow"] = max(_C_MAX["log"], int(lu.max())), max(_C_MAX["pow"], int(pu.max()))
    print("x_max %g alpha %g: max log error %d ulp, max pow error %d ulp (running max %s)"
          % (x_max, alpha, lu.max(), pu.max(), _C_MAX))
    assert (f[vals == x_max] == 1.0).all() and (f[vals == np.nextafter(x_max, np.inf)] == 1.0).all()
    _, _, _, hits, _ = run(sg, 1)
    if alpha < 0 and x_max >= 100:       # val / x_max underflows to 0: f = inf, the record is skipped
        assert np.isinf(f).any() and hits[SKIP] > 0
    if alpha == 8.5 and x_max >= 1:      # f underflows to 0 and through the subnormals
        assert (f == 0).any() and ((f > 0) & (f < DBL_MIN)).any()


# ---------------------------------------------------------------------------------------------------------------- D

def _structure(kind):
    rng = np.random.default_rng(51)
    if kind.startswith("V="):
        V = int(kind[2:])
        n = 3000
        w1, w2 = rng.integers(1, V + 1, n), rng.integers(1, V + 1, n)
        w1[::97], w2[::89] = V, V           # the top word on both sides, so the sort's top key bit is set
        return V, w1, w2
    if kind == "n=1":
        return 5, np.array([4]), np.array([2])
    if kind == "one_record_repeated":
        return 7, np.full(100_000, 3), np.full(100_000, 6)
    if kind == "two_alternating":
        return 9, np.tile([2, 8], 5000), np.tile([5, 1], 5000)
    if kind == "first_and_last_share":
        V, n = 5000, 2000
        w1, w2 = rng.permutation(np.arange(2, V + 1))[:n], rng.permutation(np.arange(2, V + 1))[:n]
        w1[0] = w1[-1] = 1
        w2[0] = w2[-1] = 1
        return V, w1, w2
    if kind == "self_pairs":
        V, n = 40, 5000
        w1 = rng.integers(1, V + 1, n)
        return V, w1, w1.copy()
    raise ValueError(kind)


STRUCTURES = ["V=1", "V=2", "V=3", "V=65536", "V=65537", "n=1", "one_record_repeated", "two_alternating",
              "first_and_last_share", "self_pairs"]


@pytest.mark.parametrize("kind", STRUCTURES)
def test_record_structure_links_and_epochs(tmp_path, kind):
    V, w1, w2 = _structure(kind)
    rng = np.random.default_rng(52)
    sg = trainer(tmp_path / "c.bin", w1, w2, np.exp(rng.uniform(-2, 7, len(w1))), V, 4)
    words = sg.words.cpu().numpy()
    prev = sg.prev.cpu().numpy()
    assert_bits(words, np.stack([w1 - 1, w2 - 1], 1).astype(np.int32), "words")
    assert_bits(prev, sgo.links(words), "links")
    if kind == "one_record_repeated":
        assert (prev[1:] == np.arange(len(w1) - 1)[:, None]).all()
    if kind == "first_and_last_share":
        assert (prev[-1] == 0).all() and (prev[1:-1] == -1).all()
    if kind.startswith("V=") and V > 2:
        assert (words == V - 1).any(axis=0).all()
    run(sg, 2)


@pytest.mark.parametrize("grid", [1, 2, 3, 37, 0, 20_000])
def test_grid_sizes_give_the_same_bits(tmp_path, grid):
    rng = np.random.default_rng(53)
    V, n = 2000, 50_000
    w1, w2 = zipf_words(rng, V, n)
    sg = trainer(tmp_path / "c.bin", w1, w2, np.exp(rng.uniform(-2, 7, n)), V, 40)
    run(sg, 2, grid=grid)


# ---------------------------------------------------------------------------------------------------------------- E

@pytest.mark.parametrize("n", [1, 2, 8191, 8192, 8193, 8192 * 8192 + 1])
def test_cost_sum_levels(tmp_path, n):
    rng = np.random.default_rng(61)
    V = 1 << 20
    w1, w2 = rng.integers(1, V + 1, n), rng.integers(1, V + 1, n)
    sg = trainer(tmp_path / "c.bin", w1, w2, np.exp(rng.uniform(-2, 7, n)), V, 1)
    del w1, w2
    levels, m = 0, n
    while True:
        m, levels = -(-m // (sgo.SUM_THREADS * sgo.SUM_PER_THREAD)), levels + 1
        if m == 1:
            break
    assert levels == (3 if n > 8192 * 8192 else 2 if n > 8192 else 1)
    run(sg, 1)          # W, gradsq, and the cost equal to sgo.kernel_cost of the oracle's record costs


# ---------------------------------------------------------------------------------------------------------------- F

FLT_MAX = float(np.finfo(np.float32).max)
ROW_SPECIALS = [FLT_MAX * (1 + 2 ** -25), np.nextafter(FLT_MAX * (1 + 2 ** -25), 0), FLT_MAX * (1 - 2 ** -25),
                np.nextafter(FLT_MAX * (1 - 2 ** -25), np.inf), -FLT_MAX * (1 + 2 ** -25), 1e-40, -1e-40, 1e-50, -1e-50,
                math.inf, -math.inf, math.nan, -0.0]


@pytest.mark.parametrize("d", [1, 254])
@pytest.mark.parametrize("V", [1, 2, 99, 100, 101])
def test_rows_edges(tmp_path, V, d):
    rng = np.random.default_rng(71 + V + d)
    sg = trainer(tmp_path / "c.bin", np.array([V, 1]), np.array([1, V]), np.array([2.0, 3.0]), V, d)
    import torch
    W = sg.W.cpu().numpy()
    for spot, v in zip(rng.integers(0, W.size, 3 * len(ROW_SPECIALS)), ROW_SPECIALS * 3):
        W.flat[spot] = v
    W.flat[rng.integers(0, W.size, max(1, W.size // 8))] = FLT_MAX * (1 + 2 ** -25) / 2   # sums that pass FLT_MAX
    sg.W.copy_(torch.from_numpy(W))
    for model in (0, 1, 2):
        for unk in (True, False):
            with np.errstate(over="ignore", invalid="ignore"):     # inf - inf and float32 overflow, as in the kernel
                want = sgo.rows(W, model, unk)
            assert_bits(sg.rows(model, unk).cpu().numpy(), want, "rows V %d d %d model %d unk %d" % (V, d, model, unk))


# ---------------------------------------------------------------------------------------------------------------- G

def _finish(which, keys, agg, V, ctx, dw):
    """Runs glove_cooc_finish_stanford (which = 'stanford', window ctx, distance weighting dw) or
    glove_cooc_finish_sorted (context ctx) on device copies of the aggregates; returns (row, col, count, value)."""
    import torch
    from glove_tensorflow_b200 import _lib
    lib, dev = _lib.lib, torch.device("cuda:0")
    n = len(keys)
    k = torch.from_numpy(keys.view(np.int64)).to(dev)
    a = torch.from_numpy(agg.reshape(-1)).to(dev)
    vc = torch.full((V,), 1000, dtype=torch.int64, device=dev)
    ws = torch.empty(lib.glove_cooc_workspace_bytes(n), dtype=torch.uint8, device=dev)
    dts = (torch.int32, torch.int32, torch.int64, torch.float64, torch.float64, torch.float64, torch.float64)
    out = [torch.empty(n, dtype=t, device=dev) for t in dts]
    got = ctypes.c_int64()
    st = torch.cuda.current_stream().cuda_stream
    if which == "stanford":
        rc = lib.glove_cooc_finish_stanford(k.data_ptr(), a.data_ptr(), n, V, ctx, dw, vc.data_ptr(), 10 ** 6, 7,
                                            ws.data_ptr(), ws.numel(), *[t.data_ptr() for t in out], n,
                                            ctypes.byref(got), st)
    else:
        rc = lib.glove_cooc_finish_sorted(k.data_ptr(), a.data_ptr(), n, V, ctx, 1, vc.data_ptr(), 10 ** 6, 7,
                                          ws.data_ptr(), ws.numel(), *[t.data_ptr() for t in out], n, ctypes.byref(got),
                                          st)
    assert rc == 0, lib.glove_last_error()
    torch.cuda.synchronize()
    assert got.value == n
    return [t[:n].cpu().numpy() for t in out[:4]]


def _numerators(rng):
    big = [2 ** 53 - 1] + [2 ** 53 + i for i in range(1001)] + [int(x) for x in rng.integers(2 ** 53, 2 ** 63, 1000,
                                                                                              dtype=np.uint64)]
    return [int(x) for x in rng.integers(1, 10 ** 6, 100)] + big + [2 ** 63 - 1]


_G_BAD = {}


@pytest.mark.parametrize("which,ctx,dw", [("stanford", w, dw) for w in range(1, 16) for dw in (1, 0)]
                         + [("sorted", c, 1) for c in range(1, 9)])
def test_cooc_finish_value_past_2_53(which, ctx, dw):
    rng = np.random.default_rng(81 + ctx + 100 * dw)
    numer = _numerators(rng)
    V = 100
    vbits = (V + 1 - 1).bit_length()     # csrc/glove_cooc.cu vbits_of(V + 1)
    pairs = rng.choice(V * V, len(numer), replace=False)
    pairs.sort()
    a, b = pairs // V, pairs % V
    keys = ((a.astype(np.uint64) << np.uint64(vbits)) | b.astype(np.uint64))
    assert (np.diff(keys.astype(np.float64)) > 0).all()
    count = rng.integers(1, 10 ** 6, len(numer))
    agg = np.stack([count, np.array(numer, dtype=np.int64)], 1).astype(np.int64)
    row, col, cnt, value = _finish(which, keys, agg, V, ctx, dw)
    unit = math.lcm(*range(1, ctx + 1)) if dw else 1
    want = {(int(x), int(y)): (int(c), m / unit) for x, y, c, m in zip(a, b, count, numer)}
    got = {(int(x), int(y)): (int(c), v) for x, y, c, v in zip(row, col, cnt, value)}
    assert got.keys() == want.keys()
    bad = [(key, got[key][1], want[key][1]) for key in want
           if got[key][0] != want[key][0] or np.float64(got[key][1]).view(np.int64) != np.float64(want[key][1]).view(np.int64)]
    _G_BAD[(which, ctx, dw)] = (len(bad), len(want))
    assert not bad, "%s ctx %d weighting %d: %d of %d values not numer / %d correctly rounded (%d of %d so far), " \
        "first %r" % (which, ctx, dw, len(bad), len(want), unit, sum(x[0] for x in _G_BAD.values()),
                      sum(x[1] for x in _G_BAD.values()), bad[0])
