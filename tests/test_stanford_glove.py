"""CPU checks of Stanford GloVe's trainer: the oracle (oracle/stanford_glove_oracle.c) in glove.c's order against a
literal Python transcription of glove.c's loop, the kernel's order against glove.c's, the seeded initialisation, the
rows of the vectors file, the CLI's defaults and refusals, and the argument errors of the glove_sgd_* entries."""
import ctypes
import math

import numpy as np
import pytest

from oracle import stanford_glove_oracle as sgo


def _fmax(a, b):   # C's fmax / fmin: a NaN operand loses
    return b if a != a else a if b != b else max(a, b)


def _fmin(a, b):
    return b if a != a else a if b != b else min(a, b)


def _check_nan(u):
    return 0.0 if math.isnan(u) or math.isinf(u) else u


def glove_c_epoch(W, G, words, lf, V, d, eta, clip):
    """glove_thread of glove.c with one thread, transcribed statement by statement (W, G: lists of rows)."""
    cost = 0.0
    for (w1, w2), (L, f) in zip(words.tolist(), lf.tolist()):
        l1, l2 = w1, V + w2
        diff = 0.0
        for b in range(d):
            diff += W[l1][b] * W[l2][b]
        diff += W[l1][d] + W[l2][d] - L
        fdiff = f * diff
        if math.isnan(diff) or math.isnan(fdiff) or math.isinf(diff) or math.isinf(fdiff):
            continue
        cost += 0.5 * fdiff * diff
        u1, u2, s1, s2 = [0.0] * d, [0.0] * d, 0.0, 0.0
        for b in range(d):
            temp1 = _fmin(_fmax(fdiff * W[l2][b], -clip), clip) * eta
            temp2 = _fmin(_fmax(fdiff * W[l1][b], -clip), clip) * eta
            u1[b] = temp1 / math.sqrt(G[l1][b])
            u2[b] = temp2 / math.sqrt(G[l2][b])
            s1 += u1[b]
            s2 += u2[b]
            G[l1][b] += temp1 * temp1
            G[l2][b] += temp2 * temp2
        if not math.isnan(s1) and not math.isinf(s1) and not math.isnan(s2) and not math.isinf(s2):
            for b in range(d):
                W[l1][b] -= u1[b]
                W[l2][b] -= u2[b]
        W[l1][d] -= _check_nan(fdiff / math.sqrt(G[l1][d]))
        W[l2][d] -= _check_nan(fdiff / math.sqrt(G[l2][d]))
        fdiff *= fdiff
        G[l1][d] += fdiff
        G[l2][d] += fdiff
    return cost / len(words)


def bin_records(w1, w2, val):
    rec = np.zeros(len(w1), np.dtype([("w1", "<i4"), ("w2", "<i4"), ("val", "<f8")]))
    rec["w1"], rec["w2"], rec["val"] = w1, w2, val
    return rec.tobytes()


def table(seed, V, n, kind="zipf", x_max=100.0):
    rng = np.random.default_rng(seed)
    if kind == "zipf":
        p = 1.0 / np.arange(1, V + 1)
        w1 = rng.choice(V, n, p=p / p.sum()) + 1
        w2 = rng.choice(V, n, p=p / p.sum()) + 1
    elif kind == "one_word":      # one word in every record, on either side
        w1 = np.where(rng.random(n) < 0.5, 3, rng.integers(1, V + 1, n))
        w2 = np.where(w1 == 3, rng.integers(1, V + 1, n), 3)
    else:                         # self pairs and repeated records
        w1 = rng.integers(1, V + 1, n)
        w2 = np.where(rng.random(n) < 0.5, w1, rng.integers(1, V + 1, n))
        rep = rng.random(n) < 0.3
        w1[1:][rep[1:]], w2[1:][rep[1:]] = w1[:-1][rep[1:]], w2[:-1][rep[1:]]
    val = np.exp(rng.uniform(-3, 6, n))        # both sides of x_max
    return sgo.records(bin_records(w1, w2, val), x_max, 0.75)


CASES = [  # (name, seed, V, d, n, kind, eta, clip, W tweak)
    ("plain", 1, 12, 5, 300, "zipf", 0.05, 100.0, None),
    ("clipping", 2, 10, 33, 300, "zipf", 0.5, 0.01, None),
    ("self_and_repeats", 3, 9, 7, 300, "repeats", 0.05, 100.0, None),
    ("one_word", 4, 15, 3, 300, "one_word", 0.1, 1.0, None),
    ("diff_skip", 5, 8, 4, 200, "zipf", 0.05, 100.0, "huge_row"),
    ("update_skip", 6, 8, 4, 200, "zipf", 1e307, 100.0, None),
]


def _start(V, d, tweak, seed):
    W = sgo.init_params(V, d, seed)
    if tweak == "huge_row":
        W[2] = 1e200           # its dot products overflow: those records are skipped
        W[V + 5, :d] = 1e160   # finite but huge: gradsq of the bias overflows, later bias steps are check_nan'ed
    return W, np.ones_like(W)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_oracle_in_glove_order_equals_the_transcription(case):
    _, seed, V, d, n, kind, eta, clip, tweak = case
    words, lf = table(seed, V, n, kind)
    W, G = _start(V, d, tweak, seed)
    Wp, Gp = W.tolist(), G.tolist()
    skipped = 0
    for _ in range(2):
        cost = sgo.epoch(W, G, words, lf, eta, clip, order=0)
        ref = glove_c_epoch(Wp, Gp, words, lf, V, d, eta, clip)
        assert sgo.glove_cost(cost) == ref or (math.isnan(ref) and math.isnan(sgo.glove_cost(cost)))
        skipped += int(np.sum(cost == 0))
        np.testing.assert_array_equal(W, np.array(Wp))
        np.testing.assert_array_equal(G, np.array(Gp))
    if tweak == "huge_row":
        assert skipped > 0 and np.isinf(G).any()
    if kind == "one_word":
        assert (words == 2).any(axis=1).all()
    if eta > 1e300:
        assert np.isinf(G).any()


def test_update_skip_leaves_vectors_but_moves_biases_and_gradsq():
    words, lf = table(6, 8, 50, "zipf")
    W, G = _start(8, 4, None, 6)
    W0 = W.copy()
    sgo.epoch(W, G, words, lf, float("inf"), 100.0, order=1)   # every step is +-inf or NaN: no vector update
    np.testing.assert_array_equal(W[:, :4], W0[:, :4])
    assert (W[:, 4] != W0[:, 4]).any() and np.isinf(G[:, :4]).any()


@pytest.mark.parametrize("d", [2, 31, 33, 50])
def test_kernel_order_stays_within_1e12_of_glove_order(d):
    V = 40
    words, lf = table(10 + d, V, 4000, "zipf")
    A, GA = sgo.init_params(V, d, 3), np.ones((2 * V, d + 1))
    B, GB = A.copy(), GA.copy()
    for _ in range(3):
        ca = sgo.epoch(A, GA, words, lf, order=0)
        cb = sgo.epoch(B, GB, words, lf, order=1)
    assert (A != B).any() or d <= 2                # the orders differ in the last bits from d = 3 on
    scale = np.abs(A).max()
    assert np.abs(A - B).max() <= 1e-12 * scale
    assert np.abs(GA - GB).max() <= 1e-12 * np.abs(GA).max()
    assert abs(sgo.glove_cost(ca) - sgo.kernel_cost(cb)) <= 1e-12 * sgo.glove_cost(ca)


def test_init_generator_restated():
    M = (1 << 64) - 1

    def mix(z):
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M
        return z ^ (z >> 31)

    for V, d, seed in ((3, 2, 0), (5, 7, 1), (4, 50, 2 ** 64 - 1)):
        W = sgo.init_params(V, d, seed)
        assert W.shape == (2 * V, d + 1)
        for i in (0, 1, d, d + 1, 2 * V * (d + 1) - 1):
            z = mix((seed * 0xD1B54A32D192ED03 + i * 0x9E3779B97F4A7C15) & M)
            assert W.flat[i] == ((z >> 11) * 2.0 ** -53 - 0.5) / d
        assert np.abs(W).max() <= 0.5 / d and len(np.unique(W)) == W.size


def test_kernel_cost_sum_shape():
    rng = np.random.default_rng(0)
    for n in (1, 255, 8192, 8193, 70000):
        c = rng.random(n)
        got = sgo.kernel_cost(c)
        assert abs(got - c.sum() / n) <= 1e-13
    c = np.arange(1, 8194, dtype=np.float64)
    parts = [sum(c[t:8192:256].tolist(), 0.0) for t in range(256)]   # thread t, ascending
    while len(parts) > 1:
        parts = [parts[i] + parts[i + len(parts) // 2] for i in range(len(parts) // 2)]
    chunk0 = parts[0]
    assert sgo.kernel_cost(c) == (chunk0 + (0.0 + c[8192])) / 8193


def test_rows_and_unk_follow_glove_c():
    V, d = 130, 3
    W = sgo.init_params(V, d, 9)
    m = 100
    vec = [0.0] * (d + 1)
    ctx = [0.0] * (d + 1)
    for a in range(V - m, V):
        for b in range(d + 1):
            vec[b] += W[a][b] / m
            ctx[b] += W[V + a][b] / m
    r0, r1, r2 = sgo.rows(W, 0), sgo.rows(W, 1), sgo.rows(W, 2)
    assert r0.shape == (V + 1, 2 * d + 2) and r1.shape == r2.shape == (V + 1, d)
    np.testing.assert_array_equal(r0[:V], np.hstack([W[:V], W[V:]]).astype(np.float32))
    np.testing.assert_array_equal(r1[:V], W[:V, :d].astype(np.float32))
    np.testing.assert_array_equal(r2[:V], (W[:V, :d] + W[V:, :d]).astype(np.float32))
    np.testing.assert_array_equal(r0[V], np.float32(vec + ctx))
    np.testing.assert_array_equal(r1[V], np.float32(vec[:d]))
    np.testing.assert_array_equal(r2[V], np.float32([vec[b] + ctx[b] for b in range(d)]))
    assert sgo.rows(W, 2, unk=False).shape == (V, d)
    small = sgo.init_params(4, 2, 1)     # V < 100: the mean of all V rows
    np.testing.assert_array_equal(sgo.rows(small, 1)[4], np.float32((((0.0 + small[0, :2] / 4) + small[1, :2] / 4)
                                                                     + small[2, :2] / 4) + small[3, :2] / 4))


def test_links_and_chain():
    words = np.array([[0, 1], [0, 2], [1, 1], [0, 1], [2, 0]], np.int32)
    prev = sgo.links(words)
    np.testing.assert_array_equal(prev, [[-1, -1], [0, -1], [-1, 0], [1, 2], [-1, -1]])
    assert sgo.chain(prev) == 3
    with pytest.raises(ValueError):
        sgo.chain(np.array([[1, -1], [-1, -1]], np.int32))


def test_cli_defaults_and_refusals(tmp_path):
    from glove_tensorflow_b200 import stanford_glove as sg
    a = sg.parser().parse_args(["--input-file", "x", "--vocab-file", "v"])
    assert (a.vector_size, a.iter, a.eta, a.alpha, a.x_max, a.grad_clip, a.model, a.binary) == \
        (50, 25, 0.05, 0.75, 100.0, 100.0, 2, 0)
    assert a.write_header is False and a.unk_vector is True and a.save_file == "vectors"
    assert a.save_gradsq is False and a.gradsq_file == "gradsq" and a.init_param_file is None
    assert {k: getattr(a, k) for k in sg.DEFAULTS} == sg.DEFAULTS
    base = ["--input-file", "x", "--vocab-file", "v"]
    for bad in (["--model", "3"], ["--binary", "-1"], ["--vector-size", "0"], ["--vector-size", "513"], ["--iter", "-1"],
                ["--x-max", "0"], ["--eta", "nan"], ["--vector-size", "300", "--model", "0"], ["--vector-size", "1"],
                ["--threads", "8"], ["--vector-size", "x"]):
        with pytest.raises(SystemExit):
            sg.main(base + bad)
    v = tmp_path / "vocab.txt"
    v.write_text("the 5\n<unk> 3\n")
    with pytest.raises(ValueError, match="<unk>"):
        sg.train(str(tmp_path / "none.bin"), str(v))


def test_sgd_entries_refuse_bad_arguments_without_a_gpu():
    from glove_tensorflow_b200 import _lib
    lib, E = _lib.lib, _lib.EINVAL
    f = ctypes.c_void_p(1 << 20)
    odd = ctypes.c_void_p((1 << 20) + 8)
    assert lib.glove_sgd_parse(None, 4, 0, 10, 100.0, 0.75, f, f, f, None) == E
    assert lib.glove_sgd_parse(f, 4, 0, 10, 100.0, 0.75, None, f, f, None) == E
    assert lib.glove_sgd_parse(odd, 4, 0, 10, 100.0, 0.75, f, f, f, None) == E
    assert lib.glove_sgd_parse(f, 4, 0, 10, 100.0, 0.75, f, odd, f, None) == E
    assert lib.glove_sgd_parse(f, 0, 0, 10, 100.0, 0.75, f, f, f, None) == E
    assert lib.glove_sgd_parse(f, 4, -1, 10, 100.0, 0.75, f, f, f, None) == E
    assert lib.glove_sgd_parse(f, 4, 0, 0, 100.0, 0.75, f, f, f, None) == E
    assert lib.glove_sgd_parse(f, 4, 0, 10, 0.0, 0.75, f, f, f, None) == E
    assert lib.glove_sgd_parse(f, 4, 0, 10, 100.0, float("nan"), f, f, f, None) == E
    assert lib.glove_sgd_links_workspace_bytes(0) == 0 and lib.glove_sgd_links_workspace_bytes(1 << 31) == 0
    ws = lib.glove_sgd_links_workspace_bytes(100)
    assert ws >= 1600
    assert lib.glove_sgd_links(None, 100, 10, f, f, ws, None) == E
    assert lib.glove_sgd_links(f, 0, 10, f, f, ws, None) == E
    assert lib.glove_sgd_links(f, 100, 0, f, f, ws, None) == E
    assert lib.glove_sgd_links(f, 100, 10, f, f, ws - 1, None) == E
    assert lib.glove_sgd_init(None, 10, 4, 1, None) == E
    assert lib.glove_sgd_init(f, 0, 4, 1, None) == E
    assert lib.glove_sgd_init(f, 10, 0, 1, None) == E
    es = lib.glove_sgd_epoch_workspace_bytes(100)
    assert es >= 800 and lib.glove_sgd_epoch_workspace_bytes(0) == 0
    ok = (f, f, 10, 4, f, f, f, 100, 0.05, 100.0, 1, f, 0, f, es, f, None)

    def epoch(**kw):
        a = list(ok)
        for i, v in kw.items():
            a[int(i[1:])] = v
        return lib.glove_sgd_epoch(*a)

    assert epoch(a0=None) == E and epoch(a11=None) == E and epoch(a15=None) == E
    assert epoch(a2=0) == E and epoch(a3=0) == E and epoch(a3=513) == E and epoch(a7=0) == E and epoch(a7=1 << 31) == E
    assert epoch(a8=float("nan")) == E and epoch(a9=float("nan")) == E
    assert epoch(a10=0) == E and epoch(a12=-1) == E and epoch(a14=es - 1) == E
    assert epoch(a5=ctypes.c_void_p((1 << 20) + 8)) == E and epoch(a4=ctypes.c_void_p((1 << 20) + 4)) == E
    assert lib.glove_sgd_rows(None, 10, 4, 2, 1, f, None) == E
    assert lib.glove_sgd_rows(f, 10, 4, 3, 1, f, None) == E
    assert lib.glove_sgd_rows(f, 10, 4, 2, 2, f, None) == E
    assert lib.glove_sgd_rows(f, 0, 4, 2, 1, f, None) == E
    assert b"glove_sgd_rows" in lib.glove_last_error()
