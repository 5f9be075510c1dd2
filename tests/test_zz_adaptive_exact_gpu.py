"""Adaptive sampling against an exact host model (tests/adaptive_model.py), bit for bit.

The other adaptive tests compare the GPU with itself (an adaptive pixel with vk_render, a batch with its frames, a
tightened session with a fresh one), so a wrong rule would pass them all.  Here the rule, the error map, the readout, the
squares of real samples and the whole pass loop are checked against a plain restatement on the host: crafted states
through vk_adaptive_import (every edge of the rule and the readout), real renders against the model's prediction from
fixed-spp states, and each sample's fixed-point square.  The model's own tests run without a GPU."""
import decimal
from fractions import Fraction

import numpy as np
import pytest

import adaptive_model as am

gpu = pytest.mark.gpu

# -------------------------------------------------------------------------------------------------------------------
# The model (no GPU)
# -------------------------------------------------------------------------------------------------------------------

# n = 2, S = 25 * 2^30, Q = 337 * 2^32: m = 12.5, q = 168.5, se = 3.5 and e = 128 (sqrt(16) - sqrt(9)) = 128 exactly
EXACT_128 = (2, (25 << 30, 2 << 30, 2 << 30), (337 << 32, 2 << 32, 2 << 32))
# n = 2 and an odd 41-bit S: m = 758.53.. and m^2 is not a double; Q = fl(m * m) * 2^33 with fl rounding up, so
# q - m^2 is 0 when m * m is rounded on its own and the (positive) rounding error of m^2 when it is fused
FUSED_S = 1628925508549
FUSED_Q = int(Fraction((FUSED_S * 2.0 ** -30 / 2) ** 2) * 2 ** 33)
FUSED = (2, (FUSED_S, 0, 0), (FUSED_Q, 0, 0))


def decimal_error(n, S, Q):
    """The header's formula for e in 50-digit decimal arithmetic."""
    D = decimal.Decimal
    with decimal.localcontext() as c:
        c.prec = 50
        e = D(0)
        for s, q in zip(S, Q):
            m = D(s) / D(2 ** 30) / n
            var = max(D(q) / D(2 ** 32) / n - m * m, D(0)) / (n - 1)
            se = var.sqrt()
            e = max(e, 128 * (max(m + se, D(0)).sqrt() - max(m - se, D(0)).sqrt()))
        return e


def one(state):
    n, S, Q = state
    return np.array([S], dtype=np.int64), np.array([Q], dtype=np.uint64), np.array([n], dtype=np.uint32)


KNOWN = [
    (4, (3 << 30, 1 << 29, 5 << 30), (4 << 32, 1 << 30, 9 << 32)),
    (17, (-(7 << 30), 123456789012, 0), (95 << 32, 987654321098765, 3 << 32)),
    (64, (1000 << 30, 64 << 30, 3 << 28), (20000 << 32, 70 << 32, 1 << 32)),
    (45, (2 ** 53 + 1, -(2 ** 53 + 1), 2 ** 45), (2 ** 63 + 12345, 2 ** 63, 2 ** 60)),
    (3, (7, -3, 1 << 20), (1 << 40, 5, 1 << 12)),  # m - se < 0 in every channel
]


@pytest.mark.parametrize("state", KNOWN + [EXACT_128])
def test_model_error_matches_the_formula_in_decimal(state):
    got = am.rule_error(*one(state))[0]
    want = decimal_error(*state)
    # a chain of about ten double operations, none of them cancelling much in these states
    assert abs(decimal.Decimal(got) - want) <= decimal.Decimal(1e-13) * max(want, decimal.Decimal(1e-300)), (got, want)


def test_model_error_exact_at_128():
    assert am.rule_error(*one(EXACT_128))[0] == 128.0
    assert am.error_map(*one(EXACT_128))[0] == np.float32(128.0)


def test_model_fuses_q_minus_m_squared():
    m = FUSED_S * 2.0 ** -30 / 2
    assert m > 724 and FUSED_S % 2 == 1 and FUSED_S.bit_length() == 41
    assert Fraction(m * m) > Fraction(m) ** 2  # fl(m * m) rounded up
    assert FUSED_Q == Fraction(m * m) * 2 ** 33 and FUSED_Q < 2 ** 53  # q = fl(m * m) exactly
    fused, unfused = am.rule_error(*one(FUSED))[0], am.rule_error(*one(FUSED), fused=False)[0]
    assert unfused == 0.0 and 2.1e-5 < fused < 2.3e-5
    # the fused value: q - m^2 exactly, rounded once
    v = float(Fraction(FUSED_Q * 2.0 ** -32 / 2) - Fraction(m) ** 2)
    se = np.sqrt(v / 1.0)
    assert fused == (np.sqrt(m + se) - np.sqrt(m - se)) * 128.0


def test_model_fma_against_fractions():
    rng = np.random.default_rng(3)
    m = rng.uniform(-2000, 2000, 500) * 2.0 ** rng.integers(-20, 5, 500)
    q = m * m * rng.uniform(0.999, 1.001, 500)
    got = am.fused_q_minus_m2(m, q)
    want = [float(Fraction(b) - Fraction(a) ** 2) for a, b in zip(m.tolist(), q.tolist())]
    assert np.array_equal(got, np.array(want))


def test_model_int_to_double_rounds_to_nearest():
    vals = [0, 1, -1, 2 ** 53 + 1, -(2 ** 53 + 1), 2 ** 53 + 3, 2 ** 62 - 1, -(2 ** 62) + 1, 2 ** 63 - 1, -(2 ** 63),
            2 ** 54 + 2, 2 ** 54 + 6, 12345678901234567]
    assert am.int64_to_double(np.array(vals, dtype=np.int64)).tolist() == [float(v) for v in vals]
    uvals = [0, 2 ** 64 - 1, 2 ** 64 - 2 ** 11, 2 ** 64 - 2 ** 11 - 1, 2 ** 63 + 2 ** 10, 2 ** 63 + 2 ** 10 + 1, 2 ** 53 + 1]
    assert am.uint64_to_double(np.array(uvals, dtype=np.uint64)).tolist() == [float(v) for v in uvals]


def test_model_below_two_samples_and_stops():
    S = np.zeros((3, 3), dtype=np.int64)
    Q = np.zeros((3, 3), dtype=np.uint64)
    e = am.rule_error(S, Q, np.array([0, 1, 2]))
    assert np.isposinf(e[0]) and np.isposinf(e[1]) and e[2] == 0.0
    n = np.array([0, 1, 2, 2, 8, 9])
    e = np.array([np.inf, np.inf, 1.0, 1.5, 1.0, 5.0])
    assert am.stops(e, n, (9, 0, 1.0)).tolist() == [False, False, True, False, True, True]
    assert am.stops(e, n, (9, 8, 1.0)).tolist() == [False, False, False, False, True, True]
    assert am.stops(e, n, (9, 0, 0.0)).tolist() == [False] * 5 + [True]
    assert am.stops(np.array([128.0]), np.array([2]), (9, 0, 128.0))[0]
    assert not am.stops(np.array([128.0]), np.array([2]), (9, 0, np.nextafter(np.float32(128), np.float32(0))))[0]


def test_model_means_on_edges():
    S = np.array([0, 1, -1, 2 ** 53 + 1, -(2 ** 53 + 1), 2 ** 62 - 1, -(2 ** 62) + 1, 3 << 30, 45 * 800 << 30],
                 dtype=np.int64).reshape(3, 3)
    n = np.array([1, 45, 3], dtype=np.uint32)
    want = (np.array([float(v) for v in S.reshape(-1).tolist()]).reshape(3, 3) * 2.0 ** -30).astype(np.float32) \
        / n.astype(np.float32)[:, None]
    assert np.array_equal(am.means(S, n), want)
    z = am.means(np.zeros((1, 3), dtype=np.int64), np.array([0]))
    assert np.all(np.isnan(z))


def test_model_square_units():
    d = np.array([0, 1 << 30, -(1 << 30), 3 << 29, 255 << 30, 256 << 30, -(800 << 30), 1 << 23, (1 << 23) + 1, 12345678])
    want = []
    for x in d.tolist():
        c = Fraction(min(abs(x), 255 << 30), 1 << 30)
        v = c * c * 2 ** 32
        want.append(round(v))  # Python's round of a Fraction: half to even
    assert am.square_units(d).tolist() == want
    assert am.square_units(np.array([800 << 30]))[0] == 65025 << 32


def test_model_predict_three_levels():
    # M = 2, cap 5: the grid is 2, 4, 5.  Pixel 0 is constant (stops at 2), pixel 1 is noisy until 4, pixel 2 until the
    # cap, pixel 3 is below the floor at 2 and stops at 4.
    def st(vals):  # per pixel the samples of channel R so far; G and B zero
        S = np.array([[sum(v) << 30, 0, 0] for v in vals], dtype=np.int64)
        Q = np.array([[sum(x * x for x in v) << 32, 0, 0] for v in vals], dtype=np.uint64)
        return S, Q
    samples = [[1] * 5, [9, 1, 5, 5, 5], [9, 1, 1, 9, 5], [1, 1, 1, 1, 1]]
    states = {b: st([s[:b] for s in samples]) for b in (2, 4, 5)}
    floor = [0, 0, 0, 4]
    n = np.zeros(4, dtype=np.uint32)
    for p in range(4):
        n_p, _, _ = am.predict({b: (v[0][p:p + 1], v[1][p:p + 1]) for b, v in states.items()}, (5, floor[p], 100.0), 2)
        n[p] = n_p[0]
    assert n.tolist() == [2, 4, 5, 4]
    got = am.predict(states, (5, 0, 100.0), 2)
    assert got[0].tolist() == [2, 4, 5, 2]
    assert np.array_equal(got[1][1], states[4][0][1]) and np.array_equal(got[2][2], states[5][1][2])
    # from an imported start: pixel 0 at 4 with pixel 1's state, the rest fresh (count 0)
    start = (np.array([4, 0, 0, 0]), states[4][0].copy(), states[4][1].copy())
    start[1][1:] = 0
    start[2][1:] = 0
    start[1][0], start[2][0] = states[4][0][1], states[4][1][1]
    got = am.predict(states, (5, 0, 100.0), 2, start=start)
    assert got[0].tolist() == [4, 4, 5, 2]


# -------------------------------------------------------------------------------------------------------------------
# The GPU against the model
# -------------------------------------------------------------------------------------------------------------------

_SCENES = {}


def scene_and_cams(vb, name, param=0, k=1):
    """A scene and k cameras: its own camera, then ones moved sideways (as tests/test_zz_adaptive_session_gpu.py)."""
    key = (name, param)
    if key not in _SCENES:
        s = vb.Scene(name, seed=1, param=param)
        base = s.next_camera()
        cams = [base]
        for f in range(1, 3):
            eye = [base.origin[i] + 0.3 * f * base.u[i] for i in range(3)]
            cams.append(vb.camera_new(eye, [eye[i] - base.w[i] for i in range(3)], list(base.v), 40.0, 1.0, 0.0, 10.0,
                                      base.time0, base.time1))
        _SCENES[key] = (s, cams)
    s, cams = _SCENES[key]
    return s, (cams[0] if k == 1 else cams[:k])


def flags_of(vb, flags):
    return vb.VK_FLAG_LEGACY_SCATTER | vb.VK_FLAG_SKY_BACKGROUND if flags == "legacy_sky" else 0


def fixed_states(ctx, cams, p, M, counts):
    """(sums, squares) after samples [0, b) for each b: a fresh session with max_error 0 capped at b."""
    out = {}
    for b in counts:
        s = ctx.adaptive_session(cams, p, M)
        s.refine(0.0, spp=b)
        sums, sq, n, _ = s.export()
        assert np.all(n == b)
        out[b] = (sums, sq)
        s.close()
    return out


def assert_reads_match_model(vb, sess, sums, squares, counts):
    """read() and read_rgb8() against the model: means, rgb8, counts and error map bit for bit (NaN, inf included); the
    rgb8 image's counts and errors are each frame's rows top-down."""
    rgb, n1, err = sess.read()
    assert np.array_equal(n1, counts)
    want = am.means(sums, counts)
    assert np.array_equal(np.isnan(rgb), np.isnan(want))
    assert np.array_equal(rgb, want, equal_nan=True), int(np.sum(rgb != want))
    want_err = am.error_map(sums, squares, counts)
    assert np.array_equal(err, want_err), int(np.sum(err != want_err))
    rgb8, n8, err8 = sess.read_rgb8()
    assert np.array_equal(rgb8, am.rgb8(vb, sums, counts))
    assert np.array_equal(n8, counts[..., ::-1, :]) and np.array_equal(err8, want_err[..., ::-1, :])


def edge_state(M, C, shape, seed):
    """A state (counts, sums, squares) of the given (K, H, W) shape built pixel by pixel: a table of edges at scattered
    pixels, random states elsewhere.  Counts are on the pass grid (multiples of M) or the cap C.  Returns the state and
    the index of the pixel whose e is exactly 128."""
    rng = np.random.default_rng(seed)
    P = int(np.prod(shape))
    on_grid = [b for b in range(0, C + 1, M)] + ([C] if C % M else [])
    n = rng.choice(on_grid, P).astype(np.uint32)
    n[n == 0] = M  # (count 0 only where the table puts it)
    nd = n.astype(np.int64)[:, None]
    mean = rng.choice([0.0, 0.02, 0.5, 3.0, 40.0], (P, 3)) * rng.uniform(0.0, 1.0, (P, 3))
    S = np.round(mean * nd * 2 ** 30).astype(np.int64)
    var = rng.choice([0.0, 0.001, 0.3, 20.0], (P, 3)) * rng.uniform(0.0, 1.0, (P, 3))
    Q = np.round((var + mean ** 2) * nd * 2 ** 32).astype(np.uint64)
    big = 65025 << 32
    rows = [
        (0, (0, 0, 0), (0, 0, 0)),                                               # no samples: NaN mean, rgb8 0, e inf
        EXACT_128, FUSED,                                                        # the threshold and the contraction
        (M, (3 << 28, 1 << 30, 5 << 29), (1 << 31, 1 << 32, 7 << 31)),
        (C, (-(3 << 30) * C, -(1 << 20), 5 << 30), (9 << 32, 1 << 12, 30 << 32)),  # negative sums
        (2, (0, 0, 0), (5 << 32, 1, 0)),                                         # zero sums
        (C, (2 ** 53 + 1, -(2 ** 53 + 1), 2 ** 53 + 3), (2 ** 63 + 1, 2 ** 60, 2 ** 62)),
        (C, (2 ** 62 - 1, -(2 ** 62) + 1, 2 ** 62 - 98765), (2 ** 64 - 1, 2 ** 64 - 2 ** 11, 2 ** 64 - 2 ** 11 - 1)),
        (2, (2 ** 62 - 5, -(2 ** 62) + 7, 1 << 30), (0, 0, 0)),                  # q < m^2 with no squares at all
        (C, ((800 << 30) * C, (600 << 30) * C, (100 << 30) * C), (big * C, big * C, (10000 << 32) * C)),  # clamped
        (M, (1 << 30, 2 << 30, 3 << 30), (2 ** 64 - 1, 2 ** 64 - 2 ** 12 + 1, 2 ** 64 - 3)),  # squares near 2^64
        (C, ((3 << 28) * C, (5 << 27) * C, 0), ((9 << 24) * C, (25 << 22) * C, 0)),  # constant samples: variance 0
        (2 * M if 2 * M <= C else C, (1 << 26, 3, -(1 << 27)), (1 << 38, 1 << 36, 1 << 37)),  # m - se < 0
        (2, (1 << 30, 1 << 30, 1 << 30), (40 << 32, 1 << 31, 1 << 31)),         # the largest e in R
        (2, (1 << 30, 1 << 30, 1 << 30), (1 << 31, 40 << 32, 1 << 31)),         # .. in G
        (2, (1 << 30, 1 << 30, 1 << 30), (1 << 31, 1 << 31, 40 << 32)),         # .. in B
    ]
    if M == 1:
        rows.append((1, (3 << 29, -(1 << 28), 7 << 30), (9 << 30, 1 << 24, 49 << 32)))  # one sample: no error
    rows = [r for r in rows if r[0] in on_grid]
    at = rng.permutation(P)[:len(rows)]
    for p, (c, s, q) in zip(at, rows):
        n[p], S[p], Q[p] = c, s, q
    i128 = int(at[[r is EXACT_128 for r in rows].index(True)])
    sh = tuple(shape)
    return (n.reshape(sh), S.reshape(sh + (3,)), Q.reshape(sh + (3,))), i128


def f32_around(e):
    """The float32 values just above (or at) and just below the double e."""
    f = np.float32(e)
    up = f if float(f) >= e else np.nextafter(f, np.float32(np.inf))
    down = np.nextafter(up, np.float32(0))
    return float(up), float(down)


@gpu
@pytest.mark.parametrize("M", [1, 2])
def test_crafted_states_rule_and_readout_bit_for_bit(vb, ctx, M):
    scene, cams = scene_and_cams(vb, "cornell_box", 0, 3)
    ctx.upload(scene)
    C, W, H, K = 9, 37, 23, 3  # (37 * 23 * 3 pixels: neither 256 nor 32 divides them; C is off the grid of M = 2)
    p = vb.render_params(W, H, C, 30, seed=11, flags=vb.VK_FLAG_STRICT_MATH)
    (n0, S0, Q0), i128 = edge_state(M, C, (K, H, W), seed=M)
    reached = (C, 0, 1e9)
    sess = ctx.adaptive_session(cams, p, M)
    sess.import_(S0, Q0, n0, reached)
    assert_reads_match_model(vb, sess, S0, Q0, n0)

    # the fixed states, and from them the state every pixel would have after samples [n0, b) rendered on top of its own
    counts = am.grid(M, C)
    fixed = fixed_states(ctx, cams, p, M, counts)
    fixed[0] = (np.zeros_like(S0), np.zeros_like(Q0))
    base_S = np.zeros_like(S0)
    base_Q = np.zeros_like(Q0)
    for b, (fs, fq) in fixed.items():
        base_S[n0 == b], base_Q[n0 == b] = fs[n0 == b], fq[n0 == b]
    states = {b: (S0 + (fixed[b][0] - base_S), Q0 + (fixed[b][1] - base_Q)) for b in counts}  # (squares wrap mod 2^64)

    e0 = am.rule_error(S0, Q0, n0)
    flat_e = e0.reshape(-1)
    assert flat_e[i128] == 128.0
    cand = np.flatnonzero((n0.reshape(-1) >= 2) & (n0.reshape(-1) < C) & np.isfinite(flat_e) & (flat_e > 0.05)
                          & (flat_e.astype(np.float32).astype(np.float64) != flat_e))
    ip = int(cand[0])
    up, down = f32_around(flat_e[ip])
    below128 = float(np.nextafter(np.float32(128.0), np.float32(0)))
    finite = flat_e[np.isfinite(flat_e) & (flat_e > 0)]
    Es = [128.0, below128, up, down, float(np.quantile(finite, 0.3)), float(np.quantile(finite, 0.7)), 0.0]
    floors = [0, 2, 4]
    for E in Es:
        for floor in floors:
            T = (C, floor, E)
            sess.import_(S0, Q0, n0, reached)  # (a target may only tighten the one reached)
            st = sess.refine(E, spp=C, min_spp=floor)
            S1, Q1, n1, _ = sess.export()
            stop0 = am.stops(e0, n0, T)
            assert np.array_equal(n1 == n0, stop0), (T, int(np.sum((n1 == n0) != stop0)))  # k_adaptive_levels
            if floor <= 2:
                assert stop0.reshape(-1)[i128] == (E >= 128.0), T
                if E in (up, down):
                    assert stop0.reshape(-1)[ip] == (E == up), T
            n_pred, S_pred, Q_pred = am.predict(states, T, M, start=(n0, S0, Q0))
            assert np.array_equal(n1, n_pred), (T, int(np.sum(n1 != n_pred)))
            assert np.array_equal(S1, S_pred) and np.array_equal(Q1, Q_pred), T
            assert st.paths == int((n1.astype(np.int64) - n0).sum())
            if floor == 0:
                assert_reads_match_model(vb, sess, S1, Q1, n1)
    sess.close()


CASES = [("cornell_box", 0, 0), ("cornell_smoke", 0, 0), ("final_scene", 0, 0), ("random_spheres_cover", 0, "legacy_sky"),
         ("stress_spheres", 300, 0), ("furnace_demo", 4, 0)]


@gpu
@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("strict", [False, True], ids=["render", "strict"])
@pytest.mark.parametrize("variant", ["AUTO", "WARPQ", "STEPQ", "MEGAKERNEL"])
@pytest.mark.parametrize("name,param,flags", CASES)
def test_adaptive_renders_equal_the_model_prediction(vb, ctx, name, param, flags, variant, strict, k):
    scene, cams = scene_and_cams(vb, name, param, k)
    ctx.upload(scene)
    M, C = 8, 45
    f = flags_of(vb, flags) | (vb.VK_FLAG_STRICT_MATH if strict else 0)
    p = vb.render_params(61, 37, C, 30, seed=5, variant=getattr(vb, "VK_VARIANT_" + variant), flags=f)
    counts = am.grid(M, C)
    fixed = fixed_states(ctx, cams, p, M, counts)
    errors = {b: am.rule_error(*fixed[b], np.full(fixed[b][0].shape[:-1], b)) for b in counts}
    finite = errors[M][np.isfinite(errors[M])]
    Es = [float(np.float32(np.quantile(finite, q))) for q in (0.3, 0.5, 0.8)]
    Es = [E if E > 0 else 0.01 for E in Es]
    seen = set()
    for E in Es:
        for floor in (0, 24):
            T = (C, floor, E)
            want = am.predict(fixed, T, M, errors=errors)
            s = ctx.adaptive_session(cams, p, M)
            s.refine(E, min_spp=floor)
            S1, Q1, n1, _ = s.export()
            assert np.array_equal(n1, want[0]), (T, int(np.sum(n1 != want[0])))
            assert np.array_equal(S1, want[1]) and np.array_equal(Q1, want[2]), T
            assert_reads_match_model(vb, s, S1, Q1, n1)
            seen |= set(np.unique(n1).tolist())
            if floor == 0:  # the one-shot calls
                rgb, _, _ = s.read()
                rgb8, n8, _ = s.read_rgb8()
                if k == 1:
                    w, wn, _ = ctx.render_adaptive(cams, p, M, E)
                    w8, wn8, _ = ctx.render_adaptive_rgb8(cams, p, M, E)
                else:
                    w, wn, _ = ctx.render_frames_adaptive(cams, p, M, E)
                    w8, wn8, _ = ctx.render_frames_adaptive_rgb8(cams, p, M, E)
                assert np.array_equal(wn, n1) and np.array_equal(w, rgb, equal_nan=True)
                assert np.array_equal(wn8, n8) and np.array_equal(w8, rgb8)
            s.close()
    assert len(seen) >= (2 if name == "furnace_demo" else 3), sorted(seen)  # (the furnace's room stops at once: e = 0)
    # a tightening sequence, each step against the model
    s = ctx.adaptive_session(cams, p, M)
    for E, floor in ((8.0, 0), (4.0, 0), (2.0, 0), (2.0, 24)):
        s.refine(E, min_spp=floor)
        S1, Q1, n1, _ = s.export()
        want = am.predict(fixed, (C, floor, E), M, errors=errors)
        assert np.array_equal(n1, want[0]) and np.array_equal(S1, want[1]) and np.array_equal(Q1, want[2]), (E, floor)
    s.close()


@gpu
@pytest.mark.parametrize("strict", [False, True], ids=["render", "strict"])
@pytest.mark.parametrize("name,param,flags", [("final_scene", 0, 0), ("cornell_smoke", 0, 0),
                                              ("random_spheres_cover", 0, "legacy_sky"), ("furnace_demo", 4, 0)])
def test_squares_of_real_samples(vb, ctx, name, param, flags, strict):
    scene, cam = scene_and_cams(vb, name, param)
    ctx.upload(scene)
    f = flags_of(vb, flags) | (vb.VK_FLAG_STRICT_MATH if strict else 0)
    p = vb.render_params(32, 18, 24, 30, seed=9, flags=f)
    s = ctx.adaptive_session(cam, p, 1)
    prev_S, prev_Q, _, _ = s.export()
    dS, dQ = [], []
    for b in range(1, 25):  # one sample per step: consecutive exports differ by one sample of every pixel
        s.refine(0.0, spp=b)
        S, Q, n, _ = s.export()
        assert np.all(n == b)
        dS.append(S - prev_S)
        dQ.append(Q - prev_Q)
        prev_S, prev_Q = S, Q
    s.close()
    dS, dQ = np.stack(dS).reshape(-1), np.stack(dQ).reshape(-1)
    want = am.square_units(dS)
    exact = np.abs(dS) >= 1 << 23  # |L| >= 2^-7: dS / 2^30 is L itself
    assert np.array_equal(dQ[exact], want[exact]), int(np.sum(dQ[exact] != want[exact]))
    diff = dQ[~exact].astype(np.int64) - want[~exact].astype(np.int64)
    assert np.all(np.abs(diff) <= 1)  # 4 |L| 2^32 2^-31 < 1 for |L| < 2^-7
    assert np.all(dQ[dS == 0] == 0)
    assert exact.any()
    if name == "furnace_demo":  # the room's samples, (800, 600, 400), clamp: 255^2 * 2^32 units each
        clamped = np.abs(dS) > 255 << 30
        assert clamped.mean() > 0.3 and np.all(dQ[clamped] == 65025 << 32)
        # the sphere's: cosine-sampled directions weigh 2 x albedo, so R = 800 and B = 600 clamp too, light-sampled ones
        # far less and stay below the clamp
        assert np.any((dS != 0) & (np.abs(dS) < 255 << 30))
