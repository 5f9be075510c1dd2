"""A host model of adaptive sampling's integer state and of every operation the library applies to it (numpy and Python
integers, no GPU): the stopping rule's error e, the error map, the means and the squares of one sample, bit for bit as
the device computes them, and the whole pass loop run from fixed states.

The rule's operation sequence is stated in include/vecchio_gpu.h (vk_render_adaptive) and DESIGN.md (section 7,
"Adaptive sampling"); the device code is adaptive_error / adaptive_stop in vecchio_b200/csrc/vk_api.cu.  Per channel of a
pixel with n >= 2 samples, sum S (int64, 2^30 units per 1.0) and squares Q (uint64, 2^32 units per 1.0), every step an
IEEE double operation rounded to nearest:

    m = (double)S * 2^-30 / n,   q = (double)Q * 2^-32 / n,   v = fma(-m, m, q)   (q - m^2, rounded once),
    se = sqrt(max(v, 0) / (n - 1)),   e_c = (sqrt(max(m + se, 0)) - sqrt(max(m - se, 0))) * 128,

and e = max(0, e_R, e_G, e_B), compared as e <= (double)max_error.  numpy's float64 operations are correctly rounded, so
they are the device's; the fused q - m^2 is computed exactly in Python integers and rounded once."""
import numpy as np

ACC_UNITS = 1 << 30  # sums: 2^30 units per 1.0
SQ_UNITS = 1 << 32   # squares: 2^32 units per 1.0
SQ_CLAMP = 255       # each channel of a sample is clamped to 255 before it is squared


def int64_to_double(a):
    """(double)(long long) a, rounded to nearest: hi * 2^32 and lo are exact doubles, so their sum rounds once."""
    a = np.asarray(a, dtype=np.int64)
    hi = (a >> 32).astype(np.float64) * 4294967296.0
    return hi + (a & 0xFFFFFFFF).astype(np.float64)


def uint64_to_double(a):
    """(double) a of an unsigned 64-bit integer, rounded to nearest (as int64_to_double)."""
    a = np.asarray(a, dtype=np.uint64)
    hi = (a >> np.uint64(32)).astype(np.float64) * 4294967296.0
    return hi + (a & np.uint64(0xFFFFFFFF)).astype(np.float64)


def fused_q_minus_m2(m, q):
    """fma(-m, m, q) of float64 arrays: q - m^2 exactly as a ratio of Python integers (the denominators are powers of
    two), rounded once by int / int, which CPython rounds correctly."""
    m, q = np.broadcast_arrays(np.asarray(m, dtype=np.float64), np.asarray(q, dtype=np.float64))
    out = np.empty(m.shape, dtype=np.float64)
    flat = out.reshape(-1)
    for i, (mi, qi) in enumerate(zip(m.reshape(-1).tolist(), q.reshape(-1).tolist())):
        a, b = mi.as_integer_ratio()
        c, d = qi.as_integer_ratio()
        flat[i] = (c * b * b - a * a * d) / (d * b * b)
    return out


def rule_error(sums, squares, counts, fused=True):
    """The rule's e per pixel as float64, bit for bit the device's (the module docstring); +inf where n < 2.  sums and
    squares have shape counts.shape + (3,).  fused=False rounds m * m on its own (what the device does NOT do), for
    showing that the two differ."""
    sums = np.asarray(sums, dtype=np.int64)
    squares = np.asarray(squares, dtype=np.uint64)
    counts = np.asarray(counts, dtype=np.uint32)
    e = np.full(counts.shape, np.inf)
    ok = counts >= 2
    if not ok.any():
        return e
    n = counts[ok].astype(np.float64)[:, None]
    m = int64_to_double(sums[ok]) * 2.0 ** -30 / n
    q = uint64_to_double(squares[ok]) * 2.0 ** -32 / n
    v = fused_q_minus_m2(m, q) if fused else q - m * m
    se = np.sqrt(np.fmax(v, 0.0) / (n - 1.0))
    ec = (np.sqrt(np.fmax(m + se, 0.0)) - np.sqrt(np.fmax(m - se, 0.0))) * 128.0
    e[ok] = np.fmax(np.fmax(np.fmax(0.0, ec[:, 0]), ec[:, 1]), ec[:, 2])
    return e


def error_map(sums, squares, counts):
    """What vk_adaptive_read's out_error holds (in the accumulators' order): (float)e, +inf below two samples."""
    return rule_error(sums, squares, counts).astype(np.float32)


def stops(e, counts, target):
    """The rule of include/vecchio_gpu.h for target (spp, min_spp, max_error): a pixel at n samples stops when n >= spp,
    or when max_error > 0, n > 1, n >= min_spp and e <= max_error (max_error as the float32 the library holds)."""
    spp, min_spp, max_error = target
    counts = np.asarray(counts, dtype=np.int64)
    E = float(np.float32(max_error))
    stop = counts >= spp
    if E > 0.0:
        stop = stop | ((counts > 1) & (counts >= min_spp) & (np.asarray(e, dtype=np.float64) <= E))
    return stop


def means(sums, counts):
    """k_finalize over an adaptive state (AccOverCount): (float)((double)S * 2^-30) / (float)n per channel (0 / 0 = NaN
    for a pixel without samples)."""
    s = int64_to_double(sums) * 2.0 ** -30
    with np.errstate(divide="ignore", invalid="ignore"):
        return s.astype(np.float32) / np.asarray(counts, dtype=np.uint32).astype(np.float32)[..., None]


def rgb8(vb, sums, counts):
    """vk_adaptive_read_rgb8's image: to_color of means() frame by frame (vb.frame_to_rgb8), each frame top-down.
    sums (..., H, W, 3) -> uint8 of the same shape."""
    mu = means(sums, counts)
    frames = mu.reshape((-1,) + mu.shape[-3:])
    return np.stack([vb.frame_to_rgb8(f) for f in frames]).reshape(mu.shape)


def square_units(sample_sum_units):
    """accumulate_square of one sample given as its sum units dS = round(L * 2^30) (exact for |L| >= 2^-7): the
    round-half-even integer nearest min(|L|, 255)^2 * 2^32, 0 for dS == 0.  Elementwise over an int64 array."""
    d = np.asarray(sample_sum_units, dtype=np.int64)
    out = np.empty(d.shape, dtype=np.uint64)
    flat = out.reshape(-1)
    cap = SQ_CLAMP * ACC_UNITS
    for i, x in enumerate(d.reshape(-1).tolist()):
        c = min(abs(x), cap)
        q, r = divmod(c * c, 1 << 28)  # c^2 * 2^32 / 2^60
        flat[i] = q + (1 if 2 * r > (1 << 28) or (2 * r == (1 << 28) and q & 1) else 0)
    return out


def grid(M, cap):
    """The counts a pixel can stop at under cap: M, 2M, .. below the cap, and the cap."""
    return list(range(M, cap, M)) + [cap]


def predict(states, target, M, start=None, errors=None):
    """The adaptive pass loop from fixed states: states[b] = (sums, squares) every pixel holds after samples [0, b), for
    each b of grid(M, target spp).  start = (counts, sums, squares) a pixel begins from (a refine of an imported state),
    None for a fresh session (every pixel at 0).  A pixel the rule lets go on at its count n renders on to the next grid
    point after n and is judged again there.  errors (optional): errors[b] = rule_error of states[b] at count b, for a
    caller that predicts several targets from the same states.  Returns each pixel's final (counts, sums, squares)."""
    spp = target[0]
    s0 = states[grid(M, spp)[0]]
    if start is None:
        n = np.zeros(s0[0].shape[:-1], dtype=np.uint32)
        S, Q = np.zeros_like(s0[0]), np.zeros_like(s0[1])
    else:
        n, S, Q = (np.array(a) for a in start)
        n = n.astype(np.uint32)
    active = ~stops(rule_error(S, Q, n), n, target)
    for b in grid(M, spp):
        sel = active & (n < b)
        if not sel.any():
            continue
        n[sel] = b
        S[sel] = states[b][0][sel]
        Q[sel] = states[b][1][sel]
        e = errors[b][sel] if errors is not None else rule_error(S[sel], Q[sel], n[sel])
        active[sel] = ~stops(e, n[sel], target)
    return n, S, Q
