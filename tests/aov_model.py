"""Host model of vk_render_aov (include/vecchio_gpu.h states the definition), in numpy float32.

The camera rays are rebuilt exactly as the strict build's camera_get_ray makes them: Philox4x32-10 on the counter
(pixel, sample, depth << 8 | block, word) with key seed + frame, u01 as the 24-bit grid, gen_range, and the get_ray
arithmetic in the kernel's operation order (no FMA, IEEE division).  A thin lens draws its disk with __sincosf on the GPU,
so rays of a camera with an aperture are close, not exact.  Tracing and texture lookups are passed in (the GPU's
vk_intersect / vk_eval_batch, or the oracle's), and the planes follow the definition's tables and sample order."""
import numpy as np

F = np.float32
M32 = np.uint64(0xFFFFFFFF)
VK_M_LAMBERTIAN, VK_M_METAL, VK_M_DIELECTRIC, VK_M_DIFFUSE_LIGHT, VK_M_ISOTROPIC, VK_M_SPECDIFFUSE = range(6)
VK_T_MEDIUM = 7
VK_EVAL_TEXTURE = 2
RAY_DTYPE = np.dtype([("origin", "<f4", 3), ("direction", "<f4", 3), ("time", "<f4"), ("tmin", "<f4"), ("tmax", "<f4")])
EVAL_DTYPE = np.dtype([("op", "<u4"), ("index", "<u4"), ("ray_o", "<f4", 3), ("ray_d", "<f4", 3), ("ray_time", "<f4"),
                       ("p", "<f4", 3), ("normal", "<f4", 3), ("t", "<f4"), ("u", "<f4"), ("v", "<f4"), ("front", "<u4"),
                       ("dir", "<f4", 3), ("xi", "<u4", 5),
                       ("alive", "<u4"), ("valid", "<u4"), ("out_o", "<f4", 3), ("out_d", "<f4", 3), ("out_time", "<f4"),
                       ("beta", "<f4", 3), ("L", "<f4", 3), ("value", "<f4")])


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Salmon et al. 2011) of broadcastable uint32 counters and key words; returns four uint32 arrays."""
    c = [np.asarray(x, dtype=np.uint64) & M32 for x in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(int(k0) & 0xFFFFFFFF), np.uint64(int(k1) & 0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & M32]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & M32, (k1 + np.uint64(0xBB67AE85)) & M32
    return [x.astype(np.uint32) for x in c]


def u01(x):
    """gen::<f32>() of the strict build: the top 24 bits times 2^-24 (exact)."""
    return (np.asarray(x, dtype=np.uint32) >> np.uint32(8)).astype(F) * F(5.9604644775390625e-8)


def gen_range(x, lo, hi):
    lo, hi = F(lo), F(hi)
    scale = hi - lo
    res = (np.uint32(0x3F800000) | (np.asarray(x, dtype=np.uint32) >> np.uint32(9))).view(F) * scale + (lo - scale)
    return np.where(res < hi, res, lo).astype(F)


def frame_key(seed, f):
    k = (int(seed) + int(f)) & 0xFFFFFFFFFFFFFFFF
    return k & 0xFFFFFFFF, k >> 32


def _v(a):
    return np.array(a[:], dtype=F)


def camera_sample(cam, width, height, key, s):
    """Sample s's camera ray of every pixel (i = y*W + x) and the ConstantMedium variates the render draws for it (depth 1,
    block 1, VK_MEDIUM_XI_SLOTS = 8 slots: the fourth counter word counts groups of four).  Returns (rays, medium_xi)."""
    n = width * height
    pix = np.arange(n, dtype=np.uint64)
    x, y = (pix % np.uint64(width)).astype(F), (pix // np.uint64(width)).astype(F)
    r = philox4x32_10(pix, s, 0, 0, *key)
    sx = ((x + u01(r[0])) / F(width - 1)).astype(F)
    ty = ((y + u01(r[1])) / F(height - 1)).astype(F)
    off = np.zeros((n, 3), dtype=F)
    if cam.lens_radius != 0.0:  # camera_lens_disk: block 1 of depth 0 (__sincosf on the GPU: not exact)
        q = philox4x32_10(pix, s, 1, 0, *key)
        rad = np.sqrt(u01(q[0])) * F(cam.lens_radius)
        ang = (F(2.0) * F(np.pi)) * u01(q[1])
        dx, dy = (rad * np.cos(ang)).astype(F), (rad * np.sin(ang)).astype(F)
        off = (_v(cam.u)[None] * dx[:, None] + _v(cam.v)[None] * dy[:, None]).astype(F)
    origin = _v(cam.origin)[None]
    rays = np.zeros(n, dtype=RAY_DTYPE)
    rays["origin"] = origin + off
    rays["direction"] = _v(cam.lower_left_corner)[None] + _v(cam.horizontal)[None] * sx[:, None] + _v(cam.vertical)[None] * ty[:, None] - origin - off
    rays["time"] = gen_range(r[2], cam.time0, cam.time1)
    rays["tmin"], rays["tmax"] = F(0.001), F(np.inf)
    b0, b1 = philox4x32_10(pix, s, (1 << 8) | 1, 0, *key), philox4x32_10(pix, s, (1 << 8) | 1, 1, *key)
    xi = np.stack([u01(w) for w in b0 + b1], axis=1).astype(F)
    return rays, xi


def texture_records(index, hits):
    recs = np.zeros(len(hits), dtype=EVAL_DTYPE)
    recs["op"] = VK_EVAL_TEXTURE
    recs["index"] = index
    recs["u"], recs["v"], recs["p"] = hits["u"], hits["v"], hits["p"]
    return recs


def materials_of(scene):
    d = scene.desc
    m = [d.materials[i] for i in range(d.n_materials)]
    return (np.array([x.type for x in m], dtype=np.uint32), np.array([x.tex for x in m], dtype=np.uint32),
            np.array([x.param for x in m], dtype=F), np.array([x.aux for x in m], dtype=np.uint32))


def sample_albedo(hits, mats, eval_batch):
    """The albedo table at every hit (rows that missed are ignored by the caller)."""
    mtype, mtex, mparam, maux = mats
    mi = np.minimum(hits["mat"], len(mtype) - 1)
    spec = mtype[mi] == VK_M_SPECDIFFUSE
    comp = [np.where(spec, mtex[mi], mi), np.where(spec, maux[mi], mi)]  # A's material: itself, or SpecDiffuse's two parts
    # (a Dielectric reads no texture: its record asks for texture 0)
    idx = [np.where(mtype[c] == VK_M_DIELECTRIC, np.uint32(0), mtex[c]) for c in comp]
    tex = eval_batch(np.concatenate([texture_records(i, hits) for i in idx]))["beta"].astype(F).reshape(2, len(hits), 3)
    front = (hits["front"] != 0)[:, None]
    out = []
    for c, t in zip(comp, tex):
        typ = mtype[c][:, None]
        a = np.where(typ == VK_M_DIELECTRIC, F(1.0), t)
        a = np.where(typ == VK_M_DIFFUSE_LIGHT, np.where(front, np.minimum(t, F(1.0)), F(0.0)), a)
        out.append(a.astype(F))
    pct = mparam[mi][:, None]
    mix = (pct * out[0] + (F(1.0) - pct) * out[1]).astype(F)
    return np.where(spec[:, None], mix, out[0]).astype(F)


def miss_color(d, background, sky):
    if not sky:
        return np.broadcast_to(np.array(background, dtype=F), d.shape).astype(F)
    n = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])
    t = (F(0.5) * (d[:, 1] / n + F(1.0)))[:, None]
    return ((F(1.0) - t) + np.array([0.5, 0.7, 1.0], dtype=F)[None] * t).astype(F)


def planes(samples, hits_per_sample, mats, eval_batch, width, height, background=(0.0, 0.0, 0.0), sky=False):
    """The four planes of one frame from its samples' rays and hits, in sample order: {"albedo": (H, W, 3), "normal":
    (H, W, 3), "depth": (H, W), "coverage": (H, W)}."""
    n_pix = width * height
    alb, nrm = np.zeros((n_pix, 3), dtype=F), np.zeros((n_pix, 3), dtype=F)
    dsum, hits = np.zeros(n_pix, dtype=F), np.zeros(n_pix, dtype=np.uint32)
    for (rays, _), h in zip(samples, hits_per_sample):
        d = rays["direction"]
        hit = h["prim"] != 0
        a = np.where(hit[:, None], sample_albedo(h, mats, eval_batch), np.clip(miss_color(d, background, sky), F(0.0), F(1.0)))
        alb = (alb + a).astype(F)
        medium = (h["prim"] >> np.uint32(28)) == VK_T_MEDIUM
        nrm = (nrm + np.where((hit & ~medium)[:, None], h["normal"], F(0.0))).astype(F)
        dist = h["t"] * np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])
        dsum = np.where(hit, dsum + dist, dsum).astype(F)
        hits += hit
    n = F(len(samples))
    with np.errstate(divide="ignore", invalid="ignore"):
        depth = np.where(hits > 0, dsum / hits.astype(F), F(np.inf)).astype(F)
    return {"albedo": (alb / n).reshape(height, width, 3), "normal": (nrm / n).reshape(height, width, 3),
            "depth": depth.reshape(height, width), "coverage": (hits.astype(F) / n).reshape(height, width)}
