"""K2 (cd_tiled.cu) against an exhaustive evaluation of every ordered pair, on airspaces built around the decision edges.

K2 decides "candidate" with an approximate, inflated hot filter and skips tile pairs that its cull finds out of reach; only
the candidates reach the exact routine.  Comparing the forms with each other cannot see a pair that the filter or the cull
wrongly drops (every form drops it), and the float64 oracle cannot see it inside its epsilon band.  tests/cd_exhaustive.cu
evaluates every ordered pair with the same exact routine and no filter, so every form must equal it exactly: pair sets,
per-row counts, tcpamax and the five attributes of every conflict, bit for bit.

The scenario generators below are test infrastructure: seeded airspaces of aircraft pairs whose closest approach, entry and
exit times, vertical separation, relative speed and vertical speed sit on either side of the thresholds, plus degenerate
geometry, across the globe and three protected-zone sizes.  ``test_generators_straddle_their_edges`` checks on the CPU,
with the float64 oracle, that each generator keeps landing pairs on both sides of the edges it targets.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import statebased

NM, FT, RE = 1852.0, 0.3048, 6371000.0
ZONES = {"small": (50.0, 15.0, 30.0), "default": (5.0 * NM, 1000.0 * FT, 300.0), "large": (20.0 * NM, 2000.0 * FT, 1200.0)}
LATS = (-45.0, 0.0, 52.0, 70.0, 85.0, 89.5)
OFFS = (1e-7, 1e-6, 1e-5, 1e-4)
SIGNED_OFFS = np.array([s * o for o in OFFS for s in (-1.0, 1.0)])
HERE = os.path.dirname(os.path.abspath(__file__))


# ---------------------------------------------------------------- scenario generators (float64, seeded)
class _Pairs:
    """Aircraft built pair by pair in a local frame: B's position relative to A (m east, north), velocities (m/s east,
    north), altitudes, vertical speeds.  ``probes[edge]``: the (i, j) index pairs built to sit at that edge."""

    def __init__(self):
        self.rows = []            # (d_east, d_north, ua, va, ub, vb, alt_a, alt_b, vs_a, vs_b)
        self.probes = {}

    def add(self, d, ua, va, ub, vb, alt_a, alt_b, vs_a=0.0, vs_b=0.0, edge=None):
        k = 2 * len(self.rows)
        self.rows.append((d[0], d[1], ua, va, ub, vb, alt_a, alt_b, vs_a, vs_b))
        if edge:
            self.probes.setdefault(edge, []).append((k, k + 1))


def _rel(rng, w, tc, e):
    """Relative position giving tcpa = tc and closest approach e (signed, to the left of w) for relative velocity w."""
    wm = np.hypot(*w)
    n = np.array([-w[1], w[0]]) / wm
    return -tc * np.asarray(w) + e * n


def _vel(rng, wm):
    """A's velocity and a relative velocity of magnitude wm, random directions."""
    gs = rng.uniform(60.0, 300.0)
    a, b = rng.uniform(0.0, 2 * np.pi, 2)
    return gs * np.sin(a), gs * np.cos(a), wm * np.sin(b), wm * np.cos(b)


def gen_zone_edges(zone, rng, dmax):
    """closest approach, entry time (vs the look-ahead), exit time, entry vs exit and |dalt| vs hpz, each at
    +-{1e-7 .. 1e-4} relative to its threshold (times: relative to the look-ahead), plus a continuous spread within
    +-1e-6 around the closest-approach edge (where the hot filter rounds differently from the exact routine)."""
    R, h, T = zone
    P = _Pairs()
    wcap = max(5.0, min(450.0, 0.5 * dmax / T))

    def pair(tc, e, edge, alt=None, dalt=0.0, vs=(0.0, 0.0), wm=None):
        ua, va, du, dv = _vel(rng, wm if wm is not None else rng.uniform(0.2, 1.0) * wcap)
        d = _rel(rng, (du, dv), tc, e)
        alt = rng.uniform(3000.0, 11000.0) if alt is None else alt
        P.add(d, ua, va, ua + du, va + dv, alt, alt + dalt, vs[0], vs[1], edge)

    for dl in np.concatenate([SIGNED_OFFS, rng.uniform(-1e-6, 1e-6, 24)]):
        pair(rng.uniform(0.05, 0.6) * T, rng.choice([-1.0, 1.0]) * R * (1.0 + dl), "dcpa")
    for dl in SIGNED_OFFS:
        wm = rng.uniform(0.2, 1.0) * wcap
        e = rng.uniform(0.0, 0.8) * R
        dtin = np.sqrt(R * R - e * e) / wm
        pair(T * (1.0 + dl) + dtin, e, "tin", wm=wm)                      # tin = T (1 + dl)
        pair(T * dl - dtin, e, "tout", wm=wm)                             # tout = T dl
    for dl in SIGNED_OFFS:
        # vertical window ends as the horizontal one opens: tinhor = t1, toutver = t1 (1 + dl)
        wm = rng.uniform(0.2, 1.0) * wcap
        e = rng.uniform(0.0, 0.8) * R
        dtin = np.sqrt(R * R - e * e) / wm
        t1 = rng.uniform(0.1, 0.6) * T
        dvs = min(rng.uniform(1.0, 15.0), 2.0 * h / t1)
        dalt = h - dvs * t1 * (1.0 + dl)                                 # toutver = (h - dalt) / dvs
        pair(t1 + dtin, e, "tin_tout", dalt=dalt, vs=(0.0, dvs), wm=wm)
    for dl in SIGNED_OFFS:
        # level pairs at |dalt| = hpz (1 + dl), converging horizontally; low and cruise altitudes (float32 resolution
        # of the altitude 3e-5 m and 1e-3 m)
        for alt in (100.0, rng.uniform(3000.0, 11000.0)):
            pair(rng.uniform(0.1, 0.5) * T, rng.uniform(0.0, 0.8) * R, "dalt", alt=alt, dalt=rng.choice([-1.0, 1.0]) * h * (1.0 + dl))
    return P


def gen_clamps(zone, rng, dmax):
    """co-moving pairs across the 1e-6 clamp of |w|^2, |dvs| across its 1e-6 clamp, level pairs at |dalt| = hpz +-
    {0, 1e-4, 1e-3} m (where the two orders of a pair differ: both clamp dvs to +1e-6)."""
    R, h, T = zone
    P = _Pairs()
    for w2 in (0.0, 1e-8, 1e-7, 5e-7, 1e-6 * (1 - 1e-3), 1e-6 * (1 + 1e-3), 2e-6, 1e-5):
        for gs in (0.5, 220.0):                                           # (float32 velocity steps 3e-8 and 1.5e-5 m/s)
            a, b = rng.uniform(0.0, 2 * np.pi, 2)
            ua, va = gs * np.sin(a), gs * np.cos(a)
            wm = np.sqrt(w2)
            dist = rng.choice([0.5, 0.99, 1.5]) * R
            c = rng.uniform(0.0, 2 * np.pi)
            alt = rng.uniform(3000.0, 11000.0)
            P.add((dist * np.sin(c), dist * np.cos(c)), ua, va, ua + wm * np.sin(b), va + wm * np.cos(b), alt,
                  alt + rng.choice([0.0, 0.5, 2.0]) * h, edge="dv2")
    wcap = max(5.0, min(450.0, 0.5 * dmax / T))
    for dvs in (0.0, 5e-7, -5e-7, 1e-6, -1e-6, 2e-6, -2e-6):
        for vs_a, dfrac in ((0.0, 0.5), (0.0, 1.0), (0.0, 1.001), (12.0, 0.5)):
            ua, va, du, dv = _vel(rng, rng.uniform(0.2, 1.0) * wcap)
            d = _rel(rng, (du, dv), rng.uniform(0.1, 0.5) * T, rng.uniform(0.0, 0.8) * R)
            alt = rng.uniform(3000.0, 11000.0)
            P.add(d, ua, va, ua + du, va + dv, alt, alt + rng.choice([-1.0, 1.0]) * dfrac * h, vs_a, vs_a + dvs, edge="dvs")
    for dh in (0.0, 1e-4, -1e-4, 1e-3, -1e-3):
        for alt in (100.0, 9000.0):
            ua, va, du, dv = _vel(rng, rng.uniform(0.2, 1.0) * wcap)
            d = _rel(rng, (du, dv), rng.uniform(0.1, 0.5) * T, rng.uniform(0.0, 0.8) * R)
            P.add(d, ua, va, ua + du, va + dv, alt, alt + rng.choice([-1.0, 1.0]) * (h + dh), edge="dalt")
    return P


def gen_degenerate(zone, rng, dmax):
    """co-located pairs (one also at the same altitude), vertical stacks converging in altitude only, head-on and in-trail
    pairs on one great circle (a meridian, the parallel through the pair), stationary aircraft, 350 m/s, |vs| to 50 m/s."""
    R, h, T = zone
    P = _Pairs()
    alt = lambda: rng.uniform(3000.0, 11000.0)
    a0 = alt()
    P.add((0.0, 0.0), 100.0, 50.0, -80.0, 20.0, a0, a0)                                  # same place, same altitude
    P.add((0.0, 0.0), 100.0, 50.0, 100.0, 50.0, a0, a0 + 0.5 * h)                         # same place, co-moving
    P.add((0.0, 0.0), 0.0, 0.0, 0.0, 0.0, a0, a0 + 2.0 * h)                               # same place, stationary, apart
    for dalt, dvs in ((3.0 * h, -10.0), (-3.0 * h, 10.0), (1.5 * h, -50.0), (4.0 * h, 5.0)):
        P.add((0.0, 0.0), 150.0, 10.0, 150.0, 10.0, a0, a0 + dalt, 0.0, dvs)             # vertical stacks
    s = min(0.9 * dmax, 400.0 * 0.5 * T)
    for gs_a, gs_b in ((200.0, 200.0), (350.0, 350.0), (0.0, 350.0), (120.0, 0.0)):
        P.add((0.0, s), 0.0, gs_a, 0.0, -gs_b, a0, a0)                                   # head-on on the meridian
        P.add((s, 0.0), gs_a, 0.0, -gs_b, 0.0, a0, a0)                                   # head-on along x
        P.add((0.0, 0.2 * s), 0.0, gs_a + 40.0, 0.0, gs_b * 0.5, a0, a0)                 # in trail, closing
    for vs_a, vs_b in ((50.0, -50.0), (-50.0, 0.0), (30.0, 30.0)):
        ua, va, du, dv = _vel(rng, 150.0)
        P.add(_rel(rng, (du, dv), 0.3 * T, 0.3 * R), ua, va, ua + du, va + dv, a0, a0 + 2.0 * h, vs_a, vs_b)
    P.add((0.3 * R, 0.1 * R), 0.0, 0.0, 0.0, 0.0, a0, a0)                                # both stationary, in LoS
    return P


def gen_clamped_far(zone, rng, dmax):
    """level pairs a few cm either side of |dalt| = hpz, closing slowly.  Both orders clamp dvs to +1e-6, so one order's
    vertical window opens (|dalt| - hpz) 1e6 s ahead while the other's closed as long ago.  The hot filter's hpz margin
    (1e-4 hpz + 1 cm) covers such pairs only up to ~4e4 s; beyond it, with a look-ahead of hours, only the symmetric
    form's fold of the two orders (cd_hot2: dalt := -|dalt|) keeps the mirrored order."""
    R, h, T = zone
    P = _Pairs()
    for dh in (0.05, 0.07, -0.05, -0.07):
        for alt in (100.0, 200.0):                                          # (float32 altitude steps below 3e-5 m)
            e = rng.uniform(0.0, 0.6) * R
            wm = np.sqrt(R * R - e * e) / (0.45 * T)                          # horizontal window 0.05 T .. 0.95 T
            ua, va, du, dv = _vel(rng, wm)
            d = _rel(rng, (du, dv), 0.5 * T, e)
            P.add(d, ua, va, ua + du, va + dv, alt, alt + rng.choice([-1.0, 1.0]) * (h + dh), edge="dalt")
    return P


GENERATORS = {"zone_edges": gen_zone_edges, "clamps": gen_clamps, "degenerate": gen_degenerate, "clamped_far": gen_clamped_far}
# a look-ahead of hours: where gen_clamped_far's pairs conflict (in one order only)
LONG = (5.0 * NM, 1000.0 * FT, 1.0e5)


def _dmax(lat):
    """largest pair extent [m] that keeps both aircraft off the pole"""
    return float(min(6.0e5, max(2.0e4, 0.45 * (90.0 - abs(lat)) * 111e3)))


def scenario(n, zone, lat_c, lon_c=4.0, seed=0, kinds=tuple(GENERATORS), dup=0, spacing=None):
    """``n`` aircraft made of generator pairs (cycling through ``kinds``), the pairs laid on a grid around (lat_c, lon_c)
    ``spacing`` metres apart (default 3 rpz), then shuffled.  ``dup`` aircraft are exact copies of others.  Returns
    (lat, lon, trk, gs, alt, vs), probes {edge: [k, 2] index pairs}."""
    rng = np.random.default_rng(seed)
    R = zone[0]
    dmax = _dmax(lat_c)
    rows, probes = [], {}
    k = 0
    while 2 * len(rows) < n - dup:
        P = GENERATORS[kinds[k % len(kinds)]](zone, rng, dmax)
        base = 2 * len(rows)
        rows += P.rows
        for e, p in P.probes.items():
            probes.setdefault(e, []).extend((i + base, j + base) for i, j in p)
        k += 1
    r = np.array(rows, dtype=np.float64)
    m = len(r)
    side = int(np.ceil(np.sqrt(m)))
    sp = 3.0 * R if spacing is None else spacing
    gx, gy = (np.arange(m) % side - 0.5 * side) * sp, (np.arange(m) // side - 0.5 * side) * sp
    lim = 0.45 * (90.0 - abs(lat_c)) * 111e3                            # the grid stays off the pole too
    if side * sp > lim:
        gx, gy = gx * lim / (side * sp), gy * lim / (side * sp)
    latc = lat_c + np.degrees(gy / RE)
    lonc = lon_c + np.degrees(gx / (RE * np.cos(np.radians(lat_c))))
    # A at -d/2, B at +d/2; the x offset uses the cos of the pair's mean latitude, as the kwik metric does
    hy = np.degrees(0.5 * r[:, 1] / RE)
    latc = np.clip(latc, -89.95 + np.abs(hy), 89.95 - np.abs(hy))
    hx = np.degrees(0.5 * r[:, 0] / (RE * np.cos(np.radians(latc))))
    lat = np.stack([latc - hy, latc + hy], 1).ravel()
    lon = np.stack([lonc - hx, lonc + hx], 1).ravel()
    u, v = np.stack([r[:, 2], r[:, 4]], 1).ravel(), np.stack([r[:, 3], r[:, 5]], 1).ravel()
    alt = np.stack([r[:, 6], r[:, 7]], 1).ravel()
    vs = np.stack([r[:, 8], r[:, 9]], 1).ravel()
    gs, trk = np.hypot(u, v), np.degrees(np.arctan2(u, v)) % 360.0
    arrs = [lat, lon, trk, gs, alt, vs]
    keep = n - dup
    arrs = [a[:keep] for a in arrs]
    if dup:
        src = rng.integers(0, keep, dup)
        arrs = [np.concatenate([a, a[src]]) for a in arrs]
    arrs[1] = (arrs[1] + 180.0) % 360.0 - 180.0
    perm = rng.permutation(n)                                       # pair members land in arbitrary tiles, either order
    inv = np.empty(n, dtype=np.int64)
    inv[perm] = np.arange(n)
    arrs = [a[perm] for a in arrs]
    pr = {e: inv[np.array([p for p in ps if p[0] < keep and p[1] < keep], dtype=np.int64).reshape(-1, 2)] for e, ps in probes.items()}
    return tuple(arrs), pr


def clustered(n, seed=0):
    """~n aircraft in 64 dense clusters about 600 km apart: random tracks, flight levels, 20 % climbing or descending.
    The cull keeps a few percent of the tile pairs of the spatially ordered records."""
    rng = np.random.default_rng(seed)
    k = 64
    cl = rng.integers(0, k, n)
    clat = 40.0 + 6.0 * (np.arange(k) // 8)
    clon = -20.0 + 8.0 * (np.arange(k) % 8)
    lat = clat[cl] + rng.uniform(-0.15, 0.15, n)
    lon = clon[cl] + rng.uniform(-0.2, 0.2, n)
    alt = np.round(rng.uniform(3000.0, 12000.0, n) / 304.8) * 304.8 + rng.uniform(-20.0, 20.0, n)
    gs = rng.uniform(150.0, 250.0, n)
    trk = rng.uniform(0.0, 360.0, n)
    vs = np.where(rng.random(n) < 0.8, 0.0, rng.choice([-1.0, 1.0], n) * rng.uniform(5.0, 15.0, n))
    return lat, lon, trk, gs, alt, vs


# ---------------------------------------------------------------- CPU: the generators keep straddling their edges
def _margins(s, probes, zone):
    """float64 oracle: signed distance of each probe to its threshold (negative: the side that detects)."""
    R, h, T = zone
    lat, lon, trk, gs, alt, vs = s
    out = {}
    for e, p in probes.items():
        i, j = p[:, 0], p[:, 1]
        o = statebased.detect_rows(i, *s, R, h, T)
        k = np.arange(len(i))
        u, v = gs * np.sin(np.radians(trk)), gs * np.cos(np.radians(trk))
        m = {"dcpa": o["dcpa2"][k, j] - R * R,
             "tin": o["tinconf"][k, j] - T,
             "tout": -o["toutconf"][k, j],
             "tin_tout": o["tinconf"][k, j] - o["toutconf"][k, j],
             "dalt": np.abs(alt[j] - alt[i]) - h,
             "dv2": (u[j] - u[i]) ** 2 + (v[j] - v[i]) ** 2 - 1e-6,
             "dvs": np.abs(vs[j] - vs[i]) - 1e-6}[e]
        out[e] = (m, o["swconfl"][k, j])
    return out


@pytest.mark.parametrize("lat", LATS)
@pytest.mark.parametrize("zone", list(ZONES))
def test_generators_straddle_their_edges(zone, lat):
    """Every generator, at every zone size and latitude, lands probes on both sides of each edge it targets, close to it;
    at the conflict-deciding edges the oracle decides both ways."""
    z = ZONES[zone]
    for kind in GENERATORS:
        s, probes = scenario(600, z, lat, seed=7, kinds=(kind,))
        assert np.isfinite(np.array(s)).all() and (np.abs(s[0]) < 90.0).all()
        for e, (m, conf) in _margins(s, probes, z).items():
            scale = {"dcpa": z[0] ** 2, "tin": z[2], "tout": z[2], "tin_tout": z[2], "dalt": z[1], "dv2": 1e-6, "dvs": 1e-6}[e]
            assert (m < 0).any() and (m > 0).any(), (kind, e, "probes on one side only")
            near = np.abs(m) < {"dv2": 10.0, "dvs": 20.0}.get(e, 1e-3) * scale + (0.1 if e == "dalt" else 0.0)
            assert near.mean() > 0.5, (kind, e, "probes drifted away from the edge")
            if e in ("dcpa", "tin", "tout", "tin_tout"):
                assert conf.any() and not conf.all(), (kind, e, "the oracle decides every probe the same way")


def _nvcc():
    return os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def _build_harness(out_dir):
    from bluesky_gym_sasha_b200 import build
    so = os.path.join(str(out_dir), "cd_exhaustive.so")
    res = subprocess.run([_nvcc()] + build.NVCC_FLAGS + ["-I", build.CSRC, "-o", so, os.path.join(HERE, "cd_exhaustive.cu"), "-lcudart"],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    return so


def test_harness_compiles_for_sm100a(tmp_path):
    """The exhaustive reference builds for sm_100a without a GPU and exports its C entry point."""
    so = _build_harness(tmp_path)
    res = subprocess.run([os.path.join(os.path.dirname(_nvcc()), "cuobjdump"), "-lelf", so], capture_output=True, text=True)
    assert res.returncode == 0 and "sm_100a" in res.stdout, res.stdout + res.stderr
    res = subprocess.run(["nm", "-D", so], capture_output=True, text=True)
    assert " T cd_exhaustive" in res.stdout


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def ex(cuda, tmp_path_factory):
    lib = C.CDLL(_build_harness(tmp_path_factory.mktemp("cd_exhaustive")))
    lib.cd_exhaustive.restype = C.c_int
    lib.cd_exhaustive.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_int,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                  C.c_void_p, C.c_void_p]
    return lib


def _keys(p):
    p = np.asarray(p, dtype=np.int64).reshape(-1, 2)
    return (p[:, 0] << 32) | p[:, 1]


def exhaustive(lib, rec, n_all, zone, wrap=False, row0=0, n_rows=None, cap=1 << 21):
    """The exhaustive reference on the records ``rec``: host arrays; pairs sorted by (i, j), attributes in that order."""
    import torch
    n_rows = n_all - row0 if n_rows is None else n_rows
    m = max(n_rows, 1)
    d = dict(nconf_row=torch.zeros(m, dtype=torch.int32, device=rec.device), nlos_row=torch.zeros(m, dtype=torch.int32, device=rec.device),
             tcpamax=torch.zeros(m, dtype=torch.float32, device=rec.device), pairs=torch.zeros((cap, 2), dtype=torch.int32, device=rec.device),
             attr=torch.zeros((cap, 5), dtype=torch.float32, device=rec.device), los=torch.zeros((cap, 2), dtype=torch.int32, device=rec.device),
             npairs=torch.zeros(2, dtype=torch.int64, device=rec.device))
    rc = lib.cd_exhaustive(rec.data_ptr(), n_all, row0, n_rows, zone[0], zone[1], zone[2], int(wrap), *(d[k].data_ptr() for k in ("nconf_row", "nlos_row", "tcpamax", "pairs", "attr")),
                           cap, d["los"].data_ptr(), cap, d["npairs"].data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, rc
    torch.cuda.synchronize()
    nc, nl = (int(x) for x in d["npairs"].cpu())
    assert nc <= cap and nl <= cap
    pairs = d["pairs"][:nc].cpu().numpy()
    o = np.argsort(_keys(pairs))
    lo = d["los"][:nl].cpu().numpy()
    return dict(nconf_row=d["nconf_row"][:n_rows].cpu().numpy(), nlos_row=d["nlos_row"][:n_rows].cpu().numpy(),
                tcpamax=d["tcpamax"][:n_rows].cpu().numpy(), keys=_keys(pairs)[o], attr=d["attr"][:nc].cpu().numpy()[o],
                los_keys=np.sort(_keys(lo)), n_conf=nc, n_los=nl)


def _assert_equal(ref, out, cap, los_cap, what, rows=None):
    """A form's device outputs (``detect_packed``) == the exhaustive reference; ``rows``: the reference rows it covers.
    Truncated lists (cap < total): exactly min(total, cap) distinct pairs, all in the reference, each attribute row the
    reference attributes of its own pair."""
    import torch
    torch.cuda.synchronize()
    sl = slice(None) if rows is None else rows
    nc, nl = (int(x) for x in out["npairs"].cpu())
    tc, tl = len(ref["keys"]), len(ref["los_keys"])
    if rows is not None:
        lo, hi = rows.start, rows.stop
        in_rows = lambda k: ((k >> 32) >= lo) & ((k >> 32) < hi)
        rk, ra, rl = ref["keys"][in_rows(ref["keys"])], ref["attr"][in_rows(ref["keys"])], ref["los_keys"][in_rows(ref["los_keys"])]
    else:
        rk, ra, rl = ref["keys"], ref["attr"], ref["los_keys"]
    assert (nc, nl) == (len(rk), len(rl)), (what, "totals", (nc, nl), (len(rk), len(rl)))
    assert np.array_equal(out["nconf_row"].cpu().numpy(), ref["nconf_row"][sl]), (what, "nconf_row")
    assert np.array_equal(out["nlos_row"].cpu().numpy(), ref["nlos_row"][sl]), (what, "nlos_row")
    assert np.array_equal(out["inconf"].cpu().numpy() != 0, ref["nconf_row"][sl] > 0), (what, "inconf")
    assert np.array_equal(out["tcpamax"].cpu().numpy().view(np.uint32), ref["tcpamax"][sl].view(np.uint32)), (what, "tcpamax")
    k = min(nc, cap)
    keys = _keys(out["pairs"][:k].cpu().numpy())
    attr = out["attr"][:k].cpu().numpy()
    assert len(np.unique(keys)) == k, (what, "duplicate conflict pairs")
    pos = np.searchsorted(rk, keys)
    assert (pos < len(rk)).all() and np.array_equal(rk[np.minimum(pos, len(rk) - 1)], keys), (what, "conflict not in the reference")
    bad = np.where((attr.view(np.uint32) != ra[pos].view(np.uint32)).any(axis=1))[0]
    assert not len(bad), (what, "attributes differ", keys[bad[:3]] >> 32, keys[bad[:3]] & 0xffffffff, attr[bad[:3]], ra[pos[bad[:3]]])
    kl = min(nl, los_cap)
    lk = np.sort(_keys(out["lospairs"][:kl].cpu().numpy()))
    assert len(np.unique(lk)) == kl and np.isin(lk, rl).all(), (what, "LoS list")
    if k == nc:
        assert np.array_equal(np.sort(keys), rk), (what, "conflict set")
    if kl == nl:
        assert np.array_equal(lk, rl), (what, "LoS set")
    return nc, nl


def _near(ref, zone):
    """reference conflicts whose closest approach or entry time sits within 1e-5 (relative) of rpz or the look-ahead"""
    a = ref["attr"].astype(np.float64)
    return int(((np.abs(a[:, 2] / zone[0] - 1.0) < 1e-5) | (np.abs(a[:, 4] / zone[2] - 1.0) < 1e-5)).sum())


def _check_forms(cd, ex, s, zone, lat0, lon0, wrap, name, shards=True, deal=True, cap=1 << 20, los_cap=None):
    """Every form on bsg_cd_pack's and bsg_cd_pack_ordered's records == the exhaustive reference on the same records."""
    import torch
    los_cap = cap if los_cap is None else los_cap
    n = len(s[0])
    cd.pair_capacity, cd.los_capacity = cap, los_cap
    rec, _ = cd.pack(*s, lat0, lon0)
    ref = exhaustive(ex, rec, n, zone, wrap)
    chk = lambda out, what, rows=None: _assert_equal(ref, out, cap, los_cap, f"{name}: {what}", rows)
    chk(cd.detect_packed(rec, n, lon_wrap=wrap), "plain")
    if shards and n > 2:
        cuts = sorted({0, n, *np.random.default_rng(n).integers(1, n, 3).tolist()})
        for a, b in zip(cuts[:-1], cuts[1:]):
            chk(cd.detect_packed(rec, n, row0=a, n_rows=b - a, lon_wrap=wrap), f"plain rows {a}:{b}", slice(a, b))
    recs = [(rec, ref, "packed")]
    if not wrap:
        reco, _, _ = cd.pack_ordered(*s, lat0, lon0)
        recs.append((reco, exhaustive(ex, reco, n, zone), "ordered"))
    for r, rf, how in recs if not wrap else []:
        ref = rf
        chk(cd.detect_packed(r, n, cull=True), f"{how} culled")
        chk(cd.detect_packed(r, n, symmetric=True), f"{how} symmetric all tiles")
        chk(cd.detect_packed(r, n, cull=True, symmetric=True), f"{how} culled + symmetric")
        if shards and n > 256:
            cuts = list(range(0, n, 256 * max(1, n // 1024))) + [n]
            for a, b in zip(cuts[:-1], cuts[1:]):
                chk(cd.detect_packed(r, n, row0=a, n_rows=b - a, cull=True), f"{how} culled rows {a}:{b}", slice(a, b))
        if deal and how == "ordered":
            for world in (2, 3, 8):
                for cull in (False, True):
                    acc = [np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, np.float32), np.zeros(2, np.int64)]
                    for rank in range(world):
                        o = cd.detect_packed(r, n, cull=cull, symmetric=True, deal=(world, rank))
                        torch.cuda.synchronize()
                        acc[0] += o["nconf_row"].cpu().numpy()
                        acc[1] += o["nlos_row"].cpu().numpy()
                        acc[2] = np.maximum(acc[2], o["tcpamax"].cpu().numpy())
                        acc[3] += o["npairs"].cpu().numpy()
                    what = f"{name}: dealt over {world}, cull={cull}"
                    assert np.array_equal(acc[0], ref["nconf_row"]) and np.array_equal(acc[1], ref["nlos_row"]), what
                    assert np.array_equal(acc[2].view(np.uint32), ref["tcpamax"].view(np.uint32)), what
                    assert tuple(acc[3]) == (len(ref["keys"]), len(ref["los_keys"])), what
    return len(recs[0][1]["keys"]), len(recs[0][1]["los_keys"]), _near(recs[0][1], zone)


def _report(name, n, nc, nl, near):
    print(f"{name}: {n * n} ordered pairs, {nc} conflicts, {nl} LoS pairs, {near} conflicts with dcpa within 1e-5 of rpz")


@pytest.fixture(scope="module")
def cd(cuda):
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    return StateBasedCD(device=0)


def _cd_for(cd, zone):
    cd.rpz, cd.hpz, cd.dtlookahead = zone
    return cd


@pytest.mark.gpu
@pytest.mark.parametrize("lat", LATS)
@pytest.mark.parametrize("zone", list(ZONES))
def test_edges_every_form_equals_exhaustive(cd, ex, zone, lat):
    """The edge, clamp and degenerate generators at every latitude and zone size, 4097 aircraft (1025 next to the pole,
    where they crowd into a few tens of km)."""
    z = ZONES[zone]
    n = 4097 if abs(lat) < 80.0 else 1025
    s, _ = scenario(n, z, lat, seed=10 * list(ZONES).index(zone) + LATS.index(lat))
    lat0 = float(np.mean(s[0]))
    nc, nl, near = _check_forms(_cd_for(cd, z), ex, s, z, lat0, 4.0, False, f"{zone} @ {lat}", deal=(lat == 52.0))
    _report(f"{zone} @ {lat}", n, nc, nl, near)
    assert nc > 100 and nl > 10


@pytest.mark.gpu
def test_clamped_pairs_far_ahead_equal_exhaustive(cd, ex):
    """Pairs that conflict in one order only, hours ahead (gen_clamped_far), with a look-ahead of 1e5 s: the symmetric
    forms must keep the mirrored order that their hot filter does not see directly."""
    s, probes = scenario(2048, LONG, 52.0, seed=8, kinds=("clamped_far",))
    nc, nl, near = _check_forms(_cd_for(cd, LONG), ex, s, LONG, 52.0, 4.0, False, "long look-ahead", deal=False)
    _report("long look-ahead", 2048, nc, nl, near)
    assert nc > 100


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 255, 256, 257, 511, 4097])
def test_sizes_every_form_equals_exhaustive(cd, ex, n):
    """Ragged and tile-boundary sizes, with duplicated aircraft."""
    z = ZONES["default"]
    s, _ = scenario(n, z, 52.0, seed=n, dup=n // 16, spacing=1.5 * z[0])
    nc, nl, near = _check_forms(_cd_for(cd, z), ex, s, z, 52.0, 4.0, False, f"N={n}")
    _report(f"N={n}", n, nc, nl, near)


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["antimeridian_culled", "antimeridian_wrap", "far_from_origin"])
def test_globe_origins_equal_exhaustive(cd, ex, where):
    """An airspace across the antimeridian with its origin next to it (culled forms), the same with the origin half a
    world away (wrap, plain form), one 150 degrees of longitude from the origin (x ~ 1.7e7 m: float32 steps of 1-2 m)."""
    z = ZONES["default"]
    lon_c, lon0, wrap = {"antimeridian_culled": (180.0, 179.9, False), "antimeridian_wrap": (180.0, 0.0, True),
                         "far_from_origin": (154.0, 4.0, False)}[where]
    s, _ = scenario(3001, z, 35.0, lon_c=lon_c, seed=3)
    if where.startswith("antimeridian"):
        assert (s[1] > 179.0).any() and (s[1] < -179.0).any()
    nc, nl, near = _check_forms(_cd_for(cd, z), ex, s, z, 35.0, lon0, wrap, where, deal=False)
    _report(where, 3001, nc, nl, near)
    assert nc > 100


@pytest.mark.gpu
def test_clustered_and_truncated_lists(cd, ex):
    """~20 000 aircraft in dense clusters (the cull keeps few tiles) in full, then with both lists well below the totals:
    npairs and the per-row outputs stay exact, the lists hold min(total, cap) distinct reference pairs, and every attribute
    row belongs to its own pair."""
    import torch
    z = ZONES["default"]
    s = clustered(20000, seed=9)
    nc, nl, near = _check_forms(_cd_for(cd, z), ex, s, z, 52.0, 4.0, False, "clustered", shards=False, deal=False)
    _report("clustered", 20000, nc, nl, near)
    assert nc > 20000 and nl > 100
    rec, _, _ = cd.pack_ordered(*s, 52.0, 4.0)
    n = len(s[0])
    n_tiles = (n + 255) // 256
    cd.detect_packed(rec, n, cull=True)
    torch.cuda.synchronize()
    cnt_off = 16 * ((n_tiles * 12 * 4 + 15) // 16)
    frac = cd._buf["cull_work"][cnt_off:cnt_off + 4 * n_tiles].view(torch.int32).cpu().numpy().sum() / float(n_tiles ** 2)
    assert frac < 0.1, frac
    cap, los_cap = nc // 3, nl // 2
    _check_forms(cd, ex, s, z, 52.0, 4.0, False, "clustered, truncated", shards=False, deal=False, cap=cap, los_cap=los_cap)
    cd.pair_capacity = cd.los_capacity = 1 << 22


@pytest.mark.gpu
@pytest.mark.parametrize("cull", [False, True])
def test_peer_form_equals_exhaustive(cd, ex, cull):
    """bsg_cd_detect_peers with four record buffers on one device (standing in for four GPUs) == the exhaustive reference."""
    import torch
    from bluesky_gym_sasha_b200 import _lib
    from bluesky_gym_sasha_b200.cd import cd_records
    z = ZONES["large"]
    zc = _cd_for(cd, z)
    W, per = 4, 768
    s, _ = scenario(W * per - 5, z, 70.0, seed=4)
    rec = cd_records(W * per, zc.device, inert=True)
    (zc.pack_ordered if cull else zc.pack)(*s, 70.0, 4.0, out=rec)
    n = W * per
    ref = exhaustive(ex, rec, n, z)
    blocks = [rec[r * per // 256:(r + 1) * per // 256].clone() for r in range(W)]
    ptrs = (C.c_void_p * W)(*[b.data_ptr() for b in blocks])
    lib = _lib.load()
    for r in range(W):
        o = dict(nconf_row=torch.zeros(per, dtype=torch.int32, device="cuda"), nlos_row=torch.zeros(per, dtype=torch.int32, device="cuda"),
                 tcpamax=torch.zeros(per, dtype=torch.float32, device="cuda"), inconf=torch.zeros(per, dtype=torch.uint8, device="cuda"),
                 npairs=torch.zeros(2, dtype=torch.int64, device="cuda"), pairs=torch.zeros((1 << 16, 2), dtype=torch.int32, device="cuda"),
                 attr=torch.zeros((1 << 16, 5), dtype=torch.float32, device="cuda"), lospairs=torch.zeros((1 << 14, 2), dtype=torch.int32, device="cuda"))
        lists = _lib.CdLists(d_conf_pairs=o["pairs"].data_ptr(), d_conf_attr=o["attr"].data_ptr(), conf_cap=1 << 16,
                             d_los_pairs=o["lospairs"].data_ptr(), los_cap=1 << 14, d_npairs=o["npairs"].data_ptr())
        nbytes = int(lib.bsg_cd_cull_workspace(n, per))
        work = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
        _lib.check(lib.bsg_cd_detect_peers(ptrs, W, r, per, *z, _lib.CD_CULL if cull else 0, *(o[k].data_ptr() for k in ("nconf_row", "nlos_row", "tcpamax", "inconf")),
                                           C.byref(lists), work.data_ptr(), nbytes, None))
        _assert_equal(ref, o, 1 << 16, 1 << 14, f"peers rank {r}, cull={cull}", slice(r * per, (r + 1) * per))
    assert len(ref["keys"]) > 100


@pytest.mark.gpu
def test_airspace_detection_equals_exhaustive(ex, cuda):
    """AirspaceTraffic's own detection (culled + symmetric, traf_pack's float32 velocities, a non-default zone) on a
    generator airspace: after each of a few substeps, the records it packed through the exhaustive reference == its outputs."""
    import torch
    from bluesky_gym_sasha_b200.traffic import AirspaceTraffic
    z = (3.0 * NM, 800.0 * FT, 180.0)
    s, _ = scenario(1500, ZONES["default"], 52.0, seed=12, spacing=2.0 * ZONES["default"][0])
    lat, lon, trk, gs, alt, vs = s
    g = AirspaceTraffic(1500, rpz=z[0], hpz=z[1], dtlookahead=z[2], lat0=52.0, lon0=4.0)
    g.create(lat, lon, trk, alt, np.clip(gs, 60.0, 250.0))
    g.alt(np.arange(0, 1500, 5), alt[::5] + 600.0, vs=np.full(300, 8.0))
    tot = 0
    for step in range(4):
        g.step(1)
        torch.cuda.synchronize()
        ref = exhaustive(ex, g.rec, g.n, z)
        out = dict(g.last)
        out = {k: (v[:g.n] if k in ("nconf_row", "nlos_row", "tcpamax", "inconf") else v) for k, v in out.items()}
        _assert_equal(ref, out, g.cd.pair_capacity, g.cd.los_capacity, f"airspace substep {step}")
        tot += len(ref["keys"])
    print(f"airspace: {tot} conflicts over 4 substeps")
    assert tot > 100
