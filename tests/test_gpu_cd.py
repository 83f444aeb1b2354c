"""K2 parity: bsg_cd_pack + bsg_cd_detect (through the C ABI) against the float64 oracle.

Bar (BASELINE.json north_star / SURVEY.md section 8c): conflict and LoS pair sets bit-exact except for
pairs whose deciding operand lies within the stated epsilon band of its threshold in the oracle
(|dcpa^2-R^2|/R^2 < 1e-4, time comparisons within 1e-2 s, |dist-rpz|/rpz < 1e-4, ||dalt|-hpz| < 0.05 m).
"""
import numpy as np
import pytest

from oracle import cbind, statebased
from tests.common import synth_airspace

pytestmark = pytest.mark.gpu
RPZ, HPZ, DTL = 9260.0, 304.8, 300.0


def _pos_quant(s, lat0=None, lon0=None):
    """Twice the float32 step of the largest |x|, |y| of the packed CD records (the origin as StateBasedCD.detect picks it
    by default): the resolution of the kernel's positions.  0.5 m within ~20 deg of the origin, 4 m half a world away."""
    import torch
    from bluesky_gym_sasha_b200 import _lib
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    lat0 = float(np.mean(s[0])) if lat0 is None else lat0
    lon0 = float(s[1][0]) if lon0 is None else lon0
    rec, n = StateBasedCD().pack(*s, lat0, lon0)
    xy = rec[:, [_lib.CD_REC_X, _lib.CD_REC_Y], :].permute(0, 2, 1).reshape(-1, 2)[:n]
    return 2.0 * float(np.spacing(np.float32(xy.abs().max().item())))


def _check_against_oracle(s, g, rows=None, stats=None, zone=(RPZ, HPZ, DTL), lat0=None, lon0=None):
    """Conflict AND LoS pair sets (as sets of ordered index pairs) identical to the float64 oracle outside the epsilon
    band; per-row outputs for rows with no banded pair; qdr / dist / dcpa / tcpa / tinconf of every common conflict.
    ``zone``: (rpz, hpz, dtlookahead) of the detection; ``lat0, lon0``: its origin (default: StateBasedCD.detect's)."""
    n = len(s[0])
    rows = np.arange(n) if rows is None else rows
    pos_quant = _pos_quant(s, lat0, lon0)
    o = statebased.detect_rows(rows, *s, *zone, with_margins=True)
    sw, near = o["swconfl"], o["near_conf"]
    gp = set(map(tuple, g["confpairs"].tolist()))
    row_of = {int(r): k for k, r in enumerate(rows)}
    gp = {p for p in gp if p[0] in row_of}
    op = {(int(rows[i]), int(j)) for i, j in zip(*np.where(sw))}
    bad = [p for p in gp ^ op if not near[row_of[p[0]], p[1]]]
    assert not bad, f"{len(bad)} pair mismatches outside the epsilon band, e.g. {bad[:5]}"
    n_exempt = len(gp ^ op)
    # LoS pairs as a set
    gl = {p for p in map(tuple, g["lospairs"].tolist()) if p[0] in row_of}
    ol = {(int(rows[i]), int(j)) for i, j in zip(*np.where(o["swlos"]))}
    badl = [p for p in gl ^ ol if not o["near_los"][row_of[p[0]], p[1]]]
    assert not badl, f"{len(badl)} LoS pair mismatches outside the epsilon band, e.g. {badl[:5]}"
    assert len(g["lospairs"]) == g["n_los"] and len(set(map(tuple, g["lospairs"].tolist()))) == g["n_los"]
    # per-row outputs, for rows with no banded pair
    clean = ~(near.any(axis=1) | o["near_los"].any(axis=1))
    nconf_o = sw.sum(axis=1)
    nlos_o = o["swlos"].sum(axis=1)
    gi = rows
    assert np.array_equal(g["nconf_row"][gi][clean], nconf_o[clean])
    assert np.array_equal(g["nlos_row"][gi][clean], nlos_o[clean])
    assert np.array_equal(g["inconf"][gi][clean], nconf_o[clean] > 0)
    tmax_o = np.max(o["tcpa"] * sw, axis=1)
    np.testing.assert_allclose(g["tcpamax"][gi][clean], tmax_o[clean], rtol=2e-4, atol=0.05)
    # attributes of the conflicts both sides report (float32 kernel vs float64 oracle; tolerances stated here):
    #   qdr 2e-3 deg (+ 2 pos_quant / dist), dist 1e-5 rel + pos_quant, dcpa 1e-4 rel + 4 pos_quant, tcpa 1e-4 rel + 0.05 s,
    #   tinconf 1e-4 rel + 0.05 s + 1e-2 of the half-width of the horizontal window (sqrt near dcpa = R), banded pairs skipped.
    #   pos_quant = resolution of the float32 record positions (_pos_quant): 0.5 m within ~20 deg of the airspace origin; the
    #   antimeridian test puts the origin half a world away (x ~ 2e7 m: 2 m steps, pos_quant 4 m) on purpose
    err = dict(qdr=0.0, dist=0.0, dcpa=0.0, tcpa=0.0, tinconf=0.0)
    for k, (i, j) in enumerate(map(tuple, g["confpairs"].tolist())):
        if i not in row_of or (i, j) not in op or near[row_of[i], j]:
            continue
        r = row_of[i]
        dist, dcpa, tcpa, tin = o["dist"][r, j], np.sqrt(o["dcpa2"][r, j]), o["tcpa"][r, j], o["tinconf"][r, j]
        dq = abs((g["qdr"][k] - o["qdr"][r, j] + 180.0) % 360.0 - 180.0)
        assert dq < 2e-3 + np.degrees(2.0 * pos_quant / max(dist, 1.0)), (i, j, "qdr", g["qdr"][k], o["qdr"][r, j])
        assert abs(g["dist"][k] - dist) < pos_quant + 1e-5 * dist, (i, j, "dist")
        assert abs(g["dcpa"][k] - dcpa) < 4.0 * pos_quant + 1e-4 * dcpa, (i, j, "dcpa", g["dcpa"][k], dcpa)
        assert abs(g["tcpa"][k] - tcpa) < 0.05 * max(1.0, 2.0 * pos_quant) + 1e-4 * abs(tcpa), (i, j, "tcpa")
        half = abs(tcpa - tin)
        assert abs(g["tinconf"][k] - tin) < 0.05 * max(1.0, 2.0 * pos_quant) + 1e-4 * abs(tin) + 1e-2 * half, (i, j, "tinconf", g["tinconf"][k], tin)
        for name, e in (("qdr", dq), ("dist", abs(g["dist"][k] - dist)), ("dcpa", abs(g["dcpa"][k] - dcpa)),
                        ("tcpa", abs(g["tcpa"][k] - tcpa)), ("tinconf", abs(g["tinconf"][k] - tin))):
            err[name] = max(err[name], float(e))
    if stats is not None:
        stats.update(err, n_los=len(ol), n_los_exempt=len(gl ^ ol))
    return n_exempt, len(op)


# zones (rpz, hpz, dtlookahead): the default, a small one and a large one
ZONES = {"default": (RPZ, HPZ, DTL), "small": (50.0, 15.0, 30.0), "large": (20 * 1852.0, 2000 * 0.3048, 1200.0)}
DENSE = [(2, 0.5, 52.0, "default"), (255, 2.0, 52.0, "default"), (256, 2.0, 52.0, "default"), (257, 2.0, 52.0, "default"),
         (1000, 4.0, 52.0, "default"), (3000, 6.0, 52.0, "default"), (4096, 40.0, 52.0, "default"),
         (2000, 0.08, -45.0, "small"), (2000, 4.0, 0.0, "default"), (2000, 8.0, 70.0, "large"), (1500, 1.5, 85.0, "default"),
         (1000, 0.6, 89.5, "default"), (2000, 5.0, -45.0, "large")]


@pytest.mark.parametrize("n,box,lat0,zone", DENSE, ids=[f"{n}-{b}" if (la, z) == (52.0, "default") else f"{n}-{b}-{la}-{z}"
                                                        for n, b, la, z in DENSE])
def test_dense_parity(cuda, n, box, lat0, zone):
    """Every ordered pair and the default form against the oracle: flight-level traffic at 52 N with the default zone, and
    with other zones in the southern hemisphere, across the equator, at high latitudes and next to the pole."""
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    zone = ZONES[zone]
    s = synth_airspace(n, box_deg=box, seed=n, lat0=lat0)
    stats = {}
    for kw in (dict(cull=False, symmetric=False), dict()):             # every ordered pair / the default (culled + symmetric) form
        g = StateBasedCD(rpz=zone[0], hpz=zone[1], dtlookahead=zone[2]).detect(*s, **kw)
        n_exempt, n_conf = _check_against_oracle(s, g, stats=stats, zone=zone)
        assert g["n_conf"] == len(g["confpairs"]) == len(g["tcpa"])
        assert n_exempt <= max(2, n_conf // 200), (n_exempt, n_conf)       # the band must stay a rarity
        assert stats["n_los_exempt"] <= max(2, stats["n_los"] // 100)
    print(f"N={n} at {lat0} N, zone {zone}: {n_conf} conflicts ({n_exempt} banded), {stats['n_los']} LoS pairs ({stats['n_los_exempt']} banded); max |error| "
          + ", ".join(f"{k} {stats[k]:.3g}" for k in ("qdr", "dist", "dcpa", "tcpa", "tinconf")))


def test_empty_and_single(cuda):
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    cd = StateBasedCD()
    e = cd.detect(*[np.zeros(0)] * 6)
    assert e["n_conf"] == 0 and e["confpairs"].shape == (0, 2)
    one = cd.detect(np.array([52.0]), np.array([4.0]), np.array([90.0]), np.array([200.0]), np.array([9000.0]), np.array([0.0]))
    assert one["n_conf"] == 0 and one["n_los"] == 0 and not one["inconf"][0] and one["tcpamax"][0] == 0.0


def test_known_geometry(cuda):
    """Head-on pair on a parallel: closed-form tcpa; co-located altitude-separated pair: no conflict."""
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    lat = np.array([0.0, 0.0, 10.0, 10.0])
    lon = np.array([0.0, 1.0, 0.0, 0.0])
    trk = np.array([90.0, 270.0, 0.0, 0.0])
    gs = np.array([200.0, 200.0, 200.0, 200.0])
    alt = np.array([9000.0, 9000.0, 5000.0, 5000.0 + 2 * HPZ])
    vs = np.zeros(4)
    g = StateBasedCD().detect(lat, lon, trk, gs, alt, vs)
    assert g["confpairs"].tolist() == [[0, 1], [1, 0]]                 # row-major, like upstream's np.where
    d = 6371000.0 * np.radians(1.0)
    assert abs(g["tcpamax"][0] - d / 400.0) < 0.05
    assert list(g["inconf"]) == [True, True, False, False]
    assert g["n_los"] == 0 and g["lospairs"].shape == (0, 2)
    # attributes of the two conflicts: bearing east / west, distance of one degree of longitude on the equator,
    # closest approach 0, entry into the zone (d - rpz) / 400 s from now
    np.testing.assert_allclose(g["qdr"], [90.0, 270.0], atol=1e-3)
    np.testing.assert_allclose(g["dist"], [d, d], rtol=1e-6)
    np.testing.assert_allclose(g["dcpa"], [0.0, 0.0], atol=1.0)
    np.testing.assert_allclose(g["tcpa"], [d / 400.0] * 2, atol=0.05)
    np.testing.assert_allclose(g["tinconf"], [(d - RPZ) / 400.0] * 2, atol=0.05)
    # two aircraft inside each other's zone: one LoS pair in each order
    lat2, lon2 = np.array([52.0, 52.02]), np.array([4.0, 4.0])
    g2 = StateBasedCD().detect(lat2, lon2, np.array([90.0, 90.0]), np.array([200.0, 210.0]), np.array([9000.0, 9100.0]), np.zeros(2))
    assert g2["lospairs"].tolist() == [[0, 1], [1, 0]] and g2["n_los"] == 2


def test_lon_wrap(cuda):
    """Pairs straddling the antimeridian: (lon + 180) % 360 - 180 differences."""
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    s = list(synth_airspace(600, box_deg=3.0, seed=5, lat0=10.0, lon0=179.9))
    s[1] = (s[1] + 180.0) % 360.0 - 180.0
    g = StateBasedCD().detect(*s, lon0=0.0)        # origin far away -> the wrap path is taken
    _check_against_oracle(tuple(s), g, lon0=0.0)


def test_row_shards_union(cuda):
    """Multi-GPU decomposition on one device: union of per-shard results == the full detection."""
    import torch
    from bluesky_gym_sasha_b200.cd import StateBasedCD, shard_rows
    n = 2048
    s = synth_airspace(n, box_deg=5.0, seed=3)
    cd = StateBasedCD()
    full = cd.detect(*s, lat0=52.0, lon0=4.0)
    rec, _ = cd.pack(*s, 52.0, 4.0)
    pairs, nconf = set(), np.zeros(n, dtype=np.int64)
    for rank in range(4):
        r0, nr = shard_rows(n, 4, rank)
        out = cd.detect_packed(rec, n, row0=r0, n_rows=nr)
        torch.cuda.synchronize()
        k = int(out["npairs"][0])
        p = out["pairs"][:k].cpu().numpy()
        assert ((p[:, 0] >= r0) & (p[:, 0] < r0 + nr)).all()
        pairs |= set(map(tuple, p.tolist()))
        nconf[r0:r0 + nr] = out["nconf_row"].cpu().numpy()
    assert pairs == set(map(tuple, full["confpairs"].tolist()))
    assert np.array_equal(nconf, full["nconf_row"])


def test_full_size_sampled_rows(cuda):
    """BASELINE config 5 size (N = 100k): sampled rows against the C restatement + size-independent
    properties (symmetry of the conflict relation, sum of row counts == pair-list length)."""
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    n = 100_000
    s = synth_airspace(n, box_deg=40.0, seed=1)
    g = StateBasedCD(pair_capacity=1 << 22).detect(*s, lat0=52.0, lon0=4.0)
    assert not g["truncated"]
    assert g["nconf_row"].sum() == g["n_conf"] == len(g["confpairs"])
    ps = set(map(tuple, g["confpairs"].tolist()))
    asym = [p for p in ps if (p[1], p[0]) not in ps]
    assert len(asym) <= max(2, len(ps) // 500)         # uniform zones => symmetric up to the epsilon band
    assert g["nlos_row"].sum() == g["n_los"] == len(g["lospairs"])
    ls = set(map(tuple, g["lospairs"].tolist()))
    assert len([p for p in ls if (p[1], p[0]) not in ls]) <= max(2, len(ls) // 200)       # LoS is symmetric
    conf_of, los_of = {}, {}
    for i, j in g["confpairs"].tolist():
        conf_of.setdefault(i, set()).add(j)
    for i, j in g["lospairs"].tolist():
        los_of.setdefault(i, set()).add(j)
    # sampled rows: every row that has a LoS pair (they are few) + 48 random ones, as SETS against the C restatement
    rows = sorted(set(np.random.default_rng(0).choice(n, 48, replace=False).tolist()) | set(list(los_of)[:64]))
    n_los_rows = 0
    for r in rows:
        c = cbind.detect_rows(*s, RPZ, HPZ, DTL, row0=int(r), nrows=1, pair_cap=4096)
        oc = {int(j) for _, j in c["confpairs"].tolist()}
        ol = {int(j) for _, j in c["lospairs"].tolist()}
        n_los_rows += bool(ol)
        if oc != conf_of.get(r, set()) or ol != los_of.get(r, set()):
            o = statebased.detect_rows(np.array([r]), *s, RPZ, HPZ, DTL, with_margins=True)
            assert all(o["near_conf"][0, j] for j in oc ^ conf_of.get(r, set())), f"row {r}: conflict sets differ outside the band"
            assert all(o["near_los"][0, j] for j in ol ^ los_of.get(r, set())), f"row {r}: LoS sets differ outside the band"
    assert n_los_rows > 0 or g["n_los"] == 0


@pytest.mark.parametrize("n,box,seed", [(20000, 40.0, 3), (5000, 3.0, 4), (1, 1.0, 5), (257, 60.0, 6), (40001, 25.0, 7)])
def test_culled_form_is_identical_to_plain(cuda, n, box, seed):
    """bsg_cd_detect_culled (Z-order sorted records, tile culling) == bsg_cd_detect: same conflict pair set, same
    per-aircraft counts / flags, bit-identical tcpamax -- culling only skips tile pairs that cannot interact."""
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    s = synth_airspace(n, box_deg=box, seed=seed)
    cd = StateBasedCD(device=0, pair_capacity=1 << 22)
    plain = cd.detect(*s, cull=False, symmetric=False)
    culled = cd.detect(*s, cull=True, symmetric=False)
    assert plain["n_conf"] == culled["n_conf"] and plain["n_los"] == culled["n_los"]
    assert np.array_equal(plain["confpairs"], culled["confpairs"]) and np.array_equal(plain["lospairs"], culled["lospairs"])
    for k in ("qdr", "dist", "dcpa", "tcpa", "tinconf"):          # the same exact routine decides in every form
        assert np.array_equal(plain[k], culled[k]), k
    assert np.array_equal(plain["nconf_row"], culled["nconf_row"]) and np.array_equal(plain["nlos_row"], culled["nlos_row"])
    assert np.array_equal(plain["inconf"], culled["inconf"])
    assert np.array_equal(plain["tcpamax"], culled["tcpamax"])
    if n >= 5000:
        assert plain["n_conf"] > 0
    # BSG_CD_SYMMETRIC: each unordered tile pair once, both ordered results emitted -- with and without culling
    for kw in (dict(symmetric=True), dict(symmetric=True, cull=True)):
        sym = cd.detect(*s, **kw)
        assert plain["n_conf"] == sym["n_conf"] and plain["n_los"] == sym["n_los"], kw
        assert np.array_equal(plain["confpairs"], sym["confpairs"]) and np.array_equal(plain["lospairs"], sym["lospairs"]), kw
        for k in ("qdr", "dist", "dcpa", "tcpa", "tinconf"):
            assert np.array_equal(plain[k], sym[k]), (kw, k)
        assert np.array_equal(plain["nconf_row"], sym["nconf_row"]) and np.array_equal(plain["nlos_row"], sym["nlos_row"]), kw
        assert np.array_equal(plain["inconf"], sym["inconf"]) and np.array_equal(plain["tcpamax"], sym["tcpamax"]), kw


def test_culled_form_against_oracle(cuda):
    """and directly against the float64 oracle (dense), like the plain form."""
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    s = synth_airspace(3000, box_deg=12.0, seed=11)
    g = StateBasedCD(device=0).detect(*s, cull=True, symmetric=False)
    n_exempt, n_pairs = _check_against_oracle(s, g)
    assert n_pairs > 50 and n_exempt <= max(2, n_pairs // 50)


def test_cull_fraction_and_speed(cuda):
    """N = 100k in the 40 x 40 degree box of SURVEY 8d: the culled form evaluates a few percent of the tile pairs."""
    import torch
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    n = 100_000
    s = synth_airspace(n, box_deg=40.0, seed=1, alt_jitter=0.0)
    cd = StateBasedCD(device=0)
    lat_d, lon_d = cd._as_dev(s[0]), cd._as_dev(s[1])
    perm = cd.spatial_order(lat_d, lon_d)
    rec, _ = cd.pack(*[cd._as_dev(x)[perm] for x in s], 52.0, 4.0)
    out = {}
    for cull in (False, True):
        for _ in range(2):
            o = cd.detect_packed(rec, n, cull=cull)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        o = cd.detect_packed(rec, n, cull=cull)
        e1.record()
        torch.cuda.synchronize()
        out[cull] = (e0.elapsed_time(e1), int(o["npairs"][0]), int(o["npairs"][1]), o["nconf_row"].clone())
    n_tiles = (n + 255) // 256
    work = cd._buf["cull_work"]
    cnt_off = 16 * ((n_tiles * 12 * 4 + 15) // 16)          # workspace layout: bounds | list_cnt | ...
    cnt = work[cnt_off:cnt_off + 4 * n_tiles].view(torch.int32).cpu().numpy()
    frac = cnt.sum() / float(n_tiles * n_tiles)
    print(f"plain {out[False][0]:.2f} ms, culled {out[True][0]:.3f} ms, tile pairs evaluated {100 * frac:.2f} %, "
          f"{out[True][1]} conflicts")
    assert out[False][1:3] == out[True][1:3] and torch.equal(out[False][3], out[True][3])
    assert frac < 0.15 and out[True][0] < 0.35 * out[False][0]


@pytest.mark.parametrize("cull", [False, True])
def test_peer_form_equals_gathered_form(cuda, cull):
    """bsg_cd_detect_peers with the blocks left in separate buffers (here: four buffers on one device standing in for
    four GPUs' symmetric memory) == bsg_cd_detect on the gathered records, for every 'rank'."""
    import ctypes as C
    import torch
    from bluesky_gym_sasha_b200 import _lib
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    W, per = 4, 1024
    n = W * per
    s = synth_airspace(n, box_deg=14.0, seed=21)
    cd = StateBasedCD(device=0)
    d = [cd._as_dev(x) for x in s]
    perm = cd.spatial_order(d[0], d[1])
    d = [x[perm] for x in d]
    rec_all, _ = cd.pack(*d, 52.0, 4.0)
    blocks = [rec_all[r * per // 256:(r + 1) * per // 256].clone() for r in range(W)]       # separate allocations
    ptrs = (C.c_void_p * W)(*[b.data_ptr() for b in blocks])
    lib = _lib.load()
    tot = 0
    for r in range(W):
        ref = cd.detect_packed(rec_all, n, row0=r * per, n_rows=per, cull=cull)
        ref = {k: (v.clone() if v is not None else None) for k, v in ref.items()}
        nconf = torch.zeros(per, dtype=torch.int32, device="cuda")
        nlos = torch.zeros(per, dtype=torch.int32, device="cuda")
        tmax = torch.zeros(per, dtype=torch.float32, device="cuda")
        inconf = torch.zeros(per, dtype=torch.uint8, device="cuda")
        npairs = torch.zeros(2, dtype=torch.int64, device="cuda")
        pairs = torch.zeros((1 << 16, 2), dtype=torch.int32, device="cuda")
        los = torch.zeros((1 << 12, 2), dtype=torch.int32, device="cuda")
        lists = _lib.CdLists(d_conf_pairs=pairs.data_ptr(), d_conf_attr=None, conf_cap=1 << 16, d_los_pairs=los.data_ptr(),
                             los_cap=1 << 12, d_npairs=npairs.data_ptr())
        nbytes = int(lib.bsg_cd_cull_workspace(n, per))
        work = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
        _lib.check(lib.bsg_cd_detect_peers(ptrs, W, r, per, RPZ, HPZ, DTL, _lib.CD_CULL if cull else 0, nconf.data_ptr(),
                                           nlos.data_ptr(), tmax.data_ptr(), inconf.data_ptr(), C.byref(lists),
                                           work.data_ptr(), nbytes, None))
        torch.cuda.synchronize()
        assert torch.equal(nconf, ref["nconf_row"]) and torch.equal(nlos, ref["nlos_row"]) and torch.equal(tmax, ref["tcpamax"])
        k = int(npairs[0])
        assert k == int(ref["npairs"][0])
        assert set(map(tuple, pairs[:k].tolist())) == set(map(tuple, ref["pairs"][:k].tolist()))
        kl = int(npairs[1])
        assert kl == int(ref["npairs"][1]) and set(map(tuple, los[:kl].tolist())) == set(map(tuple, ref["lospairs"][:kl].tolist()))
        tot += k
    assert tot > 100


def test_pack_ordered_is_a_spatial_permutation(cuda):
    """bsg_cd_pack_ordered: the order chosen on the device is a permutation, the records are bsg_cd_pack of the permuted
    aircraft bit for bit, the culled detection on them evaluates a few percent of the tile pairs (as with the exactly sorted
    order of ``spatial_order``) and finds the same conflicts as the plain form on the caller's order; ragged and tiny sizes."""
    import torch
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    cd = StateBasedCD(device=0)
    for n, box in ((100_000, 40.0), (4097, 3.0), (300, 1.0), (1, 1.0), (2, 0.0)):
        s = synth_airspace(n, box_deg=box, seed=3, alt_jitter=0.0)
        rec, _, perm = cd.pack_ordered(*s, 52.0, 4.0)
        torch.cuda.synchronize()
        p = perm.cpu().numpy()
        assert np.array_equal(np.sort(p), np.arange(n)), n
        ref, _ = cd.pack(*[np.asarray(x)[p] for x in s], 52.0, 4.0)
        assert torch.equal(rec, ref), n
        plain, _ = cd.pack(*s, 52.0, 4.0)
        a = cd.detect_packed(plain, n, cull=False)
        a_n = (int(a["npairs"][0]), int(a["npairs"][1]))
        a_rows = a["nconf_row"].cpu().numpy().copy()
        b = cd.detect_packed(rec, n, cull=True, symmetric=True)
        assert (int(b["npairs"][0]), int(b["npairs"][1])) == a_n, n
        back = np.empty(n, dtype=np.int64)
        back[p] = b["nconf_row"].cpu().numpy()
        assert np.array_equal(back, a_rows), n
        if n == 100_000:
            b = cd.detect_packed(rec, n, cull=True)
            n_tiles = (n + 255) // 256
            cnt_off = 16 * ((n_tiles * 12 * 4 + 15) // 16)
            cnt = cd._buf["cull_work"][cnt_off:cnt_off + 4 * n_tiles].view(torch.int32).cpu().numpy()
            frac = cnt.sum() / float(n_tiles * n_tiles)
            print(f"device order: {100 * frac:.2f} % of the tile pairs evaluated")
            assert frac < 0.06


@pytest.mark.parametrize("cull", [False, True])
def test_symmetric_form_dealt_over_ranks_adds_up(cuda, cull):
    """BSG_CD_DEAL: the row blocks of the symmetric form dealt round-robin to n GPUs (emulated here one after the other on
    one GPU): the per-aircraft counts and the pair totals of the shares add up to the undealt result, tcpamax is the maximum
    over the shares, and the shares are balanced (the lists shrink with the row index)."""
    import torch
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    n = 20_000
    s = synth_airspace(n, box_deg=12.0, seed=5, alt_jitter=0.0)
    cd = StateBasedCD(device=0)
    rec, _, _ = cd.pack_ordered(*s, 52.0, 4.0)
    full = cd.detect_packed(rec, n, cull=cull, symmetric=True)
    ref = {k: full[k].clone() for k in ("nconf_row", "nlos_row", "tcpamax", "npairs")}
    assert int(ref["npairs"][0]) > 1000
    for world in (2, 3, 8):
        nconf = torch.zeros_like(ref["nconf_row"])
        nlos = torch.zeros_like(ref["nlos_row"])
        tmax = torch.zeros_like(ref["tcpamax"])
        npairs = torch.zeros_like(ref["npairs"])
        share = []
        for rank in range(world):
            o = cd.detect_packed(rec, n, cull=cull, symmetric=True, deal=(world, rank))
            nconf += o["nconf_row"]
            nlos += o["nlos_row"]
            tmax = torch.maximum(tmax, o["tcpamax"])
            npairs += o["npairs"]
            share.append(int(o["npairs"][0]))
        assert torch.equal(nconf, ref["nconf_row"]) and torch.equal(nlos, ref["nlos_row"]), (cull, world)
        assert torch.equal(tmax, ref["tcpamax"]) and torch.equal(npairs, ref["npairs"]), (cull, world)
        assert max(share) < 2.5 * (sum(share) / world) + 50, share
