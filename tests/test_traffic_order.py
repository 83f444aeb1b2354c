"""AirspaceTraffic(reorder_dt=...): the culled detection on records in a spatial order kept on the device
(bsg_traf_pack_ordered, bsg_cd_unpermute).

CPU: argument checks of the two C entry points and of the constructor; no register spills in the new kernels.
GPU: an ordered airspace steps bit for bit like the same airspace without ordering (state, conflicts, events); the ordered
records are the aircraft-order records permuted; bsg_cd_unpermute on hand-made lists; and the tile pairs the culling keeps
(cd_cull_kernel's test restated in numpy) on randomly created and long-flown airspaces."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest


ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NM, FT = 1852.0, 0.3048


# ---------------------------------------------------------------------------------------------------- CPU
def _traf_structs(n=1000, fake=lambda k: C.c_void_p(0x100000 * k)):
    from bluesky_gym_sasha_b200 import _lib
    cfg = _lib.TrafConfig(n=n, max_wpts=4, simdt=1.0)
    t = _lib.TrafTensors(**{name: fake(k + 1) for k, (name, _) in enumerate(_lib.TrafTensors._fields_)})
    return cfg, t


def test_pack_ordered_rejects_bad_arguments(lib):
    """Every inconsistent argument of bsg_traf_pack_ordered is refused with BSG_EINVAL and a message before any CUDA call
    (so this runs without a GPU)."""
    from bluesky_gym_sasha_b200 import _lib
    fake = lambda k: C.c_void_p(0x100000 * k)       # never dereferenced: every case below fails validation first
    nb = lib.bsg_traf_order_workspace(1000)
    assert nb >= 4 * 1000 and lib.bsg_traf_order_workspace(2000) - nb == 4 * 1000
    cases = [("cfg", None, None, "null argument"), ("t", None, None, "null argument"), ("n", -1, None, "n out of range"),
             ("n", 1 << 31, None, "n out of range"), ("t", "pos", None, "tensor pointer is null"),
             ("row0", 256, None, "sharded"), ("perm", None, None, "d_perm"), ("rec_ordered", None, None, "d_rec_ordered"),
             ("work", None, None, "workspace too small"), ("work_bytes", nb - 1, None, "workspace too small"),
             ("work", C.c_void_p(0x100004), None, "aligned")]
    for what, value, _, msg in cases:
        cfg, t = _traf_structs(1000)
        a = dict(cfg=C.byref(cfg), t=C.byref(t), perm=fake(20), rec_ordered=fake(21), rec=fake(22), work=fake(23), work_bytes=nb)
        if what == "n":
            cfg.n = value
        elif what == "row0":
            cfg.row0 = value
        elif what == "t" and value is not None:
            setattr(t, value, None)
        else:
            a[what] = value
        rc = lib.bsg_traf_pack_ordered(a["cfg"], a["t"], 1, a["perm"], a["rec_ordered"], a["rec"], a["work"], a["work_bytes"], None)
        assert rc == _lib.BSG_EINVAL, (what, value, rc)
        assert msg.encode() in lib.bsg_last_error(), (what, value, lib.bsg_last_error())


def test_unpermute_rejects_bad_arguments(lib):
    """bsg_cd_unpermute refuses negative or too large n, a missing permutation, half a per-row pair, a per-row output that
    aliases its input, lists without their count and negative capacities, before any CUDA call."""
    from bluesky_gym_sasha_b200 import _lib
    fake = lambda k: C.c_void_p(0x100000 * k)
    cases = [("n", -1, "n must be"), ("n", 1 << 31, "n must be"), ("perm", None, "d_perm"), ("nconf_out", None, "both"),
             ("tcpamax_in", None, "both"), ("inconf_out", "alias", "distinct"), ("d_npairs", None, "d_npairs"),
             ("conf_cap", -1, "capacities")]
    for what, value, msg in cases:
        lists = _lib.CdLists(d_conf_pairs=fake(1), d_conf_attr=fake(2), conf_cap=100, d_los_pairs=fake(3), los_cap=50, d_npairs=fake(4))
        a = dict(perm=fake(5), n=1000, nconf_in=fake(6), nlos_in=fake(7), tcpamax_in=fake(8), inconf_in=fake(9),
                 nconf_out=fake(10), nlos_out=fake(11), tcpamax_out=fake(12), inconf_out=fake(13))
        if what in ("d_npairs", "conf_cap"):
            setattr(lists, what, value)
        elif value == "alias":
            a[what] = a["inconf_in"]
        else:
            a[what] = value
        rc = lib.bsg_cd_unpermute(a["perm"], a["n"], C.byref(lists), a["nconf_in"], a["nlos_in"], a["tcpamax_in"], a["inconf_in"],
                                  a["nconf_out"], a["nlos_out"], a["tcpamax_out"], a["inconf_out"], None)
        assert rc == _lib.BSG_EINVAL, (what, value, rc)
        assert msg.encode() in lib.bsg_last_error(), (what, value, lib.bsg_last_error())
    # nothing to do is not an error, and touches no device
    assert lib.bsg_cd_unpermute(None, 0, None, None, None, None, None, None, None, None, None, None) == _lib.BSG_OK


@pytest.mark.parametrize("src, pattern, count", [("cd_order.cu", r"order_\w+|cd_unpermute_kernel\w*", 8),
                                                 ("traf_airspace.cu", r"traf_pack\w*", 2)])
def test_order_kernels_compile_without_spills(tmp_path, src, pattern, count):
    """The order, unpermute and pack kernels build for sm_100a and ptxas reports no local-memory spills in them."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if shutil.which(nvcc) is None:
        pytest.skip("needs nvcc")
    from bluesky_gym_sasha_b200 import build
    path = os.path.join(ROOT, "bluesky_gym_sasha_b200", "csrc", src)
    flags = [f for f in build.NVCC_FLAGS if f != "-shared"]
    r = subprocess.run([nvcc] + flags + ["-Xptxas", "-v", "-c", "-o", str(tmp_path / "k.o"), path], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    out = r.stdout + r.stderr
    blocks = re.findall(r"Function properties for (\S*(?:%s))\s*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                        r"(\d+) bytes spill loads" % pattern, out)
    assert len(blocks) == count, out
    for name, _, st, ld in blocks:
        assert st == "0" and ld == "0", (name, st, ld)


def test_airspace_reorder_argument_errors():
    """reorder_dt is refused with a sharded airspace, without the culled detection and when not > 0, before the device or
    a process group is touched."""
    from bluesky_gym_sasha_b200.traffic import AirspaceTraffic
    with pytest.raises(ValueError, match="sharded"):
        AirspaceTraffic(1000, group=True, reorder_dt=30.0)
    with pytest.raises(ValueError, match="cull=True"):
        AirspaceTraffic(1000, cull=False, reorder_dt=30.0)
    for bad in (0.0, -5.0, float("nan")):
        with pytest.raises(ValueError, match="> 0"):
            AirspaceTraffic(1000, reorder_dt=bad)


# ---------------------------------------------------------------------------------------------------- helpers
def bench_draws(n, seed=3):
    """bench.py::bench_traffic's airspace draws (40 x 40 deg around (52, 4), four-waypoint routes with altitude constraints),
    in the order drawn: spatially random."""
    rng = np.random.default_rng(seed)
    lat, lon = 52 + 40 * (rng.random(n) - 0.5), 4 + 40 * (rng.random(n) - 0.5)
    alt = np.round(rng.uniform(3000, 12000, n) / 304.8) * 304.8
    hdg, cas = rng.uniform(0, 360, n), rng.uniform(120, 150, n)
    W = 4
    wlat, wlon, walt = np.zeros((n, W)), np.zeros((n, W)), np.full((n, W), -999.0)
    la, lo, brg = lat.copy(), lon.copy(), hdg.copy()
    for k in range(W):
        d = rng.uniform(60.0, 120.0, n) / 111.0
        la = la + d * np.cos(np.radians(brg)); lo = lo + d * np.sin(np.radians(brg)) / np.cos(np.radians(np.clip(la, -80, 80)))
        brg = brg + rng.uniform(-40, 40, n)
        wlat[:, k], wlon[:, k] = la, lo
        walt[:, k] = np.where(rng.random(n) < 0.5, np.clip(alt + rng.uniform(-2500, 1500, n), 1500, 12000), -999.0)
    return dict(lat=lat, lon=lon, hdg=hdg, alt=alt, cas=cas, wlat=wlat, wlon=wlon, walt=walt)


def bench_like_airspace(n, sorted_creation=True, reorder_dt=None, routes=True, reso="MVP", **kw):
    """bench_traffic's airspace, created in spatially coherent order (``StateBasedCD.spatial_order``, as bench.py does) or
    in the random order of the draws."""
    import torch
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    from bluesky_gym_sasha_b200.traffic import AirspaceTraffic
    d = bench_draws(n)
    if sorted_creation:
        dev = torch.device("cuda", 0)
        p = StateBasedCD.spatial_order(torch.as_tensor(d["lat"], device=dev), torch.as_tensor(d["lon"], device=dev)).cpu().numpy()
        d = {k: v[p] for k, v in d.items()}
    tr = AirspaceTraffic(n, device=0, simdt=1.0, reso=reso, reso_mode=1, max_wpts=4, reorder_dt=reorder_dt, **kw)
    tr.create(d["lat"], d["lon"], d["hdg"], d["alt"], d["cas"])
    if routes:
        tr.set_routes(np.arange(n), d["wlat"], d["wlon"], d["walt"], None)
    return tr


def kept_fraction(rec, n, symmetric=True, rpz=5.0 * NM, hpz=1000.0 * FT, T=300.0):
    """cd_cull_kernel's keep test restated in numpy over the tile bounds of cd_tile_bounds_kernel (float32, records of
    index >= n ignored): the fraction of (row block, column tile) pairs the culled detection evaluates."""
    r = rec.cpu().numpy() if hasattr(rec, "cpu") else np.asarray(rec)
    nt = -(-n // 256)
    r = r[:nt].transpose(0, 2, 1).reshape(nt * 256, 8)          # record j = r[j]
    live = (np.arange(nt * 256) < n).reshape(nt, 256)
    f = lambda c: r[:, c].reshape(nt, 256)
    x, y, ch, sh, u, v, alt, vs = (f(c) for c in range(8))
    big = np.float32(3.0e38)
    mn = lambda a: np.where(live, a, big).min(1)
    mx = lambda a, lo: np.where(live, a, lo).max(1)
    cosmin = np.where(live, ch * ch - sh * sh, np.float32(1.0)).min(1)
    vmax = mx(np.sqrt(u * u + v * v), np.float32(0.0))
    B = dict(x0=mn(x), x1=mx(x, -big), y0=mn(y), y1=mx(y, -big), c=cosmin, v=vmax, a0=mn(alt), a1=mx(alt, -big),
             s=mx(np.abs(vs), np.float32(0.0)))
    i, j = np.triu_indices(nt) if symmetric else np.indices((nt, nt)).reshape(2, -1)
    f32 = np.float32
    gx = np.maximum(f32(0), np.maximum(B["x0"][j] - B["x1"][i], B["x0"][i] - B["x1"][j]))
    gy = np.maximum(f32(0), np.maximum(B["y0"][j] - B["y1"][i], B["y0"][i] - B["y1"][j]))
    cmin = np.maximum(f32(0), np.minimum(B["c"][i], B["c"][j]) - f32(1e-6))
    dmin = np.sqrt((gx * cmin) ** 2 + gy * gy)
    reach = f32(rpz * 1.001 + 1.0) + (B["v"][i] + B["v"][j]) * f32((T + 0.05) * 1.0001)
    ga = np.maximum(f32(0), np.maximum(B["a0"][j] - B["a1"][i], B["a0"][i] - B["a1"][j]))
    vreach = f32(hpz * 1.001 + 0.1) + (B["s"][i] + B["s"][j]) * f32((T + 0.05) * 1.0001)
    return float(((dmin <= reach) & (ga <= vreach)).mean())


def _host_records(rec, n):
    """[bsg_cd_padded(n), 8] host view of tile-blocked records: row j = record j."""
    r = rec.cpu().numpy()
    return r.transpose(0, 2, 1).reshape(-1, 8)


# ---------------------------------------------------------------------------------------------------- GPU
STATE = ("pos", "kin", "cmd", "aux", "actwp", "vnav1", "vnav2", "asas", "flags", "counters")


def _assert_same(a, b, where):
    import torch
    torch.cuda.synchronize()
    n = a.n
    for k in STATE:
        x, y = a.t[k], b.t[k]
        if k != "counters":
            x, y = x[:n], y[:n]
        assert torch.equal(x.view(torch.uint8) if x.dtype.is_floating_point else x,
                           y.view(torch.uint8) if y.dtype.is_floating_point else y), (where, k)
    pa, pb = a.t["partners"][:n].cpu().numpy(), b.t["partners"][:n].cpu().numpy()
    assert np.array_equal(np.sort(pa, axis=1), np.sort(pb, axis=1)), (where, "partners")
    assert a.counters() == b.counters(), where
    ca, cb = a.conflicts(), b.conflicts()
    assert ca.keys() == cb.keys()
    for k in ca:
        va, vb = np.ascontiguousarray(ca[k]), np.ascontiguousarray(cb[k])
        assert va.dtype == vb.dtype and np.array_equal(va.view(np.uint8) if va.dtype.kind == "f" else va,
                                                       vb.view(np.uint8) if vb.dtype.kind == "f" else vb), (where, k)
    assert not ca["truncated"], where
    assert a.conflict_counts() == b.conflict_counts(), where
    la, lb = a.conflict_log(), b.conflict_log()
    for k in la:
        assert np.array_equal(np.asarray(la[k]), np.asarray(lb[k])), (where, k)
    return ca


@pytest.mark.gpu
def test_ordered_airspace_is_bit_identical(cuda):
    """20 000 aircraft of bench.py's airspace created in random order with four-waypoint VNAV routes, MVP and event
    tracking, one airspace with reorder_dt = 30 s and one without, over 600 substeps: 2000 more aircraft created at substep
    100 (forcing a fresh order), HDG and ALT commands at 200.  State, counters, conflicts and the event log are identical
    at every checkpoint.  (The airspace is sparse enough that no aircraft has more resopairs than its BSG_TRAF_PARTNERS
    slots: which ones an overflowing aircraft keeps follows the list order, in either airspace.)"""
    from bluesky_gym_sasha_b200.traffic import AirspaceTraffic
    n0, n1 = 20000, 2000
    d = bench_draws(n0 + n1, seed=11)
    air = [AirspaceTraffic(n0 + n1, simdt=1.0, reso="MVP", max_wpts=4, events=True, pair_capacity=1 << 20, reorder_dt=rd)
           for rd in (30.0, None)]

    def add(g, s):
        r = g.create(d["lat"][s], d["lon"][s], d["hdg"][s], d["alt"][s], d["cas"][s])
        g.set_routes(np.arange(r.start, r.stop), d["wlat"][s], d["wlon"][s], d["walt"][s], None)

    for g in air:
        add(g, slice(0, n0))
    rng = np.random.default_rng(5)
    cmd_idx = rng.choice(n0 + n1, 3000, replace=False)
    hdg_new, alt_new = rng.uniform(0, 360, 1500), rng.integers(20, 38, 1500) * 1000.0 * FT
    checkpoints = {1, 29, 30, 31, 100, 101, 150, 201, 300, 450, 600}
    seen = 0
    for step in range(1, 601):
        if step == 101:
            for g in air:
                add(g, slice(n0, n0 + n1))
        if step == 201:
            for g in air:
                g.hdg(cmd_idx[:1500], hdg_new)
                g.alt(cmd_idx[1500:], alt_new)
        for g in air:
            g.step(1)
        if step in checkpoints:
            assert air[1].counters()["resopair_overflow"] == 0, step
            c = _assert_same(air[0], air[1], step)
            seen = max(seen, c["n_conf"])
    counts = air[0].conflict_counts()
    print(f"ordered vs unordered airspace: identical at {len(checkpoints)} checkpoints; up to {seen} conflict pairs per "
          f"detection; events {counts}; counters {air[0].counters()}")
    assert seen > 1000 and counts["nconf_total"] > 1000 and counts["nlos_total"] > 0 and counts["truncated"] == 0


@pytest.mark.gpu
def test_record_order_and_records(cuda):
    """record_order is a permutation of range(n); the ordered records are the aircraft-order records permuted, bit for bit,
    after a fresh order and after a reused one (padding inert); bsg_traf_pack_ordered accepts d_rec = NULL."""
    import torch
    from bluesky_gym_sasha_b200 import _lib
    from bluesky_gym_sasha_b200.cd import _ptr
    n = 5000
    g = bench_like_airspace(n, sorted_creation=False, reorder_dt=10.0)
    assert g.reorder_freq == 10
    perms = []
    for step in range(1, 13):
        g.step(1)
        torch.cuda.synchronize()
        p = g.record_order.cpu().numpy()
        assert np.array_equal(np.sort(p), np.arange(n)), step
        perms.append(p)
        ro, ra = _host_records(g.rec_ordered, n), _host_records(g.rec, n)
        assert np.array_equal(ro[:n].view(np.uint32), ra[p].view(np.uint32)), step
        assert (ro[n:, 6] == 3.0e9).all() and (ro[n:, 2] == 1.0).all() and (ro[n:, [0, 1, 3, 4, 5, 7]] == 0).all()
    for k in range(1, 9):                               # steps 2..9 reuse the order of the first detection
        assert np.array_equal(perms[k], perms[0]), k
    assert not np.array_equal(perms[9], perms[0])      # step 10: a fresh order of positions that moved
    # the aircraft-order records are those of bsg_traf_pack
    ref = torch.empty_like(g.rec)
    st = g._stream()
    ordered_before = g.rec_ordered.clone()
    _lib.check(g.lib.bsg_traf_pack(C.byref(g.cfg), C.byref(g.tt), _ptr(ref), st))
    _lib.check(g.lib.bsg_traf_pack_ordered(C.byref(g.cfg), C.byref(g.tt), 0, _ptr(g.perm), _ptr(g.rec_ordered), None,
                                           _ptr(g.order_work), g.order_work.numel(), st))
    torch.cuda.synchronize()
    p = g.record_order.cpu().numpy()
    ro, rr = _host_records(g.rec_ordered, n), _host_records(ref, n)
    assert np.array_equal(ro[:n].view(np.uint32), rr[p].view(np.uint32))
    assert not torch.equal(ordered_before, g.rec_ordered)      # the state moved since the last substep's pack


@pytest.mark.gpu
def test_unpermute_hand_made_lists(cuda):
    """bsg_cd_unpermute against a numpy mapping: the conflict list holds more pairs than its capacity (every row mapped),
    the LoS list fewer (rows past the count untouched); per-row outputs scattered; NULL per-row pointers skipped."""
    import torch
    from bluesky_gym_sasha_b200 import _lib
    from bluesky_gym_sasha_b200.cd import _ptr
    lib = _lib.load()
    dev = cuda
    rng = np.random.default_rng(1)
    n, ccap, lcap = 3000, 500, 400
    perm = rng.permutation(n).astype(np.int32)
    conf = rng.integers(0, n, (ccap, 2)).astype(np.int32)
    los = rng.integers(0, n, (lcap, 2)).astype(np.int32)
    npairs = np.array([ccap + 123, 77], dtype=np.uint64)
    nconf, nlos = rng.integers(0, 9, n).astype(np.int32), rng.integers(0, 9, n).astype(np.int32)
    tcp, inc = rng.random(n).astype(np.float32), rng.integers(0, 2, n).astype(np.uint8)
    d = lambda a: torch.as_tensor(a, device=dev)
    dconf, dlos, dnp = d(conf), d(los), d(npairs.astype(np.int64))
    ins = [d(nconf), d(nlos), d(tcp), d(inc)]
    outs = [torch.full((n,), -1, dtype=torch.int32, device=dev), None, torch.zeros(n, dtype=torch.float32, device=dev),
            torch.zeros(n, dtype=torch.uint8, device=dev)]
    ins[1] = None                                    # nlos not wanted
    lists = _lib.CdLists(d_conf_pairs=_ptr(dconf), d_conf_attr=None, conf_cap=ccap, d_los_pairs=_ptr(dlos), los_cap=lcap,
                         d_npairs=_ptr(dnp))
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(lib.bsg_cd_unpermute(_ptr(d(perm)), n, C.byref(lists), *[_ptr(t) for t in ins], *[_ptr(t) for t in outs], st))
    torch.cuda.synchronize()
    assert np.array_equal(dconf.cpu().numpy(), perm[conf])
    want_los = los.copy()
    want_los[:77] = perm[los[:77]]
    assert np.array_equal(dlos.cpu().numpy(), want_los)
    for got, src in ((outs[0], nconf), (outs[2], tcp), (outs[3], inc)):
        want = np.empty_like(src)
        want[perm] = src
        assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.gpu
def test_culling_restored_on_random_creation(cuda):
    """bench.py's 100k airspace created in random order: the aircraft-order records keep (nearly) every tile pair, the
    ordered records about as few as the same airspace created sorted."""
    rnd = bench_like_airspace(100_000, sorted_creation=False, reorder_dt=60.0)
    srt = bench_like_airspace(100_000, sorted_creation=True)
    rnd.step(1)
    srt.step(1)
    f_plain, f_ord, f_sorted = (kept_fraction(r, 100_000) for r in (rnd.rec, rnd.rec_ordered, srt.rec))
    print(f"kept tile pairs at t = 0: random creation {f_plain:.2%}, its spatial order {f_ord:.2%}, sorted creation {f_sorted:.2%}")
    assert f_plain >= 0.90
    assert f_ord <= 1.5 * f_sorted


@pytest.mark.gpu
def test_culling_holds_over_flight_time(cuda):
    """1800 substeps of the sorted 100k airspace: with reorder_dt = 60 the kept fraction stays near its t = 0 value, while
    the unordered twin's records spread (each tile's box grows by about 2 x speed x time)."""
    on = bench_like_airspace(100_000, sorted_creation=True, reorder_dt=60.0)
    off = bench_like_airspace(100_000, sorted_creation=True)
    on.step(1)
    off.step(1)
    f_on0, f_off0 = kept_fraction(on.rec_ordered, 100_000), kept_fraction(off.rec, 100_000)
    on.step(1799)
    off.step(1799)
    f_on, f_off = kept_fraction(on.rec_ordered, 100_000), kept_fraction(off.rec, 100_000)
    print(f"kept tile pairs, t = 0 -> 1800 s: ordered {f_on0:.2%} -> {f_on:.2%}, unordered {f_off0:.2%} -> {f_off:.2%}")
    assert f_on <= 1.5 * f_on0
    assert f_off >= 3.0 * f_off0
