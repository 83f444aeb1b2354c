"""Conflict and loss-of-separation events of an airspace (bsg_traf_events_update, AirspaceTraffic(events=True)) against
the float64 restatement of upstream's ConflictDetection.update bookkeeping in oracle/conflict_log.py.

CPU: the oracle on hand-written detection sequences; argument checks of the C entry point; no register spills in its kernels.
GPU: hand-fed pair lists through the C ABI, real detections of AirspaceTraffic at N = 1024 and N = 100k, and the tracker
leaving the simulation and the host untouched."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from oracle import geo
from oracle.conflict_log import ConflictLog
from tests.test_traffic_ext import dense_scenario, make_device

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NM = 1852.0


# ---------------------------------------------------------------------------------------------------- CPU: the oracle
def _fixed(d):
    """dist_fn for hand-written sequences: distance and |dalt| from a dict {(a, b): (d, dalt)}."""
    return lambda a, b: (np.array([d[(i, j)][0] for i, j in zip(a, b)]), np.array([d[(i, j)][1] for i, j in zip(a, b)]))


def test_oracle_one_orientation_and_both_orientations_are_one_event():
    o = ConflictLog()
    o.update([(3, 1)], [], 1)                       # one orientation only
    o.update([(1, 3), (3, 1)], [], 2)               # both: still the same event
    o.update([(1, 3), (1, 3)], [], 3)               # a duplicate row
    lg = o.log()
    assert lg["confpairs_all"].tolist() == [[1, 3]] and lg["conf_start"].tolist() == [1] and lg["conf_end"].tolist() == [-1]
    assert o.counts() == dict(nconf_total=1, nlos_total=0, nconf_active=1, nlos_active=0, truncated=0)


def test_oracle_leave_and_reenter_is_two_events():
    o = ConflictLog()
    for step, pairs in enumerate([[(0, 5)], [(5, 0)], [], [(0, 5)], [(0, 5), (2, 4)], []], start=1):
        o.update(pairs, [], step)
    lg = o.log()
    assert lg["confpairs_all"].tolist() == [[0, 5], [0, 5], [2, 4]]
    assert lg["conf_start"].tolist() == [1, 4, 5] and lg["conf_end"].tolist() == [3, 6, 6]
    assert o.counts()["nconf_total"] == 3 and o.counts()["nconf_active"] == 0


def test_oracle_conflict_and_los_events_are_separate_with_minima():
    o = ConflictLog()
    sev = [{(1, 2): (5000.0, 80.0)}, {(1, 2): (4200.0, 95.0)}, {(1, 2): (4600.0, 60.0)}]
    for step in range(3):
        o.update([(1, 2)], [(2, 1)], step + 1, dist_fn=_fixed(sev[step]))
    o.update([(1, 2)], [], 4, dist_fn=_fixed({}))
    lg = o.log()
    assert lg["confpairs_all"].tolist() == [[1, 2]] and lg["conf_end"].tolist() == [-1]
    assert lg["lospairs_all"].tolist() == [[1, 2]] and lg["los_start"].tolist() == [1] and lg["los_end"].tolist() == [4]
    assert lg["los_dmin"].tolist() == [4200.0] and lg["los_dalt_min"].tolist() == [60.0]      # minima of separate detections
    assert o.counts() == dict(nconf_total=1, nlos_total=1, nconf_active=1, nlos_active=0, truncated=0)


def test_oracle_log_order_and_truncation_count():
    o = ConflictLog()
    o.update([(9, 4), (2, 7)], [], 10)
    o.update([(9, 4), (2, 7), (0, 1)], [], 11, truncated=True)
    lg = o.log()
    assert lg["confpairs_all"].tolist() == [[2, 7], [4, 9], [0, 1]] and lg["conf_start"].tolist() == [10, 10, 11]
    assert (lg["conf_end"] == -1).all() and o.counts()["truncated"] == 1


# ---------------------------------------------------------------------------------------------------- CPU: the C entry point
def test_events_update_rejects_bad_arguments(lib):
    """Every inconsistent argument is refused with BSG_EINVAL and a message before any CUDA call (so this runs without a
    GPU); the ctypes mirror of bsg_traf_events has the library's size."""
    from bluesky_gym_sasha_b200 import _lib
    assert lib.bsg_abi_struct_size(9) == C.sizeof(_lib.TrafEvents)
    assert lib.bsg_traf_events_workspace(-1, 4) == 0 and lib.bsg_traf_events_workspace(1 << 28, 1) == 0
    nb = lib.bsg_traf_events_workspace(100, 60)
    assert nb >= 16 * 2 * 160 + 4 * 160
    fake = lambda k: C.c_void_p(0x100000 * k)       # never dereferenced: every case below fails validation first
    cases = [("ev", None, None, "null argument"), ("lists", None, None, "null argument"),
             ("lists", "d_npairs", None, "d_npairs"), ("lists", "conf_cap", -1, "capacities"),
             ("lists", "d_conf_pairs", None, "pair list"), ("lists", "d_los_pairs", None, "pair list"),
             ("rec", None, None, "d_rec"), ("ev", "d_prev", fake(1), "distinct"), ("ev", "d_cur", None, "distinct"),
             ("ev", "d_cur", C.c_void_p(0x100008), "aligned"), ("ev", "set_bytes", nb - 1, "set_bytes"),
             ("lists", "los_cap", 61, "set_bytes"), ("ev", "conf_log_cap", -3, "log capacities"),
             ("ev", "d_conf_log", None, "log with a capacity"), ("ev", "d_los_sev", None, "log with a capacity"),
             ("ev", "d_counters", None, "d_counters"), ("nstep", None, -1, "nstep"), ("nstep", None, 1 << 31, "nstep")]
    for what, field, value, msg in cases:
        a = dict(ev=_lib.TrafEvents(d_cur=fake(1), d_prev=fake(2), set_bytes=nb, d_conf_log=fake(3), d_los_log=fake(4),
                                    d_los_sev=fake(5), conf_log_cap=10, los_log_cap=10, d_counters=fake(6)),
                 lists=_lib.CdLists(d_conf_pairs=fake(7), d_conf_attr=None, conf_cap=100, d_los_pairs=fake(8), los_cap=60,
                                    d_npairs=fake(9)),
                 rec=fake(10), nstep=5)
        if field is None:
            a[what] = value
        else:
            setattr(a[what], field, value)
        ref = lambda st: C.byref(st) if st is not None else None
        rc = lib.bsg_traf_events_update(ref(a["ev"]), a["rec"], ref(a["lists"]), a["nstep"], None)
        assert rc == _lib.BSG_EINVAL, (what, field, rc)
        assert msg.encode() in lib.bsg_last_error(), (what, field, lib.bsg_last_error())


def test_event_kernels_compile_without_spills(tmp_path):
    """csrc/traf_events.cu builds for sm_100a and ptxas reports no local-memory spills in its kernels."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if shutil.which(nvcc) is None:
        pytest.skip("needs nvcc")
    from bluesky_gym_sasha_b200 import build
    src = os.path.join(ROOT, "bluesky_gym_sasha_b200", "csrc", "traf_events.cu")
    flags = [f for f in build.NVCC_FLAGS if f != "-shared"]
    r = subprocess.run([nvcc] + flags + ["-Xptxas", "-v", "-c", "-o", str(tmp_path / "traf_events.o"), src], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    out = r.stdout + r.stderr
    blocks = re.findall(r"Function properties for (\S*traf_ev_\w+)\s*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", out)
    assert len(blocks) == 2, out
    for name, _, st, ld in blocks:
        assert st == "0" and ld == "0", (name, st, ld)


def test_events_refused_for_a_sharded_airspace():
    """The sharded airspace keeps the two orders of a pair on different GPUs: events=True with a group is refused before
    the process group (or the device) is touched."""
    from bluesky_gym_sasha_b200.traffic import AirspaceTraffic
    with pytest.raises(ValueError, match="sharded"):
        AirspaceTraffic(1000, group=True, events=True)


# ---------------------------------------------------------------------------------------------------- GPU
def severity32(rec, a, b):
    """Float32 restatement of the device's LoS distance / |dalt| (cd_pair.cuh's algebra, every operation rounded in float32)
    from host copies of the CD records [tiles][8][256]."""
    f = lambda j, k: rec[j // 256, k, j % 256]
    cav = f(a, 2) * f(b, 2) - f(a, 3) * f(b, 3)
    dx = (f(b, 0) - f(a, 0)) * cav
    dy = f(b, 1) - f(a, 1)
    return np.sqrt(dx * dx + dy * dy), np.abs(f(b, 6) - f(a, 6))


def _compare(dev, ref, severity=True):
    for k in ("confpairs_all", "conf_start", "conf_end", "lospairs_all", "los_start", "los_end"):
        assert np.array_equal(np.asarray(dev[k], dtype=np.int64), ref[k]), k
    for k in ("nconf_total", "nlos_total", "nconf_active", "nlos_active", "truncated"):
        assert dev[k] == ref[k], (k, dev[k], ref[k])


@pytest.mark.gpu
def test_synthetic_lists_through_the_abi(cuda):
    """40 hand-fed detections through bsg_traf_events_update: random pair sets that persist, leave and come back, one or
    both orientations, duplicate rows, pairs with aircraft 0 and n - 1, pairs in both lists, and a last detection whose
    npairs exceeds the capacity.  Log, counters and truncation equal the oracle's; the LoS minima equal the float32
    restatement of the records bit for bit (records packed by bsg_traf_pack from a state that moves between detections)."""
    import torch
    from bluesky_gym_sasha_b200 import _lib
    from bluesky_gym_sasha_b200.cd import _ptr
    n, cap, log_cap = 600, 384, 4096
    g = make_device(dense_scenario(n, 4))
    lib, dev = g.lib, g.device
    rng = np.random.default_rng(11)
    pool = {(0, n - 1), (0, 5), (7, n - 1)}
    while len(pool) < 250:
        a, b = sorted(rng.choice(n, 2, replace=False).tolist())
        pool.add((a, b))
    pool = sorted(pool)
    conf_on, los_on = rng.random(len(pool)) < 0.3, rng.random(len(pool)) < 0.1
    nb = int(lib.bsg_traf_events_workspace(cap, cap))
    sets = [torch.zeros(nb, dtype=torch.uint8, device=dev) for _ in range(2)]
    t = dict(conf=torch.zeros((log_cap, 4), dtype=torch.int32, device=dev), los=torch.zeros((log_cap, 4), dtype=torch.int32, device=dev),
             sev=torch.zeros((log_cap, 2), dtype=torch.float32, device=dev), ctr=torch.zeros(_lib.EV_CTR_COUNT, dtype=torch.int64, device=dev),
             pairs=torch.zeros((cap, 2), dtype=torch.int32, device=dev), lospairs=torch.zeros((cap, 2), dtype=torch.int32, device=dev),
             npairs=torch.zeros(2, dtype=torch.int64, device=dev))
    ev = _lib.TrafEvents(set_bytes=nb, d_conf_log=_ptr(t["conf"]), d_los_log=_ptr(t["los"]), d_los_sev=_ptr(t["sev"]),
                         conf_log_cap=log_cap, los_log_cap=log_cap, d_counters=_ptr(t["ctr"]))
    lists = _lib.CdLists(d_conf_pairs=_ptr(t["pairs"]), d_conf_attr=None, conf_cap=cap, d_los_pairs=_ptr(t["lospairs"]), los_cap=cap,
                         d_npairs=_ptr(t["npairs"]))
    o = ConflictLog()

    def rows_of(on, p_both):
        rows = []
        for (a, b), x in zip(pool, on):
            if x:
                r = rng.random()
                rows += [(a, b), (b, a)] if r < p_both else [(a, b)] if r < 0.5 + 0.5 * p_both else [(b, a)]
                if rng.random() < 0.05:
                    rows.append(rows[-1])                  # a duplicate row
        rng.shuffle(rows)
        return rows
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    for det in range(40):
        g.step(1, detect=False)                            # the traffic moves: every detection sees other records
        _lib.check(lib.bsg_traf_pack(C.byref(g.cfg), C.byref(g.tt), _ptr(g.rec), st))
        conf_on = np.where(conf_on, rng.random(len(pool)) < 0.8, rng.random(len(pool)) < 0.15)
        los_on = np.where(los_on, rng.random(len(pool)) < 0.7, rng.random(len(pool)) < 0.08)
        if det == 39:
            conf_on[:] = True                              # more rows than the list holds
        rc, rl = rows_of(conf_on, 0.2 if det < 39 else 1.0), rows_of(los_on, 0.2)
        assert det < 39 or len(rc) > cap
        kc, kl = min(len(rc), cap), min(len(rl), cap)
        if kc:
            t["pairs"][:kc] = torch.as_tensor(np.array(rc[:kc], dtype=np.int32), device=dev)
        if kl:
            t["lospairs"][:kl] = torch.as_tensor(np.array(rl[:kl], dtype=np.int32), device=dev)
        t["npairs"].copy_(torch.tensor([len(rc), len(rl)]))
        ev.d_cur, ev.d_prev = _ptr(sets[det % 2]), _ptr(sets[1 - det % 2])
        _lib.check(lib.bsg_traf_events_update(C.byref(ev), _ptr(g.rec), C.byref(lists), g.nstep, st))
        rec = g.rec.cpu().numpy()
        o.update(rc[:kc], rl[:kl], g.nstep, dist_fn=lambda a, b: severity32(rec, a, b), truncated=len(rc) > cap or len(rl) > cap)
    ref = o.log()
    ctr = t["ctr"].cpu().numpy()
    m, k = int(ctr[_lib.EV_CTR_NCONF_TOTAL]), int(ctr[_lib.EV_CTR_NLOS_TOTAL])
    conf, los, sev = t["conf"][:m].cpu().numpy(), t["los"][:k].cpu().numpy(), t["sev"][:k].cpu().numpy()
    oc, ol = np.lexsort((conf[:, 1], conf[:, 0], conf[:, 2])), np.lexsort((los[:, 1], los[:, 0], los[:, 2]))
    dev_log = dict(confpairs_all=conf[oc, :2], conf_start=conf[oc, 2], conf_end=conf[oc, 3], lospairs_all=los[ol, :2],
                   los_start=los[ol, 2], los_end=los[ol, 3], nconf_total=m, nlos_total=k,
                   nconf_active=int(ctr[_lib.EV_CTR_NCONF_ACTIVE]), nlos_active=int(ctr[_lib.EV_CTR_NLOS_ACTIVE]),
                   truncated=int(ctr[_lib.EV_CTR_TRUNCATED]))
    _compare(dev_log, ref)
    assert ref["truncated"] == 1 and int(ctr[_lib.EV_CTR_LOG_OVERFLOW]) == 0
    assert np.array_equal(sev[ol, 0], ref["los_dmin"].astype(np.float32)) and np.array_equal(sev[ol, 1], ref["los_dalt_min"].astype(np.float32))
    ends = ref["conf_end"]
    print(f"synthetic: {m} conflict events ({int((ends >= 0).sum())} ended), {k} LoS events over 40 detections")
    assert m > 250 and k > 40 and (ends >= 0).sum() > 100                   # the sequence exercised starts, ends and re-entries


def _kwik(lat, lon, alt):
    return lambda a, b: (geo.kwikdist(lat[a], lon[a], lat[b], lon[b]) * NM, np.abs(alt[a] - alt[b]))


@pytest.mark.gpu
@pytest.mark.parametrize("reso", ["MVP", None])
def test_real_detections_match_oracle(cuda, reso):
    """dense_scenario(1024, 2), 240 substeps: after every substep the host copy of conflicts() goes into the oracle.
    Pairs, starts, ends and totals are identical; the LoS minima are within 1 m (0.01 m for |dalt|) of the float64 kwik
    distance of the state each detection saw.  (Under MVP conflicts come and go: some 15 000 events, more than the default
    log of 8 x n_max rows.)"""
    g = make_device(dense_scenario(1024, 2), reso=reso, reso_mode=1, vnav=False, events=True, event_capacity=1 << 15)
    o = ConflictLog()
    for _ in range(240):
        lat, lon, alt = g.lat.cpu().numpy(), g.lon.cpu().numpy(), g.altitude.cpu().numpy().astype(np.float64)
        g.step(1)
        c = g.conflicts()
        o.update(c["confpairs"], c["lospairs"], g.nstep, dist_fn=_kwik(lat, lon, alt), truncated=c["truncated"])
    dev, ref = g.conflict_log(), o.log()
    _compare(dev, ref)
    assert dev["log_overflow"] == 0
    if ref["nlos_total"]:
        assert np.abs(dev["los_dmin"] - ref["los_dmin"]).max() < 1.0
        assert np.abs(dev["los_dalt_min"] - ref["los_dalt_min"]).max() < 0.01
    print(f"reso {reso}: {ref['nconf_total']} conflicts, {ref['nlos_total']} LoS over 240 s; "
          f"max |dmin - kwik| {np.abs(dev['los_dmin'] - ref['los_dmin']).max() if ref['nlos_total'] else 0:.3f} m")
    assert ref["nconf_total"] > 300 and (reso or ref["nlos_total"] > 20)


@pytest.mark.gpu
def test_tracking_only_reads(cuda):
    """The same airspace with and without events for 100 substeps: the state is bit-identical.  Left out: ``partners``
    and the resopair overflow counter.  Which of an aircraft's conflicts take its 8 resopair slots (and which overflow)
    follows the order in which atomics scatter the conflict index, with or without events; the kinematics and commands
    do not depend on that order."""
    import torch
    sc = dense_scenario(1024, 2)
    def run(events):
        g = make_device(sc, reso="MVP", reso_mode=1, vnav=False, events=events)
        g.step(100)
        torch.cuda.synchronize()
        out = {k: v.cpu() for k, v in g.t.items() if k != "partners"}
        out["counters"] = out["counters"][1:]          # [0] = BSG_TRAF_CTR_OVERFLOW
        return out
    on, off = run(True), run(False)
    for k in off:
        assert torch.equal(on[k], off[k]), k


def bench_airspace(n, events=False, event_capacity=None):
    """bench.py::bench_traffic's airspace: n aircraft over 40 x 40 deg in spatially coherent order, four-waypoint routes
    with altitude constraints under VNAV, MVP (horizontal)."""
    import torch
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    from bluesky_gym_sasha_b200.traffic import AirspaceTraffic
    rng = np.random.default_rng(3)
    lat, lon = 52 + 40 * (rng.random(n) - 0.5), 4 + 40 * (rng.random(n) - 0.5)
    dev = torch.device("cuda", 0)
    perm = StateBasedCD.spatial_order(torch.as_tensor(lat, device=dev), torch.as_tensor(lon, device=dev)).cpu().numpy()
    lat, lon = lat[perm], lon[perm]
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
    tr = AirspaceTraffic(n, device=0, simdt=1.0, reso="MVP", reso_mode=1, max_wpts=W, events=events, event_capacity=event_capacity)
    tr.create(lat, lon, hdg, alt, cas)
    tr.set_routes(np.arange(n), wlat, wlon, walt, None)
    return tr


@pytest.mark.gpu
def test_scale_100k_without_host_sync(cuda):
    """bench_traffic's airspace at N = 100 000: 20 substeps one at a time against the oracle fed with conflicts() (identical
    log and totals, default log large enough), then 20 more substeps that must not synchronise the host."""
    import torch
    g = bench_airspace(100_000, events=True)
    o = ConflictLog()
    for _ in range(20):
        g.step(1)
        c = g.conflicts()
        o.update(c["confpairs"], c["lospairs"], g.nstep, truncated=c["truncated"])
    dev, ref = g.conflict_log(), o.log()
    _compare(dev, ref)
    assert dev["log_overflow"] == 0 and dev["truncated"] == 0
    torch.cuda.set_sync_debug_mode("error")
    try:
        g.step(20)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    after = g.conflict_counts()
    print(f"N = 100k: {ref['nconf_total']} conflicts, {ref['nlos_total']} LoS in 20 substeps ({ref['nconf_active']} open); "
          f"after 40 substeps {after}")
    assert after["nconf_total"] >= ref["nconf_total"] and after["log_overflow"] == 0


@pytest.mark.gpu
def test_log_capacity_and_truncation(cuda):
    """A tiny event log overflows while the totals stay exact; tiny pair lists set the truncation counter."""
    sc = dense_scenario(1024, 2)
    g = make_device(sc, vnav=False, events=True, event_capacity=16)
    o = ConflictLog()
    for _ in range(30):
        g.step(1)
        c = g.conflicts()
        o.update(c["confpairs"], c["lospairs"], g.nstep)
    dev, ref = g.conflict_log(), o.log()
    for k in ("nconf_total", "nlos_total", "nconf_active", "nlos_active"):
        assert dev[k] == ref[k], k
    assert dev["log_overflow"] == max(0, ref["nconf_total"] - 16) + max(0, ref["nlos_total"] - 16) > 0
    rows = lambda d, p: set(map(tuple, np.column_stack([d[p + "pairs_all"], d[p + "_start"], d[p + "_end"]]).tolist()))
    assert len(dev["confpairs_all"]) == 16 and rows(dev, "conf") <= rows(ref, "conf")     # the logged events are right
    assert rows(dev, "los") <= rows(ref, "los")
    t = make_device(sc, vnav=False, events=True, pair_capacity=64)
    want = 0
    for _ in range(5):
        t.step(1)
        want += int(t.conflicts()["truncated"])
    assert want > 0 and t.conflict_counts()["truncated"] == want


@pytest.mark.gpu
def test_mvp_reduces_los_events(cuda):
    """What the feature is for: the number of LoS events over 240 s of dense traffic, with MVP against without, next to
    the pair-samples figure tests/test_traffic_ext.py uses (sum of npairs[1] every 20th substep)."""
    n = 1024
    sc = dense_scenario(n, 2)
    order = np.lexsort((sc["lon"], np.floor((sc["lat"] - 48.0) / 1.0)))
    sc = {k: (v[order] if isinstance(v, np.ndarray) and v.shape[0] == n else v) for k, v in sc.items()}
    def run(reso):
        g = make_device(sc, reso=reso, reso_mode=1, vnav=False, events=True)
        sampled = 0
        for _ in range(12):
            g.step(20)
            sampled += int(g.last["npairs"][1])
        return g.conflict_counts(), sampled
    (off, s_off), (on, s_on) = run(None), run("MVP")
    print(f"LoS events over 240 s: {off['nlos_total']} without resolution, {on['nlos_total']} with MVP "
          f"(conflicts {off['nconf_total']} / {on['nconf_total']}; LoS pair-samples every 20th substep {s_off} / {s_on})")
    assert on["nlos_total"] < off["nlos_total"]
