"""K1/K3/K4/K5/K6 parity: the batched env step (through the C ABI) against the float64 oracle envs.

Two families, per SURVEY.md section 0.6:
  * state injection -- the oracle env is reset with the *reference's* draw source (global np.random /
    random, seeded), its post-reset state is loaded into the device sim, and both are stepped with the
    same actions: trajectories, observations, rewards and termination flags must agree;
  * device reset -- the device's Philox-keyed scenario generator against the oracle env driven by the
    same Philox stream (oracle/philox.py).
Tolerances (float32 kernels vs float64 oracle; stated here as the north_star requires) -- those SURVEY.md section 8c
proposed or tighter, with the largest differences observed on a B200 over the whole suite in brackets (the parity tests
print them per run: "max |error|"):
  lat/lon 1e-5 deg = 1 m [4.9e-6; MergeEnv's LNAV-guided intruders 2e-5 (1.2e-5)], alt 0.1 m [0.049], tas 2e-3 m/s [6.4e-4],
  vs 1e-3 m/s [4.8e-7], hdg 1e-3 deg [4.8e-4], observations 2e-4 (1 + |value|) [8.4e-5 (1 + |value|)],
  reward 1e-4 [2.5e-6]; DescentEnv / VerticalCREnv 1e-3 [7.9e-4: the terminal reward is altitude * 50 / 3000],
  terminated / truncated sequences identical.
"""
import random

import numpy as np
import pytest

from bluesky_gym_sasha_b200 import _lib
from oracle import envs as oenvs
from oracle import geo as ogeo
from oracle.philox import PhiloxDraws
from tests.common import angdiff, device_traffic, inject_oracle_env

pytestmark = pytest.mark.gpu

TOL = dict(pos=1e-5, alt=0.1, tas=2e-3, vs=1e-3, hdg=1e-3)
OBS_TOL = 2e-4


def pos_tol(env_id):
    return 2.0 * TOL["pos"] if env_id == "MergeEnv-v0" else TOL["pos"]      # (LNAV: bearings to a waypoint feed back)


def reward_tol(env_id):
    return 1e-3 if env_id in ("DescentEnv-v0", "VerticalCREnv-v0") else 1e-4


class ErrStats:
    """Largest observed |device - oracle| per quantity (printed by the parity tests: the evidence behind the tolerances)."""

    def __init__(self):
        self.m = {}

    def add(self, name, err):
        err = float(np.max(err)) if np.size(err) else 0.0
        if np.isfinite(err):
            self.m[name] = max(self.m.get(name, 0.0), err)

    def __str__(self):
        return ", ".join(f"{k} {v:.3g}" for k, v in sorted(self.m.items()))


def _make_oracle(env_id, draws=None, cd=False, n_int=5, density="normal", init_alt=0.0):
    if env_id == "HorizontalCREnv-v0":
        return oenvs.HorizontalCREnv(n_intruders=n_int, draws=draws, cd_enabled=cd, init_alt=init_alt)
    if env_id == "DescentEnv-v0":
        return oenvs.DescentEnv(draws=draws)
    if env_id == "SectorCREnv-v0":
        return oenvs.SectorCREnv(draws=draws, cd_enabled=cd, ac_density_mode=density)
    if env_id == "PlanWaypointEnv-v0":
        return oenvs.PlanWaypointEnv(draws=draws)
    if env_id == "VerticalCREnv-v0":
        return oenvs.VerticalCREnv(draws=draws, cd_enabled=cd)
    if env_id == "StaticObstacleEnv-v0":
        return oenvs.StaticObstacleEnv(draws=draws)
    return oenvs.MergeEnv(draws=draws, cd_enabled=cd)


def _inject(venv, e, oenv, env_id):
    t = oenv.traf
    for cmd in t.queue:             # MergeEnv: the queued addwpt/dest run at the start of the first sim step
        cmd()
    t.queue = []
    f64, i32, poly, f32 = {}, {}, None, {}
    if env_id == "HorizontalCREnv-v0":
        f64 = {_lib.F64_WPT_LAT: oenv.wpt_lat, _lib.F64_WPT_LON: oenv.wpt_lon}
    elif env_id in ("DescentEnv-v0", "VerticalCREnv-v0"):
        f64 = {_lib.F64_TARGET_ALT: float(oenv.target_alt)}
    elif env_id == "PlanWaypointEnv-v0":
        f64 = {}
        for k in range(5):
            f64[_lib.F64_WPTS + 2 * k] = oenv.wpt_lat[k]
            f64[_lib.F64_WPTS + 2 * k + 1] = oenv.wpt_lon[k]
    elif env_id == "SectorCREnv-v0":
        w = ogeo.nm_to_latlong(oenvs.SECTOR_CENTER, oenv.wpts[0])
        f64 = {_lib.F64_WPT_LAT: float(w[0]), _lib.F64_WPT_LON: float(w[1])}
        i32 = {_lib.I32_NVERT: len(oenv.poly_lat)}
        poly = np.stack([oenv.poly_lat, oenv.poly_lon], axis=1).reshape(-1)
    elif env_id == "StaticObstacleEnv-v0":
        f64 = {_lib.F64_WPT_LAT: oenv.wpt_lat, _lib.F64_WPT_LON: oenv.wpt_lon}
        f32 = {_lib.F32_LAST_WDIST: oenv.wpt_dis_km, _lib.F32_LAST_DRIFT: oenv.drift}
        poly = np.zeros(360)
        for k, v in enumerate(oenv.obstacle_vertices):
            poly[k * 32:k * 32 + 2 * len(v)] = np.asarray(v).reshape(-1)
            poly[350 + k] = len(v)
        poly[320:340] = np.stack([oenv.obstacle_centre_lat, oenv.obstacle_centre_lon], axis=1).reshape(-1)
        poly[340:350] = oenv.obstacle_radius
    inject_oracle_env(venv, e, oenv, extra_f64=f64, extra_i32=i32, poly=poly, extra_f32=f32)


def _compare_traffic(venv, oracles, alive_mask, step, exempt=None, stats=None):
    d = device_traffic(venv)
    for e, o in enumerate(oracles):
        if not alive_mask[e]:
            continue
        t = o.traf
        n = t.ntraf
        ok = np.ones(n, dtype=bool)
        if exempt is not None and exempt[e]:
            ok[list(exempt[e])] = False
        # an FMS-guided aircraft that overflew a waypoint steered for a few substeps along a bearing to a
        # point metres away (see hdg_tol below): its track keeps a lateral offset of a few metres
        base = pos_tol(venv.env_id)
        pos_tol_ = np.where(np.asarray(t.iactwp) >= 1, 5.0 * base, base)
        assert np.all((np.abs(d["lat"][e, :n] - t.lat) < pos_tol_)[ok]), (step, e, "lat")
        assert np.all((np.abs(d["lon"][e, :n] - t.lon) < pos_tol_)[ok]), (step, e, "lon")
        assert np.max(np.abs(d["alt"][e, :n] - t.alt)[ok]) < TOL["alt"], (step, e, "alt")
        assert np.max(np.abs(d["tas"][e, :n] - t.tas)[ok]) < TOL["tas"], (step, e, "tas")
        assert np.max(np.abs(d["vs"][e, :n] - t.vs)[ok]) < TOL["vs"], (step, e, "vs")
        # an LNAV aircraft steers along the bearing to its active waypoint: a bearing to a point D metres
        # away, computed from a position that is only known to the stated 2 m, is uncertain by 2 m / D
        d2wp = np.asarray(ogeo.kwikdist(t.lat, t.lon, t.actwp_lat, t.actwp_lon)) * 1852.0
        hdg_tol = TOL["hdg"] + np.where(t.swlnav, np.degrees(2.0 / np.maximum(d2wp, 1.0)) * 3.0, 0.0)
        assert np.all((angdiff(d["hdg"][e, :n], t.hdg) < hdg_tol)[ok]), (step, e, "hdg", angdiff(d["hdg"][e, :n], t.hdg).max())
        if stats is not None and ok.any():
            plain = ok & (np.asarray(t.iactwp) < 1)                # (aircraft past a waypoint carry the documented offset)
            if plain.any():
                stats.add("pos_deg", np.maximum(np.abs(d["lat"][e, :n] - t.lat), np.abs(d["lon"][e, :n] - t.lon))[plain])
            stats.add("alt_m", np.abs(d["alt"][e, :n] - t.alt)[ok])
            stats.add("tas", np.abs(d["tas"][e, :n] - t.tas)[ok])
            stats.add("vs", np.abs(d["vs"][e, :n] - t.vs)[ok])
            stats.add("hdg_deg", angdiff(d["hdg"][e, :n], t.hdg)[ok & ~t.swlnav])


def _compare_asas_pairs(g, t, where):
    """In-sim ASAS pair lists of one env (``BlueSkyVectorEnv.asas_pairs``) against the oracle traffic's last detection:
    conflict and LoS pair SETS identical outside the epsilon band of SURVEY 8c, and qdr / dist / dcpa / tcpa / tinconf of
    every common conflict (same tolerances as tests/test_gpu_cd.py).  Returns the number of conflicts compared."""
    assert not g["truncated"], where
    gp, op = set(map(tuple, g["confpairs"].tolist())), set(t.confpairs)
    gl, ol = set(map(tuple, g["lospairs"].tolist())), set(t.lospairs)
    if gp != op or gl != ol:
        near_conf, near_los = t.near_band()
        assert all(near_conf[i, j] for i, j in gp ^ op), (where, "confpairs", sorted(gp ^ op))
        assert all(near_los[i, j] for i, j in gl ^ ol), (where, "lospairs", sorted(gl ^ ol))
    o_idx = {p: k for k, p in enumerate(t.confpairs)}
    n = 0
    for k, p in enumerate(map(tuple, g["confpairs"].tolist())):
        if p not in o_idx:
            continue
        q = o_idx[p]
        dist, dcpa, tcpa, tin = t.cd_dist[q], t.cd_dcpa[q], t.cd_tcpa[q], t.cd_tinconf[q]
        if abs(dcpa * dcpa - t.rpz ** 2) / t.rpz ** 2 < 1e-3:
            continue                                            # near-banded: the entry time is a square root near zero
        # The device evaluates ITS OWN float32 traffic state, which follows the oracle's within the trajectory tolerances
        # (TOL: 2 m in position, 2e-2 m/s per velocity component): the attributes inherit that -- a relative velocity known
        # to dv = 4e-2 m/s out of vrel turns into tcpa * dv / vrel seconds and dist * dv / vrel metres of closest approach
        i, j = p
        _, _, trk_, gs_, _, _ = t._cd_inputs                      # the traffic state the last detection saw
        vrel = max(np.hypot(gs_[j] * np.sin(np.radians(trk_[j])) - gs_[i] * np.sin(np.radians(trk_[i])),
                            gs_[j] * np.cos(np.radians(trk_[j])) - gs_[i] * np.cos(np.radians(trk_[i]))), 1e-3)
        rel = 2.0 * TOL["tas"] / vrel + 1e-4
        dpos = 2.0 * TOL["pos"] * 111e3
        timed = vrel > 0.5        # (two aircraft on the same track at the same speed: closest approach is 0 / 0, any time goes)
        assert abs((g["qdr"][k] - t.cd_qdr[q] + 180.0) % 360.0 - 180.0) < 2e-3 + np.degrees(dpos / max(dist, 1.0)), (where, p, "qdr")
        assert abs(g["dist"][k] - dist) < dpos + 1e-5 * dist, (where, p, "dist")
        half = abs(tcpa - tin)
        if timed:
            assert abs(g["dcpa"][k] - dcpa) < 2.0 * dpos + rel * max(dist, dcpa), (where, p, "dcpa", g["dcpa"][k], dcpa)
            assert abs(g["tcpa"][k] - tcpa) < 0.05 + dpos / vrel + rel * abs(tcpa), (where, p, "tcpa", g["tcpa"][k], tcpa)
            assert abs(g["tinconf"][k] - tin) < 0.05 + dpos / vrel + rel * (abs(tin) + abs(tcpa)) + 0.05 * half, (where, p, "tinconf", g["tinconf"][k], tin)
        n += 1
    return n


def _compare_tcpamax(g_tcpamax, t, where, dev_hdg=None, dev_tas=None):
    """Per-aircraft tcpamax (max of tcpa over the aircraft's conflicts) against the oracle's.  A time to closest approach is
    distance over closing speed: with the device's own float32 traffic state following the oracle's within TOL it is known
    to 2 TOL_pos / vrel + tcpa * dv / vrel, dv = how far the two aircraft's velocity vectors are from the oracle's --
    2 TOL_tas by default, or measured from the device state when given (a MergeEnv intruder turning over a waypoint
    carries a larger heading difference for a few substeps, see _compare_traffic).  Slowly converging pairs (two MergeEnv
    intruders on almost the same track: vrel of a few m/s, tcpa of thousands of seconds) inherit percents, not 1e-3."""
    _, _, trk_, gs_, _, _ = t._cd_inputs
    u, v = gs_ * np.sin(np.radians(trk_)), gs_ * np.cos(np.radians(trk_))
    verr = np.full(t.ntraf, TOL["tas"])
    if dev_hdg is not None:
        du = dev_tas * np.sin(np.radians(dev_hdg)) - t.tas * np.sin(np.radians(t.hdg))
        dv = dev_tas * np.cos(np.radians(dev_hdg)) - t.tas * np.cos(np.radians(t.hdg))
        verr = np.maximum(verr, 2.0 * np.hypot(du, dv))
    tol = np.full(t.ntraf, 0.05)
    for (i, j), tc in zip(t.confpairs, t.cd_tcpa):
        vrel = max(np.hypot(u[j] - u[i], v[j] - v[i]), 1e-3)
        if vrel < 0.5:            # same track, same speed: the time of closest approach is 0 / 0
            tol[i] = np.inf
        tol[i] = max(tol[i], 0.05 + 2.0 * TOL["pos"] * 111e3 / vrel + abs(tc) * ((verr[i] + verr[j]) / vrel + 1e-3))
    assert np.all(np.abs(g_tcpamax - t.tcpamax) <= tol), (where, "tcpamax", g_tcpamax, t.tcpamax, tol)


OWNSHIP_KEYS = ("cos(drift)", "sin(drift)", "airspeed", "waypoint_dist", "faf_reached")


def _compare_obs(gobs, oobs, e, step, vnorm=None, ownship_only=False, stats=None):
    for k, v in oobs.items():
        if ownship_only and k not in OWNSHIP_KEYS:
            continue
        atol = OBS_TOL
        if stats is not None and k not in ("cos(track)", "sin(track)"):
            stats.add("obs", np.abs(gobs[k][e] - v) / (1.0 + np.abs(v)))
        if k in ("cos(track)", "sin(track)") and vnorm is not None:
            # direction of the relative velocity: ill-conditioned when the two aircraft fly almost the same
            # vector; allow the stated TAS tolerance (2e-2 m/s) divided by the relative speed
            dv = np.hypot(oobs["vx_r"] * vnorm[0], oobs["vy_r"] * vnorm[1])
            atol = OBS_TOL + 2.0 * TOL["tas"] / np.maximum(dv, 1e-3)
        assert np.all(np.abs(gobs[k][e] - v) <= atol + OBS_TOL * np.abs(v)), \
            f"step {step} env {e} key {k}: {gobs[k][e]} vs {v}"


@pytest.mark.parametrize("env_id,n_int,cd,steps", [
    ("DescentEnv-v0", 0, False, 45),
    ("HorizontalCREnv-v0", 5, False, 40),
    ("HorizontalCREnv-v0", 20, True, 25),
    ("HorizontalCREnv-v0", 12, True, 25),          # 16-lane groups (two-phase in-group CD with G = 16)
    ("HorizontalCREnv-v0", 31, True, 12),          # a full 32-aircraft group (even n: the doubled offset n/2)
    ("SectorCREnv-v0", 0, True, 40),
    ("MergeEnv-v0", 0, False, 50),
    ("MergeEnv-v0", 0, True, 50),                  # the configuration bench.py times (FMS-guided intruders + CD every substep)
    ("PlanWaypointEnv-v0", 0, False, 60),
    ("VerticalCREnv-v0", 0, True, 45),
    ("StaticObstacleEnv-v0", 0, False, 100),
])
def test_step_parity_injected_state(cuda, env_id, n_int, cd, steps):
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    E = 12
    np.random.seed(1234)
    random.seed(1234)
    kw = dict(n_intruders=n_int) if n_int else {}
    venv = BlueSkyVectorEnv(env_id, E, seed=7, cd_enabled=cd, autoreset_mode="disabled", max_episode_steps=0, cd_pairs=cd, **kw)
    venv.reset()
    oracles = [_make_oracle(env_id, cd=cd, n_int=n_int) for _ in range(E)]
    o_obs = [o.reset()[0] for o in oracles]
    for e, o in enumerate(oracles):
        _inject(venv, e, o, env_id)
    rng = np.random.default_rng(0)
    alive = np.ones(E, dtype=bool)
    act_dim = venv.layout.act_dim
    vnorm = {"SectorCREnv-v0": (32.0, 66.0), "MergeEnv-v0": (150.0, 150.0)}.get(env_id)
    # Exemption (SURVEY.md section 8c, "operand within epsilon of its threshold"): when an FMS-guided
    # aircraft overflies its LAST waypoint, LNAV switches off and freezes ap.trk at the bearing to a
    # point a few metres away -- a quantity with unbounded sensitivity to position.  From then on that
    # aircraft is excluded, and for its env only the ownship quantities are compared.  Counted below.
    exempt = [set() for _ in range(E)]
    compared_full = 0
    n_pairs_checked = 0
    stats = ErrStats()
    for step in range(steps):
        a = rng.uniform(-1.0, 1.0, size=(E, act_dim)).astype(np.float32)
        gobs, grew, gterm, gtrunc, ginfo = venv.step(a)
        for e, o in enumerate(oracles):
            if not alive[e]:
                continue
            lnav_before = o.traf.swlnav.copy()
            oobs, orew, oterm, otrunc, oinfo = o.step(a[e].astype(np.float64))
            exempt[e] |= set(np.where(lnav_before & ~o.traf.swlnav)[0].tolist())
            _compare_obs(gobs, oobs, e, step, vnorm, ownship_only=bool(exempt[e]), stats=stats)
            if exempt[e]:
                if oterm or otrunc:
                    alive[e] = False
                continue
            compared_full += 1
            assert abs(grew[e] - orew) < reward_tol(env_id), (step, e, grew[e], orew)
            stats.add("reward", abs(grew[e] - orew))
            assert bool(gterm[e]) == bool(oterm), (step, e, "terminated")
            assert bool(gtrunc[e]) == bool(otrunc), (step, e, "truncated")
            for k, v in oinfo.items():
                if not (isinstance(v, float) and np.isnan(v)):
                    assert abs(ginfo[k][e] - v) < 1e-2 + 1e-4 * abs(v), (step, e, k, ginfo[k][e], v)
            if cd:
                d = device_traffic(venv)
                t = o.traf
                # in-sim ASAS runs before the kinematics of the last substep; the oracle keeps those results
                assert ginfo["asas_nconf"][e] == len(t.confpairs), (step, e, "nconf", ginfo["asas_nconf"][e], len(t.confpairs))
                assert ginfo["asas_nlos"][e] == len(t.lospairs), (step, e, "nlos")
                assert np.array_equal(d["inconf"][e, :t.ntraf], t.inconf), (step, e, "inconf")
                _compare_tcpamax(d["tcpamax"][e, :t.ntraf], t, (step, e), d["hdg"][e, :t.ntraf], d["tas"][e, :t.ntraf])
                n_pairs_checked += _compare_asas_pairs(venv.asas_pairs(e), t, (step, e))
            if oterm or otrunc:
                alive[e] = False
        _compare_traffic(venv, oracles, alive, step, exempt, stats)
    n_ex = sum(1 for x in exempt if x)
    print(f"{env_id}: {compared_full} env-steps compared in full, {n_ex}/{E} envs ended with an exempted aircraft"
          + (f", {n_pairs_checked} in-sim ASAS conflict pairs compared with their attributes" if cd else "")
          + f"; max |error|: {stats}")
    if cd:
        assert n_pairs_checked > 0
    assert compared_full >= (steps * E) // 4
    if env_id != "MergeEnv-v0":
        assert n_ex == 0
    venv.close()


@pytest.mark.parametrize("env_id,n_int", [("DescentEnv-v0", 0), ("HorizontalCREnv-v0", 5), ("HorizontalCREnv-v0", 20),
                                          ("SectorCREnv-v0", 0), ("MergeEnv-v0", 0), ("PlanWaypointEnv-v0", 0),
                                          ("VerticalCREnv-v0", 0), ("StaticObstacleEnv-v0", 0), ("SectorCREnv-v0", -1)])
def test_device_reset_matches_philox_oracle(cuda, env_id, n_int):
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    E, seed, off = 16, 99, 1000
    kw = dict(n_intruders=n_int) if n_int > 0 else {}
    density = "uniform" if n_int < 0 else "normal"          # SectorCREnv(ac_density_mode=...), sector_cr_env.py:98-103
    if n_int < 0:
        kw["ac_density_mode"] = density
    venv = BlueSkyVectorEnv(env_id, E, seed=seed, env_id_offset=off, autoreset_mode="disabled", **kw)
    for episode in range(2):
        gobs, ginfo = venv.reset()
        d = device_traffic(venv)
        i32 = venv.t["env_i32"].cpu().numpy()
        for e in range(E):
            o = _make_oracle(env_id, draws=PhiloxDraws(seed, off + e, episode), n_int=n_int, density=density)
            oobs, _ = o.reset()
            t = o.traf
            n = t.ntraf
            assert i32[e, _lib.I32_NUM_AC] == n, (e, i32[e, _lib.I32_NUM_AC], n)
            assert np.max(np.abs(d["lat"][e, :n] - t.lat)) < 1e-9
            assert np.max(np.abs(d["lon"][e, :n] - t.lon)) < 1e-9
            assert np.max(np.abs(d["tas"][e, :n] - t.tas)) < 1e-3
            assert np.max(np.abs(d["alt"][e, :n] - t.alt)) < 1e-3
            assert np.max(angdiff(d["hdg"][e, :n], t.hdg)) < 1e-4
            assert (d["flags"][e, n:] == 0).all()
            _compare_obs(gobs, oobs, e, -1)
    venv.close()


def test_time_limit_and_autoreset_modes(cuda):
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    E = 8
    for mode in ("next_step", "same_step"):
        venv = BlueSkyVectorEnv("HorizontalCREnv-v0", E, seed=3, autoreset_mode=mode, max_episode_steps=4)
        venv.reset()
        a = np.zeros((E, 1), dtype=np.float32)
        for k in range(3):
            _, _, term, trunc, _ = venv.step(a)
            assert not trunc.any()
        obs4, r4, term, trunc, info4 = venv.step(a)
        assert trunc.all()                                         # TimeLimit: elapsed == cap
        ep = venv.t["env_i32"].cpu().numpy()[:, _lib.I32_EPISODE]
        if mode == "same_step":
            assert (ep == 2).all() and "final_obs" in info4        # already reset; terminal obs kept aside
            assert not np.allclose(info4["final_obs"]["waypoint_distance"], obs4["waypoint_distance"])
        else:
            assert (ep == 1).all()
            obs5, r5, term5, trunc5, _ = venv.step(a)              # NEXT_STEP: this call only resets
            assert (ep + 1 == venv.t["env_i32"].cpu().numpy()[:, _lib.I32_EPISODE]).all()
            assert (r5 == 0).all() and not term5.any() and not trunc5.any()
        venv.close()


def test_shard_invariance(cuda):
    """Env e's trajectory is a pure function of (seed, global env id): 1 x 16 envs == 2 x 8 envs."""
    import torch
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    kw = dict(seed=11, n_intruders=20, cd_enabled=True, autoreset_mode="same_step", max_episode_steps=6)
    full = BlueSkyVectorEnv("HorizontalCREnv-v0", 16, **kw)
    halves = [BlueSkyVectorEnv("HorizontalCREnv-v0", 8, env_id_offset=8 * r, **kw) for r in range(2)]
    full.reset_torch()
    [h.reset_torch() for h in halves]
    g = torch.Generator(device="cpu").manual_seed(0)
    for _ in range(15):
        a = (torch.rand((16, 1), generator=g) * 2 - 1).cuda()
        of, rf, tf, uf = full.step_torch(a)
        for r, h in enumerate(halves):
            oh, rh, th, uh = h.step_torch(a[8 * r:8 * r + 8])
            assert torch.equal(rf[8 * r:8 * r + 8], rh)
            assert torch.equal(full.t["obs"][8 * r:8 * r + 8], h.t["obs"])
            assert torch.equal(tf[8 * r:8 * r + 8], th) and torch.equal(uf[8 * r:8 * r + 8], uh)
    full.close()
    [h.close() for h in halves]


def test_scalar_env_api(cuda):
    """gym.make(id) -> reset/step with the reference's spaces, dtypes, info keys (horizontal_cr_env.py:49-62,215-223)."""
    import bluesky_gym
    bluesky_gym.register_envs()
    env = bluesky_gym.make("HorizontalCREnv-v0", render_mode=None)
    obs, info = env.reset()
    assert list(obs.keys()) == ["intruder_distance", "cos_difference_pos", "sin_difference_pos", "x_difference_speed",
                                "y_difference_speed", "waypoint_distance", "cos_drift", "sin_drift"]
    assert obs["intruder_distance"].shape == (5,) and obs["cos_drift"].shape == (1,)
    assert all(v.dtype == np.float64 for v in obs.values())
    assert set(info) >= {"total_reward", "total_intrusions", "average_drift"} and np.isnan(info["average_drift"])
    obs, r, term, trunc, info = env.step(env.action_space.sample())
    assert isinstance(r, float) and isinstance(term, bool) and isinstance(trunc, bool)
    for _ in range(300):
        obs, r, term, trunc, info = env.step(np.zeros(1))
        if term or trunc:
            break
    assert term or trunc
    env.close()


@pytest.mark.parametrize("env_id", ["DescentEnv-v0", "PlanWaypointEnv-v0", "HorizontalCREnv-v0", "VerticalCREnv-v0",
                                    "SectorCREnv-v0", "StaticObstacleEnv-v0", "MergeEnv-v0"])
def test_gym_make_every_registered_id(cuda, env_id):
    """bluesky_gym/__init__.py:6-46: every registered id is constructible through ``gym.make``, resets, and steps to the
    end of an episode (termination or the registration's TimeLimit) with observations inside the declared space."""
    import bluesky_gym
    import bluesky_gym.envs  # noqa: F401  (scripts/multi_processing_example.py:17)
    from bluesky_gym_sasha_b200.spec import SPECS
    bluesky_gym.register_envs()
    env = bluesky_gym.make(env_id, render_mode=None)
    obs, info = env.reset()
    space = env.observation_space
    assert list(obs.keys()) == list(space.keys())
    for k, v in obs.items():
        assert v.dtype == np.float64 and v.shape == space[k].shape, (env_id, k)
    assert set(info) >= set(SPECS[env_id].info_keys)
    rng = np.random.default_rng(0)
    cap = SPECS[env_id].max_episode_steps
    for t in range(cap + 1):
        obs, r, term, trunc, info = env.step(rng.uniform(-1, 1, env.action_space.shape))
        assert isinstance(r, float) and isinstance(term, bool) and isinstance(trunc, bool)
        assert all(np.all(np.isfinite(v)) for v in obs.values())
        if term or trunc:
            break
    assert (term or trunc) and t < cap
    obs2, _ = env.reset()                       # a second episode starts from a new scenario
    assert list(obs2.keys()) == list(space.keys())
    env.close()


def test_sb3_adapter_contract(cuda):
    """terminal_observation / TimeLimit.truncated / per-env info dicts (bluesky_gym/utils/logger.py:18-33)."""
    from bluesky_gym_sasha_b200.sb3_vec_env import BlueSkySB3VecEnv
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    E = 6
    v = BlueSkySB3VecEnv(BlueSkyVectorEnv("DescentEnv-v0", E, seed=1, autoreset_mode="same_step", max_episode_steps=5))
    obs = v.reset()
    assert obs["altitude"].shape == (E, 1)
    for k in range(5):
        v.step_async(np.full((E, 1), -0.1))
        obs, rew, dones, infos = v.step_wait()
    assert rew.dtype == np.float32 and dones.all() and len(infos) == E
    assert all(i["TimeLimit.truncated"] and "terminal_observation" in i and "total_reward" in i for i in infos)
    assert not np.allclose(infos[0]["terminal_observation"]["altitude"], obs["altitude"][0])
    v.close()


def test_checkpoint_resume_is_bit_exact(cuda):
    """state_dict() / load_state_dict(): resuming replays exactly the same trajectory (autoreset draws included)."""
    import torch
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    E = 64
    v = BlueSkyVectorEnv("HorizontalCREnv-v0", E, seed=21, n_intruders=20, cd_enabled=True, autoreset_mode="same_step",
                         max_episode_steps=7)
    v.reset_torch()
    g = torch.Generator(device="cpu").manual_seed(1)
    acts = (torch.rand((20, E, 1), generator=g) * 2 - 1).cuda()
    for i in range(5):
        v.step_torch(acts[i])
    sd = v.state_dict()
    ref = []
    for i in range(5, 20):
        o, r, te, tr = v.step_torch(acts[i])
        ref.append((v.t["obs"].clone(), r.clone(), te.clone(), tr.clone()))
    v.load_state_dict(sd)
    for i in range(5, 20):
        o, r, te, tr = v.step_torch(acts[i])
        assert torch.equal(v.t["obs"], ref[i - 5][0]) and torch.equal(r, ref[i - 5][1])
        assert torch.equal(te, ref[i - 5][2]) and torch.equal(tr, ref[i - 5][3])
    assert any(bool(x[3].any()) for x in ref)            # the window crossed TimeLimit truncations + autoresets
    v.close()


def test_checkpoint_resumes_in_a_fresh_env_with_noise_and_wind(cuda):
    """state_dict() carries what the streams are keyed by: seed, the noise call index, the wind tables and the wind
    ground-speed state.  Loaded into a FRESHLY BUILT env (another seed, no noise, no wind yet) the rollout continues
    bit for bit; a checkpoint from another configuration is refused."""
    import torch
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    E = 32
    wind = dict(lat=np.array([51.9, 52.1]), lon=np.array([3.9, 4.1]), vnorth=np.array([[12.0, -6.0]]), veast=np.array([[4.0, 9.0]]))
    kw = dict(n_intruders=12, cd_enabled=True, autoreset_mode="same_step", max_episode_steps=6, init_alt=3000.0)
    v = BlueSkyVectorEnv("HorizontalCREnv-v0", E, seed=21, obs_noise=0.05, wind=wind, **kw)
    v.reset_torch()
    g = torch.Generator(device="cpu").manual_seed(1)
    acts = (torch.rand((20, E, 1), generator=g) * 2 - 1).cuda()
    for i in range(5):
        v.step_torch(acts[i])
    sd = v.state_dict()
    assert sd["obs_noise"] == dict(sigma=pytest.approx(0.05), calls=6) and sd["config"]["seed"] == 21
    ref = []
    for i in range(5, 20):
        o, r, te, tr = v.step_torch(acts[i])
        ref.append((v.t["obs"].clone(), r.clone(), te.clone(), tr.clone()))
    w = BlueSkyVectorEnv("HorizontalCREnv-v0", E, seed=99, **kw)          # fresh handle: other seed, no noise, no wind
    w.reset_torch()
    w.load_state_dict(sd)
    for i in range(5, 20):
        o, r, te, tr = w.step_torch(acts[i])
        assert torch.equal(w.t["obs"], ref[i - 5][0]) and torch.equal(r, ref[i - 5][1]), i
        assert torch.equal(te, ref[i - 5][2]) and torch.equal(tr, ref[i - 5][3])
    assert any(bool(x[3].any()) for x in ref)
    other = BlueSkyVectorEnv("HorizontalCREnv-v0", E, seed=21, n_intruders=5)
    with pytest.raises(ValueError, match="different configuration"):
        other.load_state_dict(sd)
    for x in (v, w, other):
        x.close()


def test_static_obstacle_scalar_env_reset_flags(cuda):
    """reset_flags() is surfaced (0 for a normal scenario); the scalar env turns flag 4 into the reference's Exception."""
    import bluesky_gym
    bluesky_gym.register_envs()
    env = bluesky_gym.make("StaticObstacleEnv-v0")
    obs, info = env.reset()
    assert int(env.unwrapped.vec.reset_flags()[0]) & 4 == 0
    env.unwrapped.vec.t["env_i32"][0, _lib.I32_RESET_FLAGS] = 4
    with pytest.raises(Exception, match="No waypoints can be generated"):
        env.unwrapped._check_reset_flags()
    env.close()


def test_reset_seed_rekeys_streams(cuda):
    """gymnasium seeding: reset(seed=s) reproduces the scenario of a fresh env built with seed=s."""
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    a = BlueSkyVectorEnv("SectorCREnv-v0", 8, seed=1)
    b = BlueSkyVectorEnv("SectorCREnv-v0", 8, seed=77)
    oa, _ = a.reset(seed=77)
    ob, _ = b.reset()
    for k in oa:
        assert np.array_equal(oa[k], ob[k]), k
    o2, _ = a.reset()                                        # next episode of the same stream differs
    assert not np.array_equal(o2["x_r"], oa["x_r"])
    # the contract holds on a used env too: after several episodes, and twice in a row (the episode counter and the
    # noise call index are part of the stream key and restart with the seed)
    for _ in range(3):
        a.reset()
    for _ in range(2):
        o3, _ = a.reset(seed=77)
        for k in oa:
            assert np.array_equal(o3[k], ob[k]), k
    a.close()
    b.close()
    n1 = BlueSkyVectorEnv("DescentEnv-v0", 8, seed=1, obs_noise=0.1)
    n1.reset()
    n1.step(np.zeros((8, 1)))
    first, _ = n1.reset(seed=5)
    n1.step(np.zeros((8, 1)))
    again, _ = n1.reset(seed=5)
    for k in first:
        assert np.array_equal(first[k], again[k]), k          # same noise draws as well
    n1.step_async(np.zeros((8, 1)))
    with pytest.raises(_lib.BsgError):
        n1.reset()                                            # a step is in flight
    n1.step_wait()
    n1.close()


@pytest.mark.parametrize("env_id,kw", [("DescentEnv-v0", {}), ("PlanWaypointEnv-v0", {}), ("HorizontalCREnv-v0", dict(n_intruders=20, cd_enabled=True)),
                                       ("VerticalCREnv-v0", dict(cd_enabled=True)), ("SectorCREnv-v0", dict(cd_enabled=True)),
                                       ("StaticObstacleEnv-v0", {}), ("MergeEnv-v0", dict(cd_enabled=True))])
def test_soak_many_episodes_stay_finite(cuda, env_id, kw):
    """Several hundred steps of random actions with same-step autoreset: every output stays finite, every env keeps
    finishing episodes within the registered cap, and no scenario generator reports a failure."""
    import torch
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    E, steps = 512, 450
    v = BlueSkyVectorEnv(env_id, E, seed=5, autoreset_mode="same_step", **kw)
    cap = v.cfg.max_episode_steps
    v.reset_torch()
    g = torch.Generator(device="cuda").manual_seed(3)
    since = torch.zeros(E, dtype=torch.int32, device="cuda")
    n_done = 0
    for i in range(steps):
        a = torch.rand((E, v.layout.act_dim), device="cuda", generator=g) * 2 - 1
        obs, rew, term, trunc = v.step_torch(a)
        since += 1
        done = (term != 0) | (trunc != 0)
        assert int(since.max()) <= cap, (env_id, i, "an env ran past its TimeLimit")
        since = torch.where(done, torch.zeros_like(since), since)
        n_done += int(done.sum())
        if i % 50 == 49 or i == steps - 1:
            assert bool(torch.isfinite(v.t["obs"]).all()) and bool(torch.isfinite(rew).all()), (env_id, i)
            assert bool(torch.isfinite(v.t["pos"]).all()) and bool(torch.isfinite(v.t["kin"]).all()), (env_id, i)
            info = v.t["info"][:3]
            assert bool(torch.isfinite(info[~torch.isnan(info)]).all())
    assert n_done >= E * (steps // cap)                                   # at least the TimeLimit-driven episodes
    assert int((v.t["env_i32"][:, _lib.I32_RESET_FLAGS] & 4).sum()) == 0        # no generator gave up
    assert int(v.t["env_i32"][:, _lib.I32_EPISODE].min()) >= 1 + steps // cap
    v.close()


@pytest.mark.parametrize("env_id,kw,nsub", [("HorizontalCREnv-v0", dict(n_intruders=20), 10), ("HorizontalCREnv-v0", dict(n_intruders=12), 10),
                                            ("SectorCREnv-v0", {}, 5), ("MergeEnv-v0", {}, 10)])
def test_in_group_cd_kept_candidates_are_a_superset(cuda, env_id, kw, nsub):
    """K3 keeps the candidate list of the pairs among the un-steered aircraft across the substeps of an env step while
    they hold their velocity (env_kernels.cuh, group_cd).  cd_enabled=2 redoes the filter in every substep with no
    allowance; both must give bit-identical results -- after every substep count (bsg_traf_update with n = 1 .. n_sub
    from saved states, so a list kept for 1 .. n_sub - 1 substeps is compared), and along whole rollouts."""
    import torch
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    E = 512
    va = BlueSkyVectorEnv(env_id, E, seed=11, cd_enabled=True, autoreset_mode="same_step", **kw)
    vb = BlueSkyVectorEnv(env_id, E, seed=11, cd_enabled=2, autoreset_mode="same_step", **kw)
    va.reset_torch()
    vb.reset_torch()
    g = torch.Generator(device="cuda").manual_seed(5)
    keys = ("tcpamax", "inconf", "env_i32", "pos", "kin")
    n_conf = 0
    for step in range(60):
        if step % 4 == 0:
            sa, sb = va.state_dict(), vb.state_dict()
            for n in range(1, nsub + 1):
                va.load_state_dict(sa)
                vb.load_state_dict(sb)
                va.traf_update(n)
                vb.traf_update(n)
                for k in keys:
                    assert torch.equal(va.t[k], vb.t[k]), (env_id, step, n, k)
                n_conf += int(va.t["env_i32"][:, _lib.I32_NCONF].sum())
            va.load_state_dict(sa)
            vb.load_state_dict(sb)
        a = torch.rand((E, va.layout.act_dim), device="cuda", generator=g) * 2 - 1
        va.step_torch(a)
        vb.step_torch(a)
        for k in keys + ("obs", "reward", "terminated", "truncated"):
            assert torch.equal(va.t[k], vb.t[k]), (env_id, step, k)
        assert torch.equal(torch.nan_to_num(va.t["info"]), torch.nan_to_num(vb.t["info"])), (env_id, step)
    assert n_conf > 0                                  # the comparison saw conflicts
    va.close()
    vb.close()


def test_horizontal_airborne_variant_matches_oracle(cuda):
    """SURVEY 8d's second C2 input: every aircraft created at 3000 m instead of the reference's 0 (no ground-phase CAS
    cap, aircraft keep 150 m/s CAS).  Device reset against the Philox-driven oracle, then 12 steps with CD on."""
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    E, seed, n_int = 8, 31, 20
    venv = BlueSkyVectorEnv("HorizontalCREnv-v0", E, seed=seed, autoreset_mode="disabled", n_intruders=n_int,
                            cd_enabled=True, init_alt=3000.0)
    gobs, _ = venv.reset()
    d = device_traffic(venv)
    orc = []
    for e in range(E):
        o = _make_oracle("HorizontalCREnv-v0", draws=PhiloxDraws(seed, e, 0), n_int=n_int, cd=True, init_alt=3000.0)
        oobs, _ = o.reset()
        assert np.max(np.abs(d["alt"][e, :n_int + 1] - 3000.0)) < 1e-3 and np.max(np.abs(d["tas"][e, :n_int + 1] - o.traf.tas)) < 1e-3
        assert np.max(np.abs(d["lat"][e, :n_int + 1] - o.traf.lat)) < 1e-9
        _compare_obs(gobs, oobs, e, -1)
        orc.append(o)
    rng = np.random.default_rng(2)
    for step in range(12):
        a = rng.uniform(-1, 1, (E, 1))
        gobs, grew, gterm, gtrunc, ginfo = venv.step(a)
        d = device_traffic(venv)
        for e, o in enumerate(orc):
            oobs, orew, oterm, _, _ = o.step(a[e])
            assert np.max(np.abs(d["tas"][e, :n_int + 1] - o.traf.tas)) < TOL["tas"]          # ~172 m/s: not capped at 88
            assert np.max(np.abs(d["lat"][e, :n_int + 1] - o.traf.lat)) < TOL["pos"]
            _compare_obs(gobs, oobs, e, step)
            assert abs(grew[e] - orew) < 1e-3 and bool(gterm[e]) == bool(oterm)
            assert ginfo["asas_nconf"][e] == len(o.traf.confpairs), (step, e)
    assert float(d["tas"][0, 0]) > 160.0
    venv.close()


@pytest.mark.parametrize("env_id,kw", [("HorizontalCREnv-v0", dict(n_intruders=20, cd_enabled=True)), ("MergeEnv-v0", dict(cd_enabled=True)),
                                       ("SectorCREnv-v0", dict(cd_enabled=True)), ("VerticalCREnv-v0", dict(cd_enabled=True)),
                                       ("DescentEnv-v0", {})])
def test_substeps_split_over_launches_are_bit_identical(cuda, env_id, kw):
    """bsg_traf_update(n) == bsg_traf_update(k) followed by bsg_traf_update(n - k), bit for bit: everything a launch
    caches in registers (ground-speed components, cos(lat), ISA / CAS targets, the kept CD candidate list) is rebuilt
    from the stored state exactly as the substep loop would have carried it."""
    import torch
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    E = 256
    v = BlueSkyVectorEnv(env_id, E, seed=17, autoreset_mode="same_step", **kw)
    v.reset_torch()
    g = torch.Generator(device="cuda").manual_seed(9)
    keys = ("pos", "kin", "cmd", "aux", "flags", "env_i32") + (("tcpamax", "inconf") if kw.get("cd_enabled") else ())
    for step in range(12):
        v.step_torch(torch.rand((E, v.layout.act_dim), device="cuda", generator=g) * 2 - 1)
        if step % 3 == 2:
            sd = v.state_dict()
            v.traf_update(7)
            one = {k: v.t[k].clone() for k in keys}
            for k in (1, 3, 6):
                v.load_state_dict(sd)
                v.traf_update(k)
                v.traf_update(7 - k)
                for name in keys:
                    assert torch.equal(v.t[name], one[name]), (env_id, step, k, name)
            v.load_state_dict(sd)
    v.close()


def test_step_async_wait_equals_step(cuda):
    """step_async() + step_wait() (bsg_step_host_begin / bsg_step_host_wait) return what step() returns, for fresh and
    for mirrored (copy=False) observation arrays, across same-step autoresets; a second step_async before step_wait and
    a step_wait without step_async are errors."""
    from bluesky_gym_sasha_b200 import _lib as L
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    E = 64
    for copy in (True, False):
        kw = dict(seed=13, n_intruders=20, cd_enabled=True, autoreset_mode="same_step", max_episode_steps=5, copy=copy)
        a, b = BlueSkyVectorEnv("HorizontalCREnv-v0", E, **kw), BlueSkyVectorEnv("HorizontalCREnv-v0", E, **kw)
        a.reset()
        b.reset()
        rng = np.random.default_rng(4)
        saw_final = False
        for step in range(12):
            act = rng.uniform(-1, 1, (E, 1))
            ra = a.step(act)
            b.step_async(act)
            if step == 3:
                with pytest.raises(L.BsgError):
                    b.step_async(act)                      # one step in flight per handle
            rb = b.step_wait()
            for k in ra[0]:
                assert np.array_equal(ra[0][k], rb[0][k]), (copy, step, k)
            for x, y in zip(ra[1:4], rb[1:4]):
                assert np.array_equal(x, y)
            assert set(ra[4]) == set(rb[4])
            if "final_obs" in ra[4]:
                saw_final = True
                for k in ra[4]["final_obs"]:
                    m = ra[4]["_final_obs"]
                    assert np.array_equal(ra[4]["final_obs"][k][m], rb[4]["final_obs"][k][m])
        assert saw_final
        with pytest.raises(RuntimeError):
            b.step_wait()
        a.close()
        b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("obs_dtype", [np.float32, np.float64])
def test_step_results_belong_to_the_caller_while_held(cuda, obs_dtype):
    """copy=True (default): the arrays of a step are views of a host block that no later step touches while the caller
    holds any of them (vector_env._HostBlock) -- results kept over many steps equal the copies taken at once, for float32
    and float64 observations, through same-step autoresets (dense terminal observations: zero rows for the envs that did not
    finish), and past the block pool's capacity (then ordinary copies are handed out)."""
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    E = 48
    kw = dict(seed=5, n_intruders=20, cd_enabled=True, autoreset_mode="same_step", max_episode_steps=4, obs_dtype=obs_dtype)
    v, w = BlueSkyVectorEnv("HorizontalCREnv-v0", E, **kw), BlueSkyVectorEnv("HorizontalCREnv-v0", E, copy=False, **kw)
    v._BLOCKS_MAX = 5
    v.reset()
    w.reset()
    rng = np.random.default_rng(2)
    held, snap = [], []

    def deep(r):
        obs, rew, term, trunc, info = r
        fo = {k: x.copy() for k, x in info["final_obs"].items()} if "final_obs" in info else None
        return ({k: x.copy() for k, x in obs.items()}, rew.copy(), term.copy(), trunc.copy(),
                {k: np.array(x, copy=True) for k, x in info.items() if k != "final_obs"}, fo)

    n_final = 0
    for step in range(14):
        act = rng.uniform(-1, 1, (E, 1))
        r = v.step(act)
        rw = deep(w.step(act))                                # the rotating-mirror mode is the independent witness
        held.append(r)
        snap.append(rw)
        assert r[0]["intruder_distance"].dtype == obs_dtype
        if step >= 9:
            held[step - 9] = None                             # blocks come back into circulation when their results are dropped
    assert len(v._blocks) <= 5
    for r, s in zip(held, snap):
        if r is None:
            continue
        obs, rew, term, trunc, info = r
        for k in obs:
            assert np.array_equal(obs[k], s[0][k]), k
        assert np.array_equal(rew, s[1]) and np.array_equal(term, s[2]) and np.array_equal(trunc, s[3])
        for k in s[4]:
            assert np.array_equal(info[k], s[4][k]), k
        assert ("final_obs" in info) == (s[5] is not None)
        if s[5] is not None:
            m = info["_final_obs"]
            n_final += int(m.sum())
            for k in s[5]:
                assert info["final_obs"][k].dtype == obs_dtype
                assert np.array_equal(info["final_obs"][k][m], s[5][k][m])
                assert not np.any(info["final_obs"][k][~m]) and not np.any(s[5][k][~m])
    assert n_final >= E
    v.close()
    w.close()
