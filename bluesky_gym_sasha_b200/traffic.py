"""AirspaceTraffic -- one airspace of N aircraft with routes, VNAV and ASAS conflict resolution on the GPU (SURVEY 8f-4).

Interface mirrored: the handful of ``bs.traf`` / ``bs.stack`` calls a BlueSky scenario with routes and resolution uses --
``cre`` (many at once), ``ADDWPT acid lat lon alt spd`` x n + ``LNAV / VNAV ON`` (``set_routes``), ``HDG / SPD / ALT``
select commands, ``RESO MVP`` / ``RESO OFF`` (``reso=``; the reference's own line is ``reso off``, merge_env.py:157),
``RESOOFF acid``, ``bs.sim.step()`` (``step``) -- with the state arrays ``lat, lon, alt, tas, hdg, vs, ...`` as properties.
Per substep: ``bsg_traf_pack`` -> ``bsg_cd_detect[_culled]`` with pair lists (K2) -> ``bsg_traf_substep`` (include/bsg.h).  Restated for checking in oracle/traffic_ext.py.  No CPU fallback.
With ``events=True`` each detection also feeds ``bsg_traf_events_update``: the conflict / LoS event counts and logs of
upstream's ConflictDetection.update (``conflict_counts``, ``conflict_log``; restated in oracle/conflict_log.py).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .cd import StateBasedCD, _ptr

NM, FT, FPM, KTS = 1852.0, 0.3048, 0.3048 / 60.0, 0.514444


# ---- bluesky.tools.aero / geo on the host, float64 (creation-time conversions and Route.calcfp only) ---------------------
def _vatmos(h):
    T = np.maximum(288.15 - 0.0065 * h, 216.65)
    rho = 1.225 * np.power(T / 288.15, 4.256848030018761) * np.exp(-np.maximum(0.0, h - 11000.0) / 6341.552161)
    return rho * 287.05287 * T, rho, T


def vcas2tas(cas, h):
    p, rho, _ = _vatmos(h)
    q = 101325.0 * (np.power(1.0 + 1.225 * cas * cas / (7.0 * 101325.0), 3.5) - 1.0)
    tas = np.sqrt(7.0 * p / rho * (np.power(q / p + 1.0, 2.0 / 7.0) - 1.0))
    return np.where(cas < 0, -tas, tas)


def vcasormach2tas(spd, h):
    """bluesky.tools.aero.vcasormach2tas: 0.1 < spd < 1 is a Mach number, anything else a CAS [m/s]."""
    spd, h = np.asarray(spd, dtype=np.float64), np.asarray(h, dtype=np.float64)
    _, _, T = _vatmos(h)
    ismach = (spd > 0.1) & (spd < 1.0)
    return np.where(ismach, spd * np.sqrt(1.4 * 287.05287 * T), vcas2tas(spd, h))


def _rwgs84(latd):
    lat = np.radians(latd)
    a, b = 6378137.0, 6356752.314245
    an, bn, ad, bd = a * a * np.cos(lat), b * b * np.sin(lat), a * np.cos(lat), b * np.sin(lat)
    return np.sqrt((an * an + bn * bn) / (ad * ad + bd * bd))


def qdrdist(latd1, lond1, latd2, lond2):
    """bluesky.tools.geo.qdrdist: bearing [deg, -180..180] and distance [m] (WGS-84 radius haversine)."""
    latd1, latd2 = np.asarray(latd1, dtype=np.float64), np.asarray(latd2, dtype=np.float64)
    a = 6378137.0
    res2 = 0.5 * (np.abs(latd1) * (_rwgs84(latd1) + a) + np.abs(latd2) * (_rwgs84(latd2) + a)) / \
        np.maximum(0.000001, np.abs(latd1) + np.abs(latd2))
    r = np.where(latd1 * latd2 >= 0.0, _rwgs84(0.5 * (latd1 + latd2)), res2)
    lat1, lon1, lat2, lon2 = np.radians(latd1), np.radians(lond1), np.radians(latd2), np.radians(lond2)
    s1, s2 = np.sin(0.5 * (lat2 - lat1)), np.sin(0.5 * (lon2 - lon1))
    root = s1 * s1 + np.cos(lat1) * np.cos(lat2) * s2 * s2
    d = 2.0 * r * np.arctan2(np.sqrt(root), np.sqrt(1.0 - root))
    q = np.degrees(np.arctan2(np.sin(lon2 - lon1) * np.cos(lat2),
                              np.cos(lat1) * np.sin(lat2) - np.sin(lat1) * np.cos(lat2) * np.cos(lon2 - lon1)))
    return q, d


def route_tables(lat, lon, alt, spd, nwp, W):
    """Route.calcfp for a batch of routes: ``lat, lon, alt, spd`` are [k, W] (alt / spd < 0 = no constraint), ``nwp`` [k].
    Returns rt_pos [k, W, 2] f64, rt_con [k, W, 4] f32 (wpalt, wpspd, wptoalt, wpxtoalt), rt_dir [k, W] f32 (direction of
    the leg leaving each waypoint, -999 after the last)."""
    lat, lon = np.asarray(lat, dtype=np.float64), np.asarray(lon, dtype=np.float64)
    k = lat.shape[0]
    alt = np.full((k, W), -999.0) if alt is None else np.asarray(alt, dtype=np.float64)
    spd = np.full((k, W), -999.0) if spd is None else np.asarray(spd, dtype=np.float64)
    nwp = np.asarray(nwp, dtype=np.int64)
    q, d = qdrdist(lat[:, :-1], lon[:, :-1], lat[:, 1:], lon[:, 1:]) if W > 1 else (np.zeros((k, 0)), np.zeros((k, 0)))
    col = np.arange(W).reshape(1, W)
    rt_dir = np.full((k, W), -999.0)
    rt_dir[:, :W - 1] = np.where(col[:, :W - 1] < (nwp.reshape(-1, 1) - 1), q, -999.0)
    toalt, xtoalt = np.full((k, W), -999.0), np.zeros((k, W))
    t, x = np.full(k, -999.0), np.zeros(k)
    for c in range(W - 1, -1, -1):                      # backwards: next altitude constraint at or after waypoint c
        live = c < nwp
        has = live & (alt[:, c] >= 0.0)
        last = c == nwp - 1
        leg = d[:, c] if c < W - 1 else np.zeros(k)     # length of the leg from c to c + 1
        x = np.where(has, 0.0, np.where(last | ~live, 0.0, x + leg))
        t = np.where(has, alt[:, c], np.where(live, t, -999.0))
        toalt[:, c], xtoalt[:, c] = t, x
    rt_pos = np.stack([lat, lon], axis=-1)
    rt_con = np.stack([alt, spd, toalt, xtoalt], axis=-1).astype(np.float32)
    return rt_pos, rt_con, rt_dir.astype(np.float32)


class AirspaceTraffic:
    COUNTERS = ("resopair_overflow", "wp_switches", "asas_active")

    def __init__(self, n_max, device=0, simdt=1.0, rpz=5.0 * NM, hpz=1000.0 * FT, dtlookahead=300.0, reso=None, reso_mode=0,
                 resofach=1.01, resofacv=1.01, perf=None, max_wpts=8, lat0=52.0, lon0=4.0, cull=True, symmetric=True,
                 pair_capacity=None, fms_dt=10.5, group=None, events=False, event_capacity=None):
        """``group``: a ``torch.distributed`` process group (``True`` = the default group) over which ONE airspace is sharded,
        one rank per GPU (SURVEY 8e): every rank owns the kinematics of up to ``n_max`` aircraft (its block); per substep the
        ranks all-gather their CD records (32 B per aircraft over NVLink), each detects the conflicts of its own rows against
        the whole airspace and advances its own aircraft.  Results equal the unsharded airspace's.

        ``events=True``: every detection also updates the conflict and LoS event record of upstream's
        ConflictDetection.update (confpairs_all / lospairs_all) on the device (bsg_traf_events_update), read with
        ``conflict_counts()`` and ``conflict_log()``.  ``event_capacity``: rows of each event log (default 8 x n_max); the
        totals stay exact when a log is full.  Not with ``group``: on a row-sharded rank the two orders of a pair sit on
        different GPUs, so counting unordered pairs would need an exchange of the pair lists."""
        if events and group is not None and group is not False:
            raise ValueError("events=True is not available for an airspace sharded over a process group")
        if not torch.cuda.is_available():
            raise _lib.BsgError("AirspaceTraffic needs a CUDA device: there is no CPU fallback")
        if reso not in (None, "OFF", "MVP"):
            raise ValueError("reso must be None / 'OFF' or 'MVP'")
        if not 1 <= max_wpts <= 127:
            raise ValueError("max_wpts must be in [1, 127]")
        self.lib = _lib.load()
        self.device = torch.device("cuda", device)
        self.n_max, self.n, self.W = int(n_max), 0, int(max_wpts)
        self.simdt = float(simdt)
        self.reso = 1 if reso == "MVP" else 0
        self.cull, self.symmetric = bool(cull), bool(symmetric)
        self.fms_rel_freq = max(1, int(fms_dt // self.simdt))
        self.nstep = 0
        cap = int(pair_capacity) if pair_capacity else max(4096, 8 * self.n_max)
        self.cd = StateBasedCD(device=device, rpz=rpz, hpz=hpz, dtlookahead=dtlookahead, pair_capacity=cap, los_capacity=cap)
        from .spec import A320_PERF
        self.perf = dict(A320_PERF, **(perf or {}))
        self.cfg = _lib.TrafConfig(n=0, max_wpts=self.W, reso=self.reso, reso_mode=int(reso_mode), simdt=self.simdt,
                                   rpz=float(rpz), hpz=float(hpz), dtlookahead=float(dtlookahead), resofach=float(resofach),
                                   resofacv=float(resofacv), perf=_lib.Perf(**self.perf), lat0=float(lat0), lon0=float(lon0))
        n, W, dev = self.n_max, self.W, self.device
        z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device=dev)
        self.t = dict(pos=z(n, 2, dt=torch.float64), kin=z(n, 4), cmd=z(n, 4), aux=z(n, 4), actwp=z(n, 2, dt=torch.float64),
                      vnav1=z(n, 4), vnav2=z(n, 4), asas=z(n, 4), flags=z(n, dt=torch.int32),
                      partners=torch.full((n, _lib.TRAF_PARTNERS), -1, dtype=torch.int32, device=dev),
                      rt_pos=z(n, W, 2, dt=torch.float64), rt_con=z(n, W, 4), rt_dir=z(n, W),
                      counters=z(_lib.TRAF_CTR_COUNT, dt=torch.int32))
        self.tt = _lib.TrafTensors(**{k: _ptr(v) for k, v in self.t.items()})
        n_pad = int(self.lib.bsg_cd_padded(n))
        self.rec = torch.empty((max(n_pad // 256, 1), 8, 256), dtype=torch.float32, device=dev)
        self.work = torch.zeros(int(self.lib.bsg_traf_workspace(n, cap)), dtype=torch.uint8, device=dev)      # (zeroed once)
        self.last = None                    # device outputs of the last substep's detection
        self.gpu_launches = 0
        self.events = bool(events)
        if self.events:
            ecap = int(event_capacity) if event_capacity is not None else 8 * self.n_max
            if ecap < 0:
                raise ValueError("event_capacity must be >= 0")
            nb = int(self.lib.bsg_traf_events_workspace(cap, cap))
            self.ev_sets = [torch.zeros(nb, dtype=torch.uint8, device=dev) for _ in range(2)]    # (zeroed once)
            rows = max(ecap, 1)
            self.ev = dict(conf_log=z(rows, 4, dt=torch.int32), los_log=z(rows, 4, dt=torch.int32), los_sev=z(rows, 2),
                           counters=z(_lib.EV_CTR_COUNT, dt=torch.int64))
            self.ev_struct = _lib.TrafEvents(set_bytes=nb, d_conf_log=_ptr(self.ev["conf_log"]), d_los_log=_ptr(self.ev["los_log"]),
                                             d_los_sev=_ptr(self.ev["los_sev"]), conf_log_cap=ecap, los_log_cap=ecap,
                                             d_counters=_ptr(self.ev["counters"]))
            self.event_capacity = ecap
        # one airspace over several GPUs: block k of the records belongs to rank k, `per` records each (whole tiles)
        self.group, self.world, self.rank, self.row0 = None, 1, 0, 0
        if group is not None and group is not False:
            import torch.distributed as dist
            self.group = None if group is True else group
            self.world, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
            self.per = max(n_pad, 256)
            self.row0 = self.rank * self.per
            self.cfg.row0 = self.row0
            self.rec.zero_()                # records this rank never packs (beyond its aircraft count) stay inert
            self.rec[:, 2, :] = 1.0
            self.rec[:, 6, :] = 3.0e9
            self.allrec = torch.empty((self.per // 256 * self.world, 8, 256), dtype=torch.float32, device=dev)
            self.nconf_all = torch.zeros(2, dtype=torch.int64, device=dev)

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _dev(self, x, dtype):
        return torch.as_tensor(np.ascontiguousarray(x), device=self.device).to(dtype)

    # ------------------------------------------------------------------ bs.traf.cre (SI arguments), many at once
    def create(self, lat, lon, hdg, alt, spd, resooff=None):
        """Appends aircraft: ``spd`` is a CAS [m/s] (or a Mach number when 0.1 < spd < 1), as in Traffic.cre.
        Returns the index range of the new aircraft."""
        lat, lon, hdg, alt, spd = (np.atleast_1d(np.asarray(v, dtype=np.float64)) for v in (lat, lon, hdg, alt, spd))
        k = lat.shape[0]
        if self.n + k > self.n_max:
            raise ValueError("AirspaceTraffic: more aircraft than n_max")
        lon = np.where(lon > 180.0, lon - 360.0, np.where(lon < -180.0, lon + 360.0, lon))
        tas = vcasormach2tas(spd, alt)
        s = slice(self.n, self.n + k)
        t = self.t
        t["pos"][s] = self._dev(np.stack([lat, lon], axis=1), torch.float64)
        t["kin"][s] = self._dev(np.stack([alt, tas, hdg, np.zeros(k)], axis=1), torch.float32)
        t["cmd"][s] = self._dev(np.stack([spd, alt, np.zeros(k), hdg], axis=1), torch.float32)
        t["aux"][s] = self._dev(np.stack([np.zeros(k), np.full(k, -999.0), np.full(k, -999.0), np.zeros(k)], axis=1), torch.float32)
        t["actwp"][s] = self._dev(np.stack([np.full(k, 89.99), np.zeros(k)], axis=1), torch.float64)      # ActiveWaypoint.create
        t["vnav1"][s] = self._dev(np.stack([np.full(k, -999.0), np.zeros(k), np.zeros(k), np.full(k, -999.0)], axis=1), torch.float32)
        t["vnav2"][s] = self._dev(np.stack([np.full(k, -999.0), np.full(k, -999.0), np.full(k, -999.0), np.zeros(k)], axis=1), torch.float32)
        t["asas"][s] = self._dev(np.stack([hdg, tas, np.zeros(k), alt], axis=1), torch.float32)
        # perf.create: phase of the initial state (vs = 0)
        alt_ft = alt / FT
        fl = np.full(k, _lib.TF_ALIVE, dtype=np.int64) | np.where(alt_ft <= 75.0, _lib.TF_PH_GD, 0)
        if resooff is not None:
            fl |= np.where(np.asarray(resooff, dtype=bool), _lib.TF_RESOOFF, 0)
        t["flags"][s] = self._dev(fl, torch.int32)
        t["partners"][s] = -1
        self.n += k
        self.cfg.n = self.n
        return range(s.start, s.stop)

    # ------------------------------------------------------------------ ADDWPT x n + LNAV / VNAV ON
    def set_routes(self, idx, lat, lon, alt=None, spd=None, nwp=None, vnav=True):
        """Routes for the aircraft ``idx`` [k]: ``lat, lon`` [k, <= W] waypoints, optional altitude [m] / CAS [m/s]
        constraints (< 0: none), ``nwp`` [k] waypoints actually used (default: all columns).  The first waypoint becomes
        the active one (Route.direct), LNAV on, VNAV (+ VNAV speed) as requested."""
        idx = np.atleast_1d(np.asarray(idx, dtype=np.int64))
        lat, lon = np.atleast_2d(np.asarray(lat, dtype=np.float64)), np.atleast_2d(np.asarray(lon, dtype=np.float64))
        k, w = lat.shape
        if w > self.W:
            raise ValueError("route longer than max_wpts")
        pad = lambda a, fill: np.concatenate([np.asarray(a, dtype=np.float64).reshape(k, w), np.full((k, self.W - w), fill)], axis=1)
        nwp = np.full(k, w, dtype=np.int64) if nwp is None else np.asarray(nwp, dtype=np.int64)
        if (nwp < 1).any() or (nwp > w).any():
            raise ValueError("nwp must be in [1, number of waypoint columns]")
        rt_pos, rt_con, rt_dir = route_tables(pad(lat, 0.0), pad(lon, 0.0), None if alt is None else pad(alt, -999.0),
                                              None if spd is None else pad(spd, -999.0), nwp, self.W)
        di = torch.as_tensor(idx, device=self.device)
        self.t["rt_pos"][di] = self._dev(rt_pos, torch.float64)
        self.t["rt_con"][di] = self._dev(rt_con, torch.float32)
        self.t["rt_dir"][di] = self._dev(rt_dir, torch.float32)
        vn = np.broadcast_to(np.asarray(vnav, dtype=bool), (k,))
        keep = _lib.TF_ALIVE | _lib.TF_RESOOFF | _lib.TF_PH_GD | _lib.TF_PH_AP | _lib.TF_ASAS
        fl = self.t["flags"][di].to(torch.int64) & keep
        add = _lib.TF_ACTIVATE | np.where(vn, _lib.TF_VNAV | _lib.TF_VNAVSPD, 0) | (nwp << _lib.TF_NWP_SHIFT)
        self.t["flags"][di] = (fl | self._dev(add, torch.int64)).to(torch.int32)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.bsg_traf_activate(C.byref(self.cfg), C.byref(self.tt), self._stream()))
        self.gpu_launches += 1

    # ------------------------------------------------------------------ select-mode commands (stack HDG / SPD / ALT)
    def hdg(self, idx, hdg):
        """HDG acid hdg: ap.trk = hdg, LNAV off."""
        di = torch.as_tensor(np.atleast_1d(idx), device=self.device)
        self.t["cmd"][di, 3] = self._dev(np.atleast_1d(hdg), torch.float32)
        self.t["flags"][di] &= ~_lib.TF_LNAV

    def spd(self, idx, cas):
        """SPD acid cas [m/s] (or Mach): selspd, VNAV speed off."""
        di = torch.as_tensor(np.atleast_1d(idx), device=self.device)
        self.t["cmd"][di, 0] = self._dev(np.atleast_1d(cas), torch.float32)
        self.t["flags"][di] &= ~_lib.TF_VNAVSPD

    def alt(self, idx, alt, vs=None):
        """ALT acid alt [m] (, vs [m/s]): selalt (selvs), VNAV off."""
        di = torch.as_tensor(np.atleast_1d(idx), device=self.device)
        self.t["cmd"][di, 1] = self._dev(np.atleast_1d(alt), torch.float32)
        if vs is not None:
            self.t["cmd"][di, 2] = self._dev(np.atleast_1d(vs), torch.float32)
        self.t["flags"][di] &= ~_lib.TF_VNAV

    # ------------------------------------------------------------------ bs.sim.step() x n_sub
    def step(self, n_sub=1, detect=True):
        """``n_sub`` simulator substeps, asynchronous on the current stream.  ``detect=False`` skips ASAS (only without
        resolution)."""
        if not detect and self.reso:
            raise ValueError("resolution needs the detection")
        n = self.n
        if n == 0 and self.world == 1:
            return
        cd = self.cd
        with torch.cuda.device(self.device):
            st = self._stream()
            for _ in range(n_sub):
                self.nstep += 1
                fms_ready = (self.nstep % self.fms_rel_freq) == 0
                pairs = attr = npairs = nall = None
                rec = self.rec
                if detect:
                    _lib.check(self.lib.bsg_traf_pack(C.byref(self.cfg), C.byref(self.tt), _ptr(self.rec), st))
                    if self.world > 1:
                        import torch.distributed as dist
                        dist.all_gather_into_tensor(self.allrec, self.rec[:self.per // 256], group=self.group)
                        rec = self.allrec
                        out = cd.detect_packed(rec, self.per * self.world, row0=self.row0, n_rows=n, want_pairs=True, cull=self.cull)
                        if self.reso:       # upstream resolves whenever ANY conflict exists in the airspace
                            self.nconf_all.copy_(out["npairs"])
                            dist.all_reduce(self.nconf_all, group=self.group)
                            nall = self.nconf_all
                    else:
                        out = cd.detect_packed(rec, n, want_pairs=True, cull=self.cull, symmetric=self.symmetric)
                    self.last = out
                    self.gpu_launches += 1
                    if self.events:
                        self._track_events(out, st)
                    if self.reso:
                        pairs, attr, npairs = out["pairs"], out["attr"], out["npairs"]
                        self.gpu_launches += 3
                _lib.check(self.lib.bsg_traf_substep(C.byref(self.cfg), C.byref(self.tt), _ptr(rec), int(fms_ready),
                                                     _ptr(pairs), _ptr(attr), _ptr(npairs), _ptr(nall),
                                                     cd.pair_capacity if pairs is not None else 0,
                                                     _ptr(self.work), self.work.numel(), st))
                self.gpu_launches += 1

    def _track_events(self, out, st):
        """bsg_traf_events_update on this detection's lists, then the sets swap roles."""
        ev, cd = self.ev_struct, self.cd
        ev.d_cur, ev.d_prev = _ptr(self.ev_sets[0]), _ptr(self.ev_sets[1])
        lists = _lib.CdLists(d_conf_pairs=_ptr(out["pairs"]), d_conf_attr=_ptr(out["attr"]), conf_cap=cd.pair_capacity,
                             d_los_pairs=_ptr(out["lospairs"]), los_cap=cd.los_capacity, d_npairs=_ptr(out["npairs"]))
        _lib.check(self.lib.bsg_traf_events_update(C.byref(ev), _ptr(self.rec), C.byref(lists), self.nstep, st))
        self.ev_sets.reverse()
        self.gpu_launches += 2

    # ------------------------------------------------------------------ state (device tensors, views)
    def _col(self, name, c):
        return self.t[name][:self.n, c]

    lat = property(lambda s: s._col("pos", 0))
    lon = property(lambda s: s._col("pos", 1))
    altitude = property(lambda s: s._col("kin", 0))
    tas = property(lambda s: s._col("kin", 1))
    heading = property(lambda s: s._col("kin", 2))
    vs = property(lambda s: s._col("kin", 3))
    selspd = property(lambda s: s._col("cmd", 0))
    selalt = property(lambda s: s._col("cmd", 1))
    selvs = property(lambda s: s._col("cmd", 2))
    ap_trk = property(lambda s: s._col("cmd", 3))
    flags = property(lambda s: s.t["flags"][:s.n])
    asas_active = property(lambda s: (s.t["flags"][:s.n] & _lib.TF_ASAS) != 0)
    swlnav = property(lambda s: (s.t["flags"][:s.n] & _lib.TF_LNAV) != 0)
    swvnav = property(lambda s: (s.t["flags"][:s.n] & _lib.TF_VNAV) != 0)
    iactwp = property(lambda s: (s.t["flags"][:s.n] >> _lib.TF_IWP_SHIFT) & 0xff)

    def counters(self):
        c = self.t["counters"].cpu().numpy()
        return {k: int(c[i]) for i, k in enumerate(self.COUNTERS)}

    def conflicts(self):
        """Host copy of the last substep's detection: ``confpairs`` [m, 2] (own, intruder) in upstream's row-major order with
        ``qdr, dist, dcpa, tcpa, tinconf`` per conflict, ``lospairs``, ``inconf``, ``tcpamax``."""
        out = self.last
        if out is None:
            raise _lib.BsgError("no detection has run yet")
        torch.cuda.synchronize(self.device)
        n_conf, n_los = (int(v) for v in out["npairs"].cpu())
        k, kl = min(n_conf, self.cd.pair_capacity), min(n_los, self.cd.los_capacity)
        pairs, los, attr = out["pairs"][:k].cpu().numpy(), out["lospairs"][:kl].cpu().numpy(), out["attr"][:k].cpu().numpy()
        o, ol = np.lexsort((pairs[:, 1], pairs[:, 0])), np.lexsort((los[:, 1], los[:, 0]))
        res = dict(confpairs=pairs[o], lospairs=los[ol], inconf=out["inconf"][:self.n].cpu().numpy().astype(bool),
                   tcpamax=out["tcpamax"][:self.n].cpu().numpy().astype(np.float64), n_conf=n_conf, n_los=n_los,
                   truncated=n_conf > self.cd.pair_capacity or n_los > self.cd.los_capacity)
        for c, name in enumerate(_lib.CD_ATTR):
            res[name] = attr[o, c].astype(np.float64)
        return res

    def conflict_counts(self):
        """Event totals since creation (``events=True``): ``nconf_total`` = len(confpairs_all), ``nlos_total`` =
        len(lospairs_all), the events open after the last detection (``nconf_active``, ``nlos_active``), ``log_overflow``
        (events not logged: log full) and ``truncated`` (detections whose pair lists were incomplete, npairs > pair_capacity:
        from the first one on, the events are unreliable).  Copies only the counter array."""
        if not self.events:
            raise _lib.BsgError("AirspaceTraffic was created without events=True")
        c = self.ev["counters"].cpu().numpy()
        keys = ("nconf_total", "nlos_total", "nconf_active", "nlos_active", "log_overflow", "truncated")
        return {k: int(c[i]) for i, k in enumerate(keys)}

    def conflict_log(self):
        """Host copy of the event logs (``events=True``), sorted by (start, a, b): ``confpairs_all`` [m, 2] (a < b),
        ``conf_start``, ``conf_end`` (the ``nstep`` of the first detection with / without the pair; end -1 = still open),
        ``lospairs_all`` [k, 2], ``los_start``, ``los_end``, ``los_dmin`` / ``los_dalt_min`` [m] (least horizontal distance /
        |dalt| over the event's detections), and the counts of ``conflict_counts()``.  The time of step s is (s - 1) * simdt."""
        res = self.conflict_counts()
        mc, ml = min(res["nconf_total"], self.event_capacity), min(res["nlos_total"], self.event_capacity)
        conf, los = self.ev["conf_log"][:mc].cpu().numpy(), self.ev["los_log"][:ml].cpu().numpy()
        sev = self.ev["los_sev"][:ml].cpu().numpy().astype(np.float64)
        o, ol = np.lexsort((conf[:, 1], conf[:, 0], conf[:, 2])), np.lexsort((los[:, 1], los[:, 0], los[:, 2]))
        res.update(confpairs_all=conf[o, :2], conf_start=conf[o, 2], conf_end=conf[o, 3], lospairs_all=los[ol, :2],
                   los_start=los[ol, 2], los_end=los[ol, 3], los_dmin=sev[ol, 0], los_dalt_min=sev[ol, 1])
        return res
