"""Conflict and loss-of-separation events of an airspace: what upstream's ConflictDetection.update keeps besides the
pair lists of the detection.  float64, pure Python.

[UPSTREAM-RECALL] bluesky/traffic/asas/detection.py::ConflictDetection.update (not checked against an install):

    confpairs_unique = {frozenset(pair) for pair in self.confpairs}
    lospairs_unique  = {frozenset(pair) for pair in self.lospairs}
    self.confpairs_all.extend(confpairs_unique - self.confpairs_unique)
    self.lospairs_all.extend(lospairs_unique - self.lospairs_unique)
    self.confpairs_unique, self.lospairs_unique = confpairs_unique, lospairs_unique

so len(confpairs_all) / len(lospairs_all) are the numbers of conflicts / LoS.  On top of that each event here carries the
nstep of the detection it started at and of the first later one without it (-1 while open), and a LoS event the least
horizontal distance and |dalt| over its detections.  Reference for bsg_traf_events_update (AirspaceTraffic(events=True)).
Test infrastructure only (see oracle/__init__.py).
"""
import numpy as np


def _unique(pairs):
    return {(min(int(i), int(j)), max(int(i), int(j))) for i, j in pairs if int(i) != int(j)}


class ConflictLog:
    def __init__(self):
        self.confpairs_unique, self.lospairs_unique = set(), set()
        self.conf, self.los = [], []                # rows [a, b, start, end] / [a, b, start, end, dmin, dalt_min]
        self._open_conf, self._open_los = {}, {}    # open pair -> its row
        self.truncated = 0

    def update(self, confpairs, lospairs, nstep, dist_fn=None, truncated=False):
        """One detection: ``confpairs`` / ``lospairs`` ordered (own, intruder) pairs in any order and orientation, ``nstep``
        its simulator step.  ``dist_fn(a, b)`` (arrays of the LoS pairs of this detection, a < b) -> (horizontal distance,
        |dalt|) arrays, or None to skip the severity.  ``truncated``: the lists were incomplete (counted only)."""
        self.truncated += int(bool(truncated))
        cu, lu = _unique(confpairs), _unique(lospairs)
        for rows, is_open, old, new in ((self.conf, self._open_conf, self.confpairs_unique, cu),
                                        (self.los, self._open_los, self.lospairs_unique, lu)):
            for p in old - new:
                rows[is_open.pop(p)][3] = nstep
            for p in sorted(new - old):
                is_open[p] = len(rows)
                rows.append([p[0], p[1], nstep, -1] + ([np.inf, np.inf] if rows is self.los else []))
        if dist_fn is not None and lu:
            pl = sorted(lu)
            d, dalt = dist_fn(np.array([p[0] for p in pl]), np.array([p[1] for p in pl]))
            for p, dk, ak in zip(pl, np.atleast_1d(d), np.atleast_1d(dalt)):
                r = self.los[self._open_los[p]]
                r[4], r[5] = min(r[4], float(dk)), min(r[5], float(ak))
        self.confpairs_unique, self.lospairs_unique = cu, lu

    def counts(self):
        return dict(nconf_total=len(self.conf), nlos_total=len(self.los), nconf_active=len(self.confpairs_unique),
                    nlos_active=len(self.lospairs_unique), truncated=self.truncated)

    def log(self):
        """The events sorted by (start, a, b), keyed like AirspaceTraffic.conflict_log()."""
        conf = np.array(sorted(self.conf, key=lambda r: (r[2], r[0], r[1])), dtype=np.int64).reshape(-1, 4)
        los = sorted(self.los, key=lambda r: (r[2], r[0], r[1]))
        li = np.array([r[:4] for r in los], dtype=np.int64).reshape(-1, 4)
        lf = np.array([r[4:] for r in los], dtype=np.float64).reshape(-1, 2)
        return dict(confpairs_all=conf[:, :2], conf_start=conf[:, 2], conf_end=conf[:, 3], lospairs_all=li[:, :2],
                    los_start=li[:, 2], los_end=li[:, 3], los_dmin=lf[:, 0], los_dalt_min=lf[:, 1], **self.counts())
