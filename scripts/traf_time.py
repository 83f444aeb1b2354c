"""Device time of the stages of one AirspaceTraffic substep on bench.py's airspace (N = 100k, four-waypoint VNAV routes, MVP;
CUDA events, median of 20), and of the whole substep with conflict-event tracking (events=True) against without, the two
airspaces stepped alternately in one run (20 repetitions each, medians).  Prints the card and its power limit with them."""
import os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes as C
import torch
from bluesky_gym_sasha_b200 import _lib
from bluesky_gym_sasha_b200.cd import _ptr
from tests.test_traffic_events import bench_airspace

REPS = 20
dev = torch.device("cuda", 0)
stages = {}
def timed(name, fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); r = fn(); b.record()
    stages.setdefault(name, []).append((a, b))
    return r
def staged_step(self):
    """AirspaceTraffic.step(1) of an unsharded airspace with detection, each stage between its own events."""
    cd = self.cd
    with torch.cuda.device(self.device):
        st = self._stream()
        self.nstep += 1
        fms_ready = (self.nstep % self.fms_rel_freq) == 0
        timed("pack", lambda: _lib.check(self.lib.bsg_traf_pack(C.byref(self.cfg), C.byref(self.tt), _ptr(self.rec), st)))
        out = timed("detect", lambda: cd.detect_packed(self.rec, self.n, want_pairs=True, cull=self.cull, symmetric=self.symmetric))
        self.last = out
        if self.events:
            timed("events", lambda: self._track_events(out, st))
        timed("substep", lambda: _lib.check(self.lib.bsg_traf_substep(C.byref(self.cfg), C.byref(self.tt), _ptr(self.rec), int(fms_ready),
              _ptr(out["pairs"]), _ptr(out["attr"]), _ptr(out["npairs"]), None, cd.pair_capacity, _ptr(self.work), self.work.numel(), st)))

median = lambda ts: sorted(ts)[len(ts) // 2]
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.TimeoutExpired):
    power = "unknown"
print(f"card {torch.cuda.get_device_name(dev)}, power limit {power}")

tr = bench_airspace(100_000, events=True)
tr.step(20)                                        # warm-up, as bench_traffic
for _ in range(REPS):
    staged_step(tr)
torch.cuda.synchronize()
for k, v in stages.items():
    ts = sorted(a.elapsed_time(b) * 1e3 for a, b in v)
    print(f"{k:12s} median {median(ts):8.1f} us   min {ts[0]:8.1f}")
print(f"after {tr.nstep} substeps: {tr.conflict_counts()}")

on, off = bench_airspace(100_000, events=True), bench_airspace(100_000, events=False)
on.step(20); off.step(20)
ev = {k: [] for k in ("on", "off")}
for _ in range(REPS):
    for k, g in (("on", on), ("off", off)):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); g.step(1); b.record()
        ev[k].append((a, b))
torch.cuda.synchronize()
t = {k: median([a.elapsed_time(b) * 1e3 for a, b in v]) for k, v in ev.items()}
print(f"whole substep, median of {REPS}: events on {t['on']:.1f} us, off {t['off']:.1f} us, "
      f"+{t['on'] - t['off']:.1f} us ({100.0 * (t['on'] / t['off'] - 1.0):+.1f} %)")
