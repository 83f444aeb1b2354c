"""Device time per AirspaceTraffic substep with the spatial order of the CD records on (reorder_dt = 60 s) and off, on
bench.py's airspace (N = 100k, four-waypoint VNAV routes, MVP; CUDA events, medians of REPS substeps, the two airspaces
stepped alternately in one run):
  - created sorted (as bench.py does), at t = 20-40 s and after 600, 1800 and 3600 simulated seconds;
  - created in random order, at t = 20-40 s;
and the stages of the ordered pack (fresh order, reused order) against bsg_traf_pack and bsg_cd_unpermute alone.  With
each airspace the fraction of tile pairs the culled detection keeps (tests/test_traffic_order.py::kept_fraction).
Prints the card and its power limit with them."""
import os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes as C
import torch
from bluesky_gym_sasha_b200 import _lib
from bluesky_gym_sasha_b200.cd import _ptr
from tests.test_traffic_order import bench_like_airspace, kept_fraction

N, REPS = 100_000, int(os.environ.get("REPS", "20"))
dev = torch.device("cuda", 0)
median = lambda ts: sorted(ts)[len(ts) // 2]
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.TimeoutExpired):
    power = "unknown"
print(f"card {torch.cuda.get_device_name(dev)}, power limit {power}")


def alternate(pair):
    """Median device time [us] of one substep of each airspace, stepped alternately REPS times."""
    ev = {k: [] for k in pair}
    for _ in range(REPS):
        for k, g in pair.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); g.step(1); b.record()
            ev[k].append((a, b))
    torch.cuda.synchronize()
    return {k: median([a.elapsed_time(b) * 1e3 for a, b in v]) for k, v in ev.items()}


def report(label, pair):
    t = alternate(pair)
    on, off = pair["on"], pair["off"]
    f_on, f_off = kept_fraction(on.rec_ordered, N), kept_fraction(off.rec, N)
    print(f"{label:34s} t = {on.nstep * on.simdt:6.0f} s   on {t['on']:8.1f} us (keeps {f_on:6.2%})   "
          f"off {t['off']:8.1f} us (keeps {f_off:6.2%})   off / on {t['off'] / t['on']:5.2f}", flush=True)
    return t


for sorted_creation, label in ((True, "created sorted"), (False, "created in random order")):
    pair = {"on": bench_like_airspace(N, sorted_creation, reorder_dt=60.0), "off": bench_like_airspace(N, sorted_creation)}
    for g in pair.values():
        g.step(20)                                      # warm-up, as bench_traffic
    base = report(label, pair)
    if sorted_creation:
        for t_end in (600, 1800, 3600):
            for g in pair.values():
                g.step(t_end - g.nstep)
            t = report(label, pair)
            print(f"{'':34s} on: {t['on'] / base['on']:.2f} x its t = 20-40 s time, off: {t['off'] / base['off']:.2f} x")
    del pair
    torch.cuda.empty_cache()

# stages, on the sorted airspace: pack alone, ordered pack with a fresh / reused order, unpermute of the last detection
g = bench_like_airspace(N, True, reorder_dt=60.0)
g.step(20)
st = g._stream()
stages = {k: [] for k in ("bsg_traf_pack", "pack_ordered fresh order", "pack_ordered reused order", "bsg_cd_unpermute")}
ref = torch.empty_like(g.rec)
out = g.last
for r in range(2 * REPS):
    for k in stages:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        if k == "bsg_traf_pack":
            _lib.check(g.lib.bsg_traf_pack(C.byref(g.cfg), C.byref(g.tt), _ptr(ref), st))
        elif k == "bsg_cd_unpermute":           # (maps the lists again: a timing of the kernel, not of a valid result)
            _lib.check(g.lib.bsg_cd_unpermute(_ptr(g.perm), N, C.byref(g.cd.lists), *[_ptr(g.cd._buf[b_]) for b_ in
                                              ("nconf", "nlos", "tcpamax", "inconf")], *[_ptr(g.per_row[b_]) for b_ in
                                              ("nconf_row", "nlos_row", "tcpamax", "inconf")], st))
        else:
            _lib.check(g.lib.bsg_traf_pack_ordered(C.byref(g.cfg), C.byref(g.tt), int("fresh" in k), _ptr(g.perm),
                                                   _ptr(g.rec_ordered), _ptr(g.rec), _ptr(g.order_work), g.order_work.numel(), st))
        b.record()
        stages[k].append((a, b))
torch.cuda.synchronize()
nconf, nlos = (int(v) for v in out["npairs"].cpu())
print(f"stages at N = {N} (medians of {2 * REPS}; last detection listed {nconf} conflicts, {nlos} LoS):")
for k, v in stages.items():
    print(f"  {k:28s} {median([a.elapsed_time(b) * 1e3 for a, b in v]):8.1f} us")
