"""StateBasedCD -- single-airspace state-based conflict detection on the GPU (kernel K2).

Interface mirrored: ``StateBased.detect(ownship, intruder, rpz, hpz, dtlookahead)`` of upstream BlueSky
(restated in oracle/statebased.py) -> ``confpairs, lospairs, inconf, tcpamax, qdr, dist, dcpa, tcpa, tinconf``.  The reference
never switches ASAS on (merge_env.py:157 issues only ``reso off``); BASELINE.json's north_star adds it.
Inputs are float64 aircraft state (degrees, m/s, m) as numpy arrays or CUDA tensors; the work is done by
``bsg_cd_pack`` + ``bsg_cd_detect`` (include/bsg.h).  Multi-GPU: rows are block-sharded over ranks after
an NCCL all-gather of the 32-byte CD records (``detect_sharded``).  No CPU fallback.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib

NM, FT = 1852.0, 0.3048
ROW_OUTPUTS = ("nconf_row", "nlos_row", "tcpamax", "inconf")     # per-row outputs of a detection, bsg_cd_unpermute's order


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def cd_records(n, device, inert=False):
    """CD records for ``n`` aircraft (include/bsg.h: BSG_CD_TILE, BSG_CD_REC_*): a float32 tensor
    [tiles, CD_REC_FIELDS, CD_TILE] holding bsg_cd_padded(n) records, at least one tile.  ``inert=True``: every record
    starts as the inert padding record bsg_cd_pack writes (alt 3e9: never a conflict candidate)."""
    tiles = max(int(_lib.load().bsg_cd_padded(n)) // _lib.CD_TILE, 1)
    rec = (torch.zeros if inert else torch.empty)((tiles, _lib.CD_REC_FIELDS, _lib.CD_TILE), dtype=torch.float32, device=device)
    if inert:
        rec[:, _lib.CD_REC_CH, :] = 1.0
        rec[:, _lib.CD_REC_ALT, :] = 3.0e9
    return rec


def all_gather_records(rec_local, n_local, group=None, out=None):
    """The first ``n_local`` records of every rank's ``rec_local`` (whole tiles), all-gathered in rank order: the records
    of ``n_local * world`` aircraft.  ``out``: the buffer of an earlier call, reused when it is large enough."""
    import torch.distributed as dist
    assert n_local % _lib.CD_TILE == 0, "shard size must be a multiple of the 256-aircraft tile"
    tiles = n_local // _lib.CD_TILE
    world = dist.get_world_size(group)
    if out is None or out.shape[0] < tiles * world:
        out = cd_records(n_local * world, rec_local.device)
    dist.all_gather_into_tensor(out[:tiles * world], rec_local[:tiles].contiguous(), group=group)
    return out


def host_lists(out, lists, per_aircraft):
    """Host form of a detection's pair lists (``detect_packed`` with ``want_pairs``; ``lists``: its ``StateBasedCD.lists``),
    as upstream's detect() returns them: ``confpairs``, ``lospairs`` (up to the lists' capacity, row-major order), the
    host arrays of ``per_aircraft``, ``n_conf``, ``n_los``, ``truncated`` (more pairs found than the lists hold), ``qdr,
    dist, dcpa, tcpa, tinconf`` per conflict.  Synchronises the device."""
    torch.cuda.synchronize(out["npairs"].device)
    n_conf, n_los = (int(v) for v in out["npairs"].cpu())
    k, kl = min(n_conf, lists.conf_cap), min(n_los, lists.los_cap)
    pairs, lospairs, attr = out["pairs"][:k], out["lospairs"][:kl], out["attr"][:k]
    # upstream's order: row-major np.where (own index, then intruder index).  Keys are unique, so one sort of the
    # combined 64-bit key on the device orders a list
    o = torch.argsort(pairs[:, 0].long() * (1 << 32) + pairs[:, 1].long())
    ol = torch.argsort(lospairs[:, 0].long() * (1 << 32) + lospairs[:, 1].long())
    attr = attr[o].cpu().numpy().astype(np.float64)
    res = dict(confpairs=pairs[o].cpu().numpy(), lospairs=lospairs[ol].cpu().numpy(), **per_aircraft,
               n_conf=n_conf, n_los=n_los, truncated=n_conf > lists.conf_cap or n_los > lists.los_cap)
    for c, name in enumerate(_lib.CD_ATTR):           # qdr, dist, dcpa, tcpa, tinconf of each conflict (detect()'s tail)
        res[name] = attr[:, c]
    return res


class StateBasedCD:
    def __init__(self, device=0, rpz=5.0 * NM, hpz=1000.0 * FT, dtlookahead=300.0, pair_capacity=1 << 22,
                 los_capacity=None):
        if not torch.cuda.is_available():
            raise _lib.BsgError("StateBasedCD needs a CUDA device: there is no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device("cuda", device)
        self.rpz, self.hpz, self.dtlookahead = float(rpz), float(hpz), float(dtlookahead)
        self.pair_capacity = int(pair_capacity)
        self.los_capacity = int(pair_capacity if los_capacity is None else los_capacity)
        self.gpu_launches = 0
        self._buf = {}
        self.lists = None                   # bsg_cd_lists of the last detection (_lists)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _as_dev(self, x):
        if isinstance(x, torch.Tensor):
            return x.to(device=self.device, dtype=torch.float64).contiguous()
        return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device=self.device)

    def _get(self, name, shape, dtype):
        t = self._buf.get(name)
        if t is None or t.shape != tuple(shape) or t.dtype != dtype:
            t = torch.zeros(shape, dtype=dtype, device=self.device)
            self._buf[name] = t
        return t

    # ---------------------------------------------------------------- packing
    def pack(self, lat, lon, trk, gs, alt, vs, lat0, lon0, out=None):
        """float64 SoA -> CD records (``cd_records``; padding = inert aircraft)."""
        arrs = [self._as_dev(a) for a in (lat, lon, trk, gs, alt, vs)]
        n = arrs[0].numel()
        rec = out if out is not None else cd_records(n, self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.bsg_cd_pack(*[_ptr(a) for a in arrs], n, float(lat0), float(lon0), _ptr(rec),
                                            self._stream()))
        self.gpu_launches += 1
        return rec, n

    def pack_ordered(self, lat, lon, trk, gs, alt, vs, lat0, lon0, out=None):
        """``pack`` with the aircraft laid out in a spatially coherent order chosen on the device (bsg_cd_pack_ordered:
        grid binning, counting sort -- what makes the culled detection effective).  Returns (rec, n, perm): record k holds
        aircraft ``perm[k]`` (int32 device tensor)."""
        arrs = [self._as_dev(a) for a in (lat, lon, trk, gs, alt, vs)]
        n = arrs[0].numel()
        rec = out if out is not None else cd_records(n, self.device)
        perm = torch.empty((n,), dtype=torch.int32, device=self.device)
        nbytes = int(self.lib.bsg_cd_order_workspace(n))
        work = self._get("order_work", (nbytes,), torch.uint8)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.bsg_cd_pack_ordered(*[_ptr(a) for a in arrs], n, float(lat0), float(lon0), _ptr(rec), _ptr(perm),
                                                    _ptr(work), nbytes, self._stream()))
        self.gpu_launches += 6
        return rec, n, perm

    # ---------------------------------------------------------------- detection on packed records
    def _lists(self, want_pairs, want_attr=True):
        """Device pair lists of one detection (include/bsg.h::bsg_cd_lists) and the ctypes view handed to the library, which
        also stays in ``self.lists``."""
        npairs = self._get("npairs", (2,), torch.int64)
        pairs = self._get("pairs", (max(self.pair_capacity, 1), 2), torch.int32) if want_pairs else None
        attr = self._get("attr", (max(self.pair_capacity, 1), len(_lib.CD_ATTR)), torch.float32) if want_pairs and want_attr else None
        los = self._get("lospairs", (max(self.los_capacity, 1), 2), torch.int32) if want_pairs else None
        lists = _lib.CdLists(d_conf_pairs=_ptr(pairs), d_conf_attr=_ptr(attr), conf_cap=self.pair_capacity if want_pairs else 0,
                             d_los_pairs=_ptr(los), los_cap=self.los_capacity if want_pairs else 0, d_npairs=_ptr(npairs))
        self.lists = lists
        return lists, dict(pairs=pairs, attr=attr, lospairs=los, npairs=npairs)

    def detect_packed(self, rec, n_all, row0=0, n_rows=None, lon_wrap=False, want_pairs=True, cull=False, symmetric=False,
                      want_attr=True, deal=None):
        """Rows [row0, row0+n_rows) x all n_all columns.  Asynchronous; returns device tensors: per-row ``nconf_row``,
        ``nlos_row``, ``tcpamax``, ``inconf``; ``npairs`` = (conflicts, LoS pairs) found; with ``want_pairs`` the lists
        ``pairs`` [cap, 2] (+ ``attr`` [cap, 5] = qdr, dist, dcpa, tcpa, tinconf per conflict) and ``lospairs`` [cap, 2].
        ``self.lists`` holds the ``_lib.CdLists`` view of those lists that the detection wrote.
        ``cull=True``: bsg_cd_detect_culled (identical outputs; pays off on spatially sorted records).
        ``symmetric=True`` (full N x N only): each unordered tile pair is evaluated once and both ordered results are
        emitted (BSG_CD_SYMMETRIC; identical outputs, half the pair evaluations); combines with ``cull``."""
        n_rows = n_all - row0 if n_rows is None else n_rows
        m = max(n_rows, 1)
        nconf = self._get("nconf", (m,), torch.int32)
        nlos = self._get("nlos", (m,), torch.int32)
        tcpamax = self._get("tcpamax", (m,), torch.float32)
        inconf = self._get("inconf", (m,), torch.uint8)
        lists, lt = self._lists(want_pairs, want_attr)
        flags = _lib.CD_LON_WRAP if lon_wrap else 0
        if symmetric:
            flags |= _lib.CD_SYMMETRIC | (0 if cull else _lib.CD_ALLTILES)
        if deal is not None:                # (BSG_CD_DEAL(n, k): this GPU's share of the row blocks, see detect_sharded_symmetric)
            flags |= ((int(deal[0]) & 0xff) << 8) | ((int(deal[1]) & 0xff) << 16)
        with torch.cuda.device(self.device):
            if cull or symmetric:
                nbytes = int(self.lib.bsg_cd_cull_workspace(n_all, n_rows))
                work = self._get("cull_work", (nbytes,), torch.uint8)
                _lib.check(self.lib.bsg_cd_detect_culled(_ptr(rec), n_all, row0, n_rows, self.rpz, self.hpz, self.dtlookahead,
                                                         flags, _ptr(nconf), _ptr(nlos), _ptr(tcpamax), _ptr(inconf),
                                                         C.byref(lists), _ptr(work), nbytes, self._stream()))
                self.gpu_launches += 5 if n_rows else 0
            else:
                _lib.check(self.lib.bsg_cd_detect(_ptr(rec), n_all, row0, n_rows, self.rpz, self.hpz, self.dtlookahead,
                                                  flags, _ptr(nconf), _ptr(nlos), _ptr(tcpamax), _ptr(inconf),
                                                  C.byref(lists), self._stream()))
                self.gpu_launches += 2 if n_rows else 0
        return dict(nconf_row=nconf[:n_rows], nlos_row=nlos[:n_rows], tcpamax=tcpamax[:n_rows],
                    inconf=inconf[:n_rows], **lt)

    # ---------------------------------------------------------------- spatial order for the culled form
    @staticmethod
    def spatial_order(lat_d, lon_d, tile=256):
        """Permutation that makes consecutive records -- hence the kernel's 256-record tiles -- spatially compact,
        which is what makes tile culling effective: aircraft are cut into latitude strips holding a whole number of
        tiles each and sorted by longitude within a strip, with the strip count chosen so that a tile's footprint is
        roughly square.
        (torch ops: plumbing, O(N log N) on the device.)"""
        n = lat_d.numel()
        la0, la1 = float(lat_d.min()), float(lat_d.max())
        lo0, lo1 = float(lon_d.min()), float(lon_d.max())
        h = max(la1 - la0, 1e-9)
        w = max((lo1 - lo0) * np.cos(np.radians(0.5 * (la0 + la1))), 1e-9)
        n_tiles = max(1, -(-n // tile))
        strips = int(max(1, round(np.sqrt(n_tiles * h / w))))
        per_strip = -(-n_tiles // strips) * tile          # whole tiles per strip: no tile straddles two strips
        rank = torch.empty(n, dtype=torch.int64, device=lat_d.device)
        rank[torch.argsort(lat_d)] = torch.arange(n, device=lat_d.device)
        key = (rank // per_strip).to(torch.float64) * 1024.0 + (lon_d - lo0)          # lon span < 360 < 1024
        return torch.argsort(key)

    # ---------------------------------------------------------------- convenience: StateBased.detect
    def detect(self, lat, lon, trk, gs, alt, vs, lat0=None, lon0=None, cull=True, symmetric=True):
        """Full N x N detection.  Returns host results shaped like upstream's ``detect`` outputs.  By default the fastest
        form with identical outputs is used (culled + symmetric); ``cull=False, symmetric=False`` evaluates every ordered
        pair.  ``cull=True`` sorts the aircraft into spatially compact tiles and skips tile pairs that are out of each other's
        reach (bsg_cd_detect_culled); results are identical, indices are mapped back to the caller's order."""
        lat_d, lon_d = self._as_dev(lat), self._as_dev(lon)
        n = lat_d.numel()
        if n == 0:
            z = np.zeros(0)
            return dict(confpairs=np.zeros((0, 2), np.int32), lospairs=np.zeros((0, 2), np.int32), inconf=z.astype(bool),
                        tcpamax=z, nconf_row=z.astype(np.int64), nlos_row=z.astype(np.int64), n_conf=0, n_los=0,
                        truncated=False, **{k: z.copy() for k in _lib.CD_ATTR})
        if lat0 is None:
            lat0 = float(lat_d.mean())
        if lon0 is None:
            lon0 = float(lon_d[0])
        span = float((((lon_d - lon0) + 180.0) % 360.0 - 180.0).abs().max())
        cull = cull and span < 90.0                       # (airspaces across the antimeridian: plain form)
        if cull:
            rec, n, perm = self.pack_ordered(lat_d, lon_d, trk, gs, alt, vs, lat0, lon0)
        else:
            rec, n = self.pack(lat_d, lon_d, trk, gs, alt, vs, lat0, lon0)
        out = self.detect_packed(rec, n, lon_wrap=span >= 90.0, cull=cull, symmetric=symmetric and span < 90.0)
        if cull:                                          # back to the caller's aircraft order
            out = self.unpermute(perm, n, out)
        return host_lists(out, self.lists, dict(inconf=out["inconf"].cpu().numpy().astype(bool),
                                                tcpamax=out["tcpamax"].cpu().numpy().astype(np.float64),
                                                nconf_row=out["nconf_row"].cpu().numpy().astype(np.int64),
                                                nlos_row=out["nlos_row"].cpu().numpy().astype(np.int64)))

    def unpermute(self, perm, n, out, per_row=None):
        """Outputs of ``detect_packed`` on records in the order ``perm`` (record k = aircraft ``perm[k]``) in aircraft
        order (bsg_cd_unpermute, asynchronous): the pair lists of ``self.lists`` are rewritten in place, the per-row outputs
        scattered into ``per_row`` (dict of ``nconf_row, nlos_row, tcpamax, inconf`` tensors of at least n rows; default:
        buffers of this object).  Returns ``out`` with the per-row entries replaced by the first n rows of those."""
        if per_row is None:
            per_row = {k: self._get("unperm_" + k, (max(n, 1),), out[k].dtype) for k in ROW_OUTPUTS}
        with torch.cuda.device(self.device):
            _lib.check(self.lib.bsg_cd_unpermute(_ptr(perm), n, C.byref(self.lists), *[_ptr(out[k]) for k in ROW_OUTPUTS],
                                                 *[_ptr(per_row[k]) for k in ROW_OUTPUTS], self._stream()))
        self.gpu_launches += 1
        return dict(out, **{k: per_row[k][:n] for k in ROW_OUTPUTS})

    # ---------------------------------------------------------------- multi-GPU: rows sharded over ranks
    def detect_sharded(self, rec_local, n_local, group=None, lon_wrap=False, want_pairs=False, cull=False):
        """Each rank owns ``n_local`` aircraft (the same count on every rank, a multiple of 256 so blocks
        stay tile-aligned).  One NCCL all-gather of the packed records, then this rank evaluates its own
        rows against all columns; per-row outputs stay with the owner.  ``cull=True`` (bsg_cd_detect_culled) pays off when
        the global record order is spatially coherent (``spatial_order`` applied before the blocks were dealt out)."""
        import torch.distributed as dist
        world = dist.get_world_size(group)
        rank = dist.get_rank(group)
        allrec = self._buf["allrec"] = all_gather_records(rec_local, n_local, group, self._buf.get("allrec"))
        return self.detect_packed(allrec, n_local * world, row0=rank * n_local, n_rows=n_local,
                                  lon_wrap=lon_wrap, want_pairs=want_pairs, cull=cull)


    def detect_sharded_symmetric(self, rec_local, n_local, group=None, cull=False, want_pairs=False):
        """Like ``detect_sharded``, but every unordered tile pair is evaluated once in the whole job (BSG_CD_SYMMETRIC) with
        the row blocks dealt round-robin to the ranks (BSG_CD_DEAL): half the pair evaluations of the row-sharded form.  A
        rank's kernel posts results to rows anywhere in the airspace, so the per-aircraft outputs are all-reduced (three small
        collectives) and every rank ends up with the complete ``nconf_row / nlos_row / tcpamax / inconf`` of ALL aircraft;
        ``npairs`` holds the global totals.  Pair lists (``want_pairs``) stay partitioned by tile-pair owner."""
        import torch.distributed as dist
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        allrec = self._buf["allrec"] = all_gather_records(rec_local, n_local, group, self._buf.get("allrec"))
        out = self.detect_packed(allrec, n_local * world, want_pairs=want_pairs, cull=cull, symmetric=True, deal=(world, rank))
        counts = self._get("sym_counts", (2, n_local * world), torch.int32)
        counts[0].copy_(out["nconf_row"])
        counts[1].copy_(out["nlos_row"])
        dist.all_reduce(counts, group=group)
        dist.all_reduce(out["tcpamax"], op=dist.ReduceOp.MAX, group=group)
        dist.all_reduce(out["npairs"], group=group)
        out["nconf_row"], out["nlos_row"] = counts[0], counts[1]
        out["inconf"] = counts[0] > 0
        return out

    # ---------------------------------------------------------------- multi-GPU without a gather (peer memory)
    def detect_sharded_p2p(self, rec_local, n_local, group=None, want_pairs=False, cull=False):
        """Same decomposition as ``detect_sharded`` but with NO collective on the data path: every rank copies its packed
        block into a symmetric-memory buffer (torch.distributed._symmetric_memory: peer-addressable allocation +
        device-side barrier; plumbing), and ``bsg_cd_detect_peers`` reads the column tiles it needs straight from the
        owners over NVLink with the kernel's TMA bulk copies.  With ``cull=True`` only tiles that survive culling
        ever cross the link."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        group = group if group is not None else dist.group.WORLD
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        assert n_local % _lib.CD_TILE == 0 and world <= 8, "shard size must be a multiple of 256; one node (<= 8 GPUs)"
        local = rec_local[:n_local // _lib.CD_TILE]
        st = self._buf.get("symm")
        if st is None or st[0] != n_local:
            buf = symm.empty(local.shape, dtype=torch.float32, device=self.device)
            hdl = symm.rendezvous(buf, group)
            ptrs = (C.c_void_p * world)(*[int(p) for p in hdl.buffer_ptrs])
            st = (n_local, buf, hdl, ptrs)
            self._buf["symm"] = st
        _, buf, hdl, ptrs = st
        buf.copy_(local)
        hdl.barrier(channel=0)                  # every rank's block is in place (device-side, on the current stream)
        m = n_local
        nconf = self._get("nconf", (m,), torch.int32)
        nlos = self._get("nlos", (m,), torch.int32)
        tcpamax = self._get("tcpamax", (m,), torch.float32)
        inconf = self._get("inconf", (m,), torch.uint8)
        lists, lt = self._lists(want_pairs)
        work, nbytes = None, 0
        if cull:
            nbytes = int(self.lib.bsg_cd_cull_workspace(n_local * world, n_local))
            work = self._get("cull_work", (nbytes,), torch.uint8)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.bsg_cd_detect_peers(ptrs, world, rank, n_local, self.rpz, self.hpz, self.dtlookahead,
                                                    _lib.CD_CULL if cull else 0, _ptr(nconf), _ptr(nlos), _ptr(tcpamax),
                                                    _ptr(inconf), C.byref(lists), _ptr(work), nbytes, self._stream()))
        hdl.barrier(channel=1)                  # nobody overwrites a block that a peer may still be reading
        self.gpu_launches += 5 if cull else 2
        return dict(nconf_row=nconf, nlos_row=nlos, tcpamax=tcpamax, inconf=inconf, **lt)


def shard_rows(n_all, world, rank):
    """Block partition used by ``detect_sharded`` and its CPU (gloo) tests: [row0, row0 + n_rows)."""
    per = n_all // world
    return rank * per, per
