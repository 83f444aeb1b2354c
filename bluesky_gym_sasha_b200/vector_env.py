"""BlueSkyVectorEnv -- the batched, device-resident front-end of the accelerated step path.

API boundary mirrored: ``gymnasium.vector.VectorEnv`` over the reference's env classes
(``Env.reset`` / ``Env.step`` of bluesky_gym/envs/*.py, registered in bluesky_gym/__init__.py:4-46).
PyTorch is plumbing only: it owns the device tensors (structure-of-arrays aircraft state, per-env
records, obs / reward / flag outputs) and the pinned host mirrors; every computation is a call into
libbsg_b200.so through the C ABI of include/bsg.h.  There is no CPU path.

Two ways to drive it:
  * ``reset()`` / ``step(actions)``      -- numpy in / numpy float64 out (gymnasium, SB3, RLlib);
    each step copies actions host->device and obs / reward / flags / info device->host
    (``bsg_step_host_block``).
  * ``reset_torch()`` / ``step_torch(a)`` -- CUDA float32 tensors in / out, no host sync.
"""
import ctypes as C
import sys
from collections import OrderedDict

import numpy as np
import torch

from . import _lib
from .gym_compat import VectorEnv, batch_space, spaces
from .spec import A320_PERF, AUTORESET, NOT_ACCELERATED, SPECS


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class _HostBlock:
    """One pinned host block with the device output block's layout, a dense terminal-observation area behind it, and the
    numpy views of both, made ONCE.  Every array handed to the caller is a view whose ``.base`` collapses to ``root`` (numpy
    keeps the base of a view of a view pointing at the first array that is not itself an ndarray view), so
    ``sys.getrefcount(root)`` above its value at construction means the caller still holds results of the step that
    used this block: the caller owns a step's results for exactly as long as it keeps them and nothing is copied."""
    __slots__ = ("tensor", "root", "ptr", "v", "final", "dirty", "refs", "wroot", "wide", "wfinal", "wdirty", "wrefs")

    def __init__(self, env, pinned=True):
        E, L = env.num_envs, env.layout
        n_dense = E * L.obs_dim * 4 if env.autoreset_mode == "same_step" else 0
        self.tensor = torch.zeros((env._out_bytes + n_dense,), dtype=torch.uint8)
        if pinned:
            self.tensor = self.tensor.pin_memory()
        self.root = self.tensor.numpy()
        self.ptr = self.tensor.data_ptr()
        v = {k: self.root[off:off + n * np.dtype(dt).itemsize].view(dt) for k, (off, dt, n) in env._off.items()}
        v["obs"] = v["obs"].reshape(E, L.obs_dim)
        v["info"] = v["info"].reshape(L.info_dim, E)
        v["final_obs"] = v["final_obs"].reshape(env._final_cap, L.obs_dim)
        self.v = v
        self.final = self.root[env._out_bytes:].view(np.float32).reshape(E, L.obs_dim) if n_dense else None
        self.dirty = None               # rows of `final` written by the last step that used this block
        self.wroot = self.wide = self.wfinal = self.wdirty = None
        self.wrefs = 0
        self.refs = sys.getrefcount(self.root)

    def widen_area(self, env):
        """float64 twin of the obs and dense terminal-obs areas (the dtype the reference's spaces declare): ordinary
        memory, touched once here so that no step pays its page faults"""
        if self.wroot is None:
            E, L = env.num_envs, env.layout
            self.wroot = np.zeros(2 * E * L.obs_dim, dtype=np.float64)
            self.wroot.fill(0.0)
            self.wide = self.wroot[:E * L.obs_dim].reshape(E, L.obs_dim)
            self.wfinal = self.wroot[E * L.obs_dim:].reshape(E, L.obs_dim)
            self.wrefs = sys.getrefcount(self.wroot)
        return self.wide

    def held(self):
        return sys.getrefcount(self.root) != self.refs or (self.wroot is not None and sys.getrefcount(self.wroot) != self.wrefs)


class BlueSkyVectorEnv(VectorEnv):
    metadata = {"render_modes": ["rgb_array"], "autoreset_mode": "next_step"}

    def __init__(self, env_id, num_envs, device=0, seed=0, cd_enabled=False, n_intruders=None,
                 autoreset_mode="next_step", env_id_offset=0, max_episode_steps=None, perf=None,
                 default_hdg="random", rpz=0.0, hpz=0.0, dtlookahead=0.0, render_mode=None,
                 obs_dtype=np.float32, copy=True, obs_noise=0.0, wind=None, wind_obs=False,
                 ac_density_mode="normal", init_alt=0.0, cd_pairs=False):
        if env_id in NOT_ACCELERATED:
            raise NotImplementedError(f"{env_id} is registered by the reference but is not on the accelerated "
                                      "path yet (SURVEY.md section 8f)")
        if env_id not in SPECS:
            raise KeyError(f"unknown env id {env_id!r}")
        assert render_mode in (None, "rgb_array"), "render_mode is None or 'rgb_array' (frames of one env index: render())"
        if not torch.cuda.is_available():
            raise _lib.BsgError("BlueSkyVectorEnv needs a CUDA device: there is no CPU fallback")
        self.spec_b200 = SPECS[env_id]
        self.env_id = env_id
        self.num_envs = int(num_envs)
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        self.render_mode = render_mode
        # float32 arrays are valid members of the reference's float64 Box spaces (gymnasium checks
        # np.can_cast); the scalar Env classes ask for float64 to be byte-for-byte drop-in.
        self.obs_dtype = np.dtype(obs_dtype)
        self.copy = bool(copy)          # False: return views of two rotating pinned buffers (valid for 2 steps)
        self.autoreset_mode = autoreset_mode
        self.metadata = dict(self.metadata, autoreset_mode=autoreset_mode)
        n_int = n_intruders if n_intruders is not None else self.spec_b200.default_kwargs.get("n_intruders", 0)
        self.n_intruders = n_int

        lib = _lib.load()
        pf = _lib.Perf(**{**A320_PERF, **(perf or {})})
        self.cfg = _lib.Config(
            env_type=self.spec_b200.env_type, num_envs=self.num_envs, n_intruders=n_int,
            cd_enabled=(2 if cd_enabled == 2 else int(bool(cd_enabled))), autoreset_mode=AUTORESET[autoreset_mode],
            max_episode_steps=self.spec_b200.max_episode_steps if max_episode_steps is None else int(max_episode_steps),
            default_hdg_random=1 if default_hdg == "random" else 0, device=self.device.index,
            seed=int(seed) & (2 ** 64 - 1), env_id_offset=int(env_id_offset), rpz=rpz, hpz=hpz,
            dtlookahead=dtlookahead, perf=pf, wind_obs=int(bool(wind_obs)),
            sector_density_uniform=0 if ac_density_mode == "normal" else 1,     # sector_cr_env.py:98-103: anything else = uniform
            init_alt=float(init_alt))                   # HorizontalCR only: 0 = the reference; 3000 = SURVEY 8d's airborne variant
        self.layout = _lib.query_layout(self.cfg)
        L, E, G = self.layout, self.num_envs, self.layout.slots
        self.slots = G
        # in-sim ASAS pair lists (bs.traf.cd.confpairs / lospairs + per-conflict attributes of the last substep):
        # cd_pairs=True keeps up to 128 unordered pairs per env (or all of them when there are fewer), an int = that many
        self.cd_pair_cap = 0
        if cd_pairs and cd_enabled and G > 1:
            self.cd_pair_cap = min(G * (G - 1) // 2, 128) if cd_pairs is True else int(cd_pairs)
        self.cfg.cd_pair_cap = self.cd_pair_cap

        # ---- spaces (identical keys / shapes / dtype to the reference declarations)
        self.obs_layout, obs_dim = self.spec_b200.obs_layout(n_int)
        self.wind_obs = bool(wind_obs)
        if self.wind_obs:                       # wrappers/wind.py:17-23: two more keys at the end of the Dict
            self.obs_layout["wind_u"] = (obs_dim, 1, -np.inf, np.inf)
            self.obs_layout["wind_v"] = (obs_dim + 1, 1, -np.inf, np.inf)
            obs_dim += 2
        assert obs_dim == L.obs_dim, (obs_dim, L.obs_dim)
        self.single_observation_space = spaces.Dict(OrderedDict(
            (k, spaces.Box(lo, hi, shape=(w,), dtype=np.float64)) for k, (off, w, lo, hi) in self.obs_layout.items()))
        self.single_action_space = spaces.Box(-1, 1, shape=(L.act_dim,), dtype=np.float64)
        self.observation_space = batch_space(self.single_observation_space, E)
        self.action_space = batch_space(self.single_action_space, E)

        # ---- device state (torch owns the memory; the library only borrows pointers)
        dev = self.device
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)
        # step outputs live in ONE block (obs | reward | info | final_count | terminated | truncated | pad |
        # final_ids | final_obs rows) so that the host API brings them back with a single device->host copy
        # of the block's head (bsg_step_host_block): everything up to and including the first `_final_cap`
        # compacted terminal observations, which covers all envs that finish in a typical step
        n_obs, n_rew, n_info, n_cnt = E * L.obs_dim * 4, E * 4, E * L.info_dim * 4, 16
        o_info, o_cnt, o_term = n_obs + n_rew, n_obs + n_rew + n_info, n_obs + n_rew + n_info + n_cnt
        o_fids = (o_term + 2 * E + 15) // 16 * 16
        o_fobs = o_fids + 4 * E
        self._final_cap = min(E, max(8, E // 32))
        self._out_bytes = o_fobs + self._final_cap * L.obs_dim * 4       # mirrored on the host every step
        dev_bytes = o_fobs + E * L.obs_dim * 4

        def carve(block, n_final):
            o = block[:n_obs].view(torch.float32).view(E, L.obs_dim)
            r = block[n_obs:o_info].view(torch.float32)
            i = block[o_info:o_cnt].view(torch.float32).view(L.info_dim, E)          # key-major: one row per info key
            c = block[o_cnt:o_term].view(torch.int32)
            te = block[o_term:o_term + E]
            tr = block[o_term + E:o_term + 2 * E]
            fi = block[o_fids:o_fobs].view(torch.int32)
            fo = block[o_fobs:o_fobs + n_final * L.obs_dim * 4].view(torch.float32).view(n_final, L.obs_dim)
            return o, r, i, c, te, tr, fi, fo
        self._out_dev = z((dev_bytes,), torch.uint8)
        d_obs, d_rew, d_info, d_cnt, d_term, d_trunc, d_fids, d_fobs = carve(self._out_dev, E)
        self.t = OrderedDict(
            pos=z((E, G, 2), torch.float64), kin=z((E, G, 4), torch.float32), cmd=z((E, G, 4), torch.float32),
            aux=z((E, G, 4), torch.float32), flags=z((E, G), torch.int32),
            tcpamax=z((E, G), torch.float32), inconf=z((E, G), torch.uint8),
            env_f64=z((E, L.env_f64), torch.float64), env_f32=z((E, L.env_f32), torch.float32),
            env_i32=z((E, L.env_i32), torch.int32),
            poly=z((E, max(L.poly_f64, 1)), torch.float64) if L.poly_f64 else None,
            obs=d_obs, final_obs=d_fobs, final_ids=d_fids, final_count=d_cnt,
            reward=d_rew, terminated=d_term, truncated=d_trunc,
            info=d_info, actions_staging=z((E, L.act_dim), torch.float32),
            cd_pairs=z((E, self.cd_pair_cap), torch.int32) if self.cd_pair_cap else None,
            cd_attr=z((E, self.cd_pair_cap, _lib.PAIR_ATTR_COUNT), torch.float32) if self.cd_pair_cap else None)
        # host side of the numpy API: pinned blocks with the device block's layout (+ a dense terminal-observation area),
        # their numpy views made once (_HostBlock).  copy=True (default): a step takes a block none of whose views the
        # caller still holds, so the device->host transfer lands directly in memory the caller may keep -- no host copy;
        # the pool grows on demand (a rollout buffer that copies what it needs holds 1-2 blocks) up to `_BLOCKS_MAX`, a
        # caller that hoards more than that gets ordinary copies instead.  copy=False: the first two blocks take turns.
        self._off = dict(obs=(0, np.float32, E * L.obs_dim), reward=(n_obs, np.float32, E), info=(o_info, np.float32, E * L.info_dim),
                         final_count=(o_cnt, np.int32, 4), terminated=(o_term, np.uint8, E), truncated=(o_term + E, np.uint8, E),
                         final_ids=(o_fids, np.int32, E), final_obs=(o_fobs, np.float32, self._final_cap * L.obs_dim))
        self._blocks = [_HostBlock(self) for _ in range(3)]
        self._bsel = 0
        self._obs_views = None      # per-key views of the device observation tensor (made on first use)
        self._scratch = None        # (made on first use: the block behind copied-out results when the pool is exhausted)
        self._pending = None        # (block, copy_out) of a step_async() whose step_wait() has not run yet
        ph = lambda shape, dt: torch.zeros(shape, dtype=dt).pin_memory()
        self.h = dict(actions=ph((E, L.act_dim), torch.float32))
        self._act_np, self._act_ptr = self.h["actions"].numpy(), _ptr(self.h["actions"])
        self._h_final = ph((E, L.obs_dim), torch.float32)          # overflow beyond `_final_cap` rows (rare)
        self._h_final_np = self._h_final.numpy()

        self._h = C.c_void_p(0)
        with torch.cuda.device(dev):
            _lib.check(lib.bsg_create(C.byref(self.cfg), C.byref(self._h)))
            tt = _lib.TensorTable(**{k: _ptr(v) for k, v in self.t.items()})
            _lib.check(lib.bsg_bind_state(self._h, C.byref(tt)))
        self._lib = lib
        self.gpu_launches = 0
        self.closed = False
        self.obs_noise = 0.0
        if obs_noise:
            self.set_obs_noise(obs_noise)
        self._wind_t = None
        if wind is not None:
            self.set_wind(**wind)

    # ------------------------------------------------------------------ helpers
    def set_obs_noise(self, noise_level):
        """NoisyObservationWrapper on the device (bluesky_gym/wrappers/uncertainty.py): N(0, noise_level) on every
        observation element returned from now on; 0 switches it off."""
        _lib.check(self._lib.bsg_set_obs_noise(self._h, float(noise_level)))
        self.obs_noise = float(noise_level)

    ALT_STEP = 100.0 * 0.3048           # upstream windfield altitude axis: 100 ft steps up to 45 000 ft
    N_ALT = 451

    def set_wind(self, lat=None, lon=None, vnorth=None, veast=None, alt=None):
        """WindFieldWrapper on the device (bluesky_gym/wrappers/wind.py:28 ``bs.traf.wind.addpointvne``): wind vectors
        [m/s north / east] at the given lat / lon points; ``vnorth[k, i]`` is point i at ``alt[k]`` (``alt=None`` and one
        row = no altitude dependence).  ``set_wind()`` without arguments switches the wind off."""
        if lat is None:
            _lib.check(self._lib.bsg_set_wind(self._h, None))
            self._wind_t = None
            return
        dev = self.device
        lat = np.atleast_1d(np.asarray(lat, dtype=np.float64))
        lon = np.atleast_1d(np.asarray(lon, dtype=np.float64))
        vn = np.atleast_2d(np.asarray(vnorth, dtype=np.float64))
        ve = np.atleast_2d(np.asarray(veast, dtype=np.float64))
        n = len(lat)
        assert len(lon) == n and vn.shape[1] == n and ve.shape == vn.shape, "one wind vector (column) per point"
        if alt is None:
            n_alt, tab_n, tab_e = 1, vn[:1], ve[:1]
        else:                                   # per-point profile resampled on upstream's altitude axis
            axis = np.arange(self.N_ALT) * self.ALT_STEP
            wa = np.atleast_1d(np.asarray(alt, dtype=np.float64))
            n_alt = self.N_ALT
            tab_n = np.stack([np.interp(axis, wa, vn[:, i]) for i in range(n)], axis=1)
            tab_e = np.stack([np.interp(axis, wa, ve[:, i]) for i in range(n)], axis=1)
        f32 = lambda x: torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32), device=dev)
        t = dict(lat=f32(lat), lon=f32(lon), vn=f32(tab_n), ve=f32(tab_e))
        if self._wind_t is None or "gs" not in self._wind_t:
            # ground speed becomes state: start from the no-wind value of the current aircraft (tas along hdg)
            kin = self.t["kin"]
            h = torch.deg2rad(kin[..., 2])
            t["gs"] = torch.stack([kin[..., 1] * torch.cos(h), kin[..., 1] * torch.sin(h)], dim=-1).contiguous()
        else:
            t["gs"] = self._wind_t["gs"]
        self._install_wind(t, n, n_alt)

    def _install_wind(self, t, n, n_alt):
        w = _lib.Wind(n_points=n, n_alt=n_alt, alt_step=self.ALT_STEP, d_lat=t["lat"].data_ptr(), d_lon=t["lon"].data_ptr(),
                      d_vn=t["vn"].data_ptr(), d_ve=t["ve"].data_ptr(), d_gs=t["gs"].data_ptr())
        _lib.check(self._lib.bsg_set_wind(self._h, C.byref(w)))
        self._wind_t = t                         # keeps the device arrays alive while the library points at them
        self._wind_meta = dict(n_points=int(n), n_alt=int(n_alt))

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _obs_dict_np(self, flat):
        if flat.dtype != self.obs_dtype:
            f = flat.astype(self.obs_dtype)
        else:
            f = flat.copy() if self.copy else flat
        return OrderedDict((k, f[:, off:off + w]) for k, (off, w, _, _) in self.obs_layout.items())

    def _obs_dict_torch(self, flat):
        """Views of the bound observation tensor, one per key; made once (slicing a tensor costs ~2 us, eight of them per
        step were most of step_torch's host time) and handed out as a fresh dict per call."""
        if self._obs_views is None:
            self._obs_views = [(k, flat[:, off:off + w]) for k, (off, w, _, _) in self.obs_layout.items()]
        return OrderedDict(self._obs_views)

    def _infos_np(self, info):
        """info: [info_dim, E] float32 (key-major, as the device writes it): one row view per key, no conversion."""
        out = {k: info[i] for i, k in enumerate(self.spec_b200.info_keys)}
        if self.cfg.cd_enabled:
            out["asas_nconf"] = info[4].astype(np.int64)
            out["asas_nlos"] = info[5].astype(np.int64)
        return out

    # ------------------------------------------------------------------ device-tensor API (no host sync)
    def reset_torch(self, mask=None):
        """Resets every env (or those where ``mask`` is non-zero); returns the obs dict of CUDA tensors."""
        m = None if mask is None else mask.to(device=self.device, dtype=torch.uint8).contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.bsg_reset(self._h, _ptr(m), self._stream()))
        self.gpu_launches += 1
        return self._obs_dict_torch(self.t["obs"])

    def step_torch(self, actions):
        """actions: CUDA float32 [E, act_dim].  Returns (obs dict, reward, terminated, truncated) as views
        of the bound device tensors (overwritten by the next call)."""
        a = actions
        if a.dtype != torch.float32 or a.device != self.device or not a.is_contiguous():
            a = a.to(device=self.device, dtype=torch.float32).contiguous()
        assert a.shape == (self.num_envs, self.layout.act_dim), a.shape
        rc = self._lib.bsg_step(self._h, a.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream)
        if rc:
            _lib.check(rc)
        self.gpu_launches += 1
        return self._obs_dict_torch(self.t["obs"]), self.t["reward"], self.t["terminated"], self.t["truncated"]

    def traf_update(self, n_sub):
        """n_sub x bs.sim.step() only (kinematics + autopilot, no obs / reward); parity-test entry point."""
        with torch.cuda.device(self.device):
            _lib.check(self._lib.bsg_traf_update(self._h, int(n_sub), self._stream()))
        self.gpu_launches += 1

    # ------------------------------------------------------------------ gymnasium VectorEnv API (numpy)
    def reset(self, *, seed=None, options=None):
        if self._pending is not None:
            raise _lib.BsgError("reset(): a step_async() is in flight; call step_wait() first")
        if seed is not None:
            # gymnasium: reset(seed=s) re-seeds -- the same s always gives the same scenarios.  The streams are keyed by
            # (seed, global env id, episode) and the noise stream by (seed, global env id, call index), so the episode
            # counters and the call index restart with the new key.
            _lib.check(self._lib.bsg_set_seed(self._h, int(seed) & (2 ** 64 - 1)))
            self.cfg.seed = int(seed) & (2 ** 64 - 1)
            self.t["env_i32"][:, _lib.I32_EPISODE] = 0
            _lib.check(self._lib.bsg_set_noise_calls(self._h, 0))
        self.reset_torch()
        torch.cuda.synchronize(self.device)
        obs = self.t["obs"].cpu().numpy()
        info = self.t["info"].cpu().numpy()
        return self._obs_dict_np(obs), self._infos_np(info)

    _BLOCKS_MAX = 64

    def _acquire(self):
        """The host block for this step's results (see the constructor); second value: the results must be copied out
        because the caller holds every block of a full pool."""
        blocks = self._blocks
        if not self.copy:
            self._bsel ^= 1
            return blocks[self._bsel], False
        for b in blocks:
            if not b.held():
                return b, False
        if len(blocks) < self._BLOCKS_MAX:
            blocks.append(_HostBlock(self))
            return blocks[-1], False
        if self._scratch is None:
            self._scratch = _HostBlock(self)
        return self._scratch, True

    def step(self, actions):
        if self._pending is not None:
            raise _lib.BsgError("step(): a step_async() is in flight; call step_wait() first")
        E = self.num_envs
        self._act_np[...] = np.asarray(actions, dtype=np.float32).reshape(E, self.layout.act_dim)
        b, copy_out = self._acquire()
        # (the library sets the device itself; the stream is looked up per call because callers may switch streams)
        rc = self._lib.bsg_step_host_block(self._h, self._act_ptr, b.ptr, self._out_bytes,
                                           torch.cuda.current_stream(self.device).cuda_stream)
        if rc:
            _lib.check(rc)
        self.gpu_launches += 1
        return self._step_results(b, copy_out)

    def step_async(self, actions):
        """First half of ``step`` (the SB3 / older-gymnasium ``step_async`` / ``step_wait`` pair): copies the actions in,
        enqueues the step and the transfer of its results, and returns at once -- the caller's own work (policy
        bookkeeping, logging, the optimiser) overlaps the ~0.1 ms the device and the bus are busy."""
        if self._pending is not None:
            raise _lib.BsgError("step_async(): the previous step has not been waited for (one step in flight per env batch)")
        E = self.num_envs
        self._act_np[...] = np.asarray(actions, dtype=np.float32).reshape(E, self.layout.act_dim)
        b, copy_out = self._acquire()
        rc = self._lib.bsg_step_host_begin(self._h, self._act_ptr, b.ptr, self._out_bytes,
                                           torch.cuda.current_stream(self.device).cuda_stream)
        if rc:
            _lib.check(rc)
        self.gpu_launches += 1
        self._pending = (b, copy_out)

    def step_wait(self):
        """Second half: waits for the step enqueued by ``step_async`` and returns what ``step`` returns."""
        pend = getattr(self, "_pending", None)
        if pend is None:
            raise RuntimeError("step_wait() without step_async()")
        self._pending = None
        rc = self._lib.bsg_step_host_wait(self._h, pend[0].ptr, None, 0)
        if rc:
            _lib.check(rc)
        return self._step_results(*pend)

    def _step_results(self, b, copy_out=False):
        """The (obs, reward, terminated, truncated, infos) tuple from host block ``b``: views of the block (the caller's
        for as long as it keeps them, see _HostBlock), float64 observations widened into the block's float64 twin."""
        h = b.v
        flat = h["obs"]
        wide = self.obs_dtype == np.float64
        if wide:                                 # the reference's declared dtype: widened by the library's host threads
            dst = b.widen_area(self)
            _lib.check(self._lib.bsg_host_widen(dst.ctypes.data, flat.ctypes.data, flat.size))
            flat = dst
        elif flat.dtype != self.obs_dtype:
            flat = flat.astype(self.obs_dtype)
        if copy_out:
            flat = flat.copy()
        obs = OrderedDict((k, flat[:, off:off + w]) for k, (off, w, _, _) in self.obs_layout.items())
        rew = h["reward"].astype(np.float64)
        term = h["terminated"].astype(bool)
        trunc = h["truncated"].astype(bool)
        infos = self._infos_np(h["info"].copy() if copy_out else h["info"])
        if self.autoreset_mode == "same_step":
            # terminal observations, dense [E, obs_dim] with zero rows for the envs that did not finish: the block's own
            # area; only the rows written by the block's previous step are cleared, only the finished envs' rows written
            fo = b.wfinal if wide else b.final
            dirty = b.wdirty if wide else b.dirty
            if dirty is not None:
                fo[dirty] = 0.0
                dirty = None
            fc = h["final_count"]
            n_fin = int(fc[fc[2]])              # two counters take turns; [2] names the live one (include/bsg.h)
            if n_fin:                   # compacted terminal observations of the envs that finished in this step
                ids = h["final_ids"][:n_fin].copy()
                cap = self._final_cap
                fo[ids[:cap]] = h["final_obs"][:min(n_fin, cap)]
                if n_fin > cap:         # more finished than the mirrored window holds: fetch the rest
                    self._h_final[cap:n_fin].copy_(self.t["final_obs"][cap:n_fin], non_blocking=True)
                    torch.cuda.current_stream(self.device).synchronize()
                    fo[ids[cap:]] = self._h_final_np[cap:n_fin]
                dirty = ids
                out = fo.copy() if copy_out else (fo if fo.dtype == self.obs_dtype else fo.astype(self.obs_dtype))
                infos["final_obs"] = OrderedDict((k, out[:, off:off + w]) for k, (off, w, _, _) in self.obs_layout.items())
                infos["_final_obs"] = term | trunc
            if wide:
                b.wdirty = dirty
            else:
                b.dirty = dirty
        return obs, rew, term, trunc, infos

    def asas_pairs(self, e):
        """In-sim ASAS pair lists of env ``e`` after the last simulator substep, shaped like upstream's
        ``StateBased.detect`` outputs (what ``bs.traf.cd`` holds after ``bs.sim.step()``): ``confpairs`` / ``lospairs`` as
        ordered (own slot, intruder slot) pairs in row-major order, and per conflict ``qdr, dist, dcpa, tcpa, tinconf``.
        Needs ``cd_enabled`` and ``cd_pairs`` at construction.  ``truncated`` tells that the env had more pairs than the
        list holds."""
        if not self.cd_pair_cap:
            raise _lib.BsgError("asas_pairs(): construct the env with cd_enabled=True, cd_pairs=True")
        n = int(self.t["env_i32"][e, _lib.I32_NPAIRS])
        k = min(n, self.cd_pair_cap)
        ent = self.t["cd_pairs"][e, :k].cpu().numpy().view(np.uint32)
        att = self.t["cd_attr"][e, :k].cpu().numpy().astype(np.float64)
        i, j = (ent & 0xff).astype(np.int64), ((ent >> 8) & 0xff).astype(np.int64)
        cij, cji, los = (ent & _lib.PAIR_CONF_IJ) != 0, (ent & _lib.PAIR_CONF_JI) != 0, (ent & _lib.PAIR_LOS) != 0
        own = np.concatenate([i[cij], j[cji]])
        intr = np.concatenate([j[cij], i[cji]])
        qdr = np.concatenate([att[cij, 0], (att[cji, 0] + 180.0) % 360.0])
        cols = {"dist": 1, "dcpa": 2, "tcpa": 3}
        vals = {name: np.concatenate([att[cij, c], att[cji, c]]) for name, c in cols.items()}
        tin = np.concatenate([att[cij, 4], att[cji, 5]])
        o = np.lexsort((intr, own))
        lown, lintr = np.concatenate([i[los], j[los]]), np.concatenate([j[los], i[los]])
        ol = np.lexsort((lintr, lown))
        return dict(confpairs=np.stack([own[o], intr[o]], axis=1), lospairs=np.stack([lown[ol], lintr[ol]], axis=1),
                    qdr=qdr[o], tinconf=tin[o], truncated=n > self.cd_pair_cap, **{k_: v[o] for k_, v in vals.items()})

    def reset_flags(self):
        """Per-env bit mask left by the last scenario generation (include/bsg.h BSG_I32_RESET_FLAGS): 1 = polygon area
        below the reference's threshold when the vertex cap was hit, 2 = aircraft count clipped to the slot count,
        4 = rejection sampling gave up (the reference raises there, static_obstacle_env.py:215-216)."""
        return self.t["env_i32"][:, _lib.I32_RESET_FLAGS].cpu().numpy()

    # ------------------------------------------------------------------ state access (parity tests, checkpoints)
    def _config_key(self):
        c = self.cfg
        return dict(env_id=self.env_id, num_envs=self.num_envs, n_intruders=self.n_intruders, seed=int(c.seed),
                    env_id_offset=int(c.env_id_offset), cd_enabled=int(c.cd_enabled), autoreset_mode=self.autoreset_mode,
                    max_episode_steps=int(c.max_episode_steps), wind_obs=int(c.wind_obs), init_alt=float(c.init_alt),
                    sector_density_uniform=int(c.sector_density_uniform), default_hdg_random=int(c.default_hdg_random),
                    cd_pair_cap=int(c.cd_pair_cap))

    def state_dict(self):
        """Checkpoint: clones of every device tensor that carries simulator state (aircraft SoA, per-env records,
        polygons, last outputs), the wind field with its ground-speed state, the observation-noise level and the noise
        stream's call index, and the configuration the streams are keyed by (seed, env id offset, ...)."""
        sd = {k: v.clone() for k, v in self.t.items() if v is not None and k != "actions_staging"}
        if self._wind_t is not None:
            sd["wind"] = {k: v.clone() for k, v in self._wind_t.items()}
            sd["wind_meta"] = dict(self._wind_meta)
        calls = C.c_uint32(0)
        _lib.check(self._lib.bsg_get_noise_calls(self._h, C.byref(calls)))
        sd["obs_noise"] = dict(sigma=float(self.obs_noise), calls=int(calls.value))
        sd["config"] = self._config_key()
        return sd

    def load_state_dict(self, sd):
        """Resume from ``state_dict()``: the env continues bit for bit (same future scenario draws and noise stream),
        also when loaded into a freshly built env.  The seed is taken from the checkpoint; any other difference between
        the checkpoint's configuration and this env's raises."""
        cfg = sd.get("config")
        if cfg is not None:
            mine = self._config_key()
            diff = {k: (v, mine[k]) for k, v in cfg.items() if k != "seed" and mine[k] != v}
            if diff:
                raise ValueError(f"load_state_dict: checkpoint was taken from a different configuration {diff}")
            if cfg["seed"] != mine["seed"]:
                _lib.check(self._lib.bsg_set_seed(self._h, cfg["seed"]))
                self.cfg.seed = cfg["seed"]
        if "wind" in sd:
            w, m = sd["wind"], sd["wind_meta"]
            t = {k: v.clone() for k, v in w.items()}
            self._install_wind(t, m["n_points"], m["n_alt"])
        elif cfg is not None and self._wind_t is not None:
            self.set_wind()
        for k, v in sd.items():
            if k in self.t and self.t[k] is not None and k != "final_count":      # (an output whose slot parity lives in the handle)
                self.t[k].copy_(v)
        if "obs_noise" in sd:
            self.set_obs_noise(sd["obs_noise"]["sigma"])
            _lib.check(self._lib.bsg_set_noise_calls(self._h, sd["obs_noise"]["calls"]))

    def load_state(self, e, lat, lon, alt, tas, hdg, vs, selspd, selalt, selvs, ap_trk, cas, ax=None,
                   lnav=None, iactwp=None, curlegdir=None, env_f64=None, env_i32=None, env_f32=None, poly=None):
        """Injects a (reference / oracle) post-reset traffic state into env ``e`` through ``bsg_load_state``
        (include/bsg.h; SURVEY 8b).  ``env_f64`` / ``env_i32`` / ``env_f32`` are {index: value} patches of the env's
        current records; ``poly`` replaces the polygon record (zero-padded)."""
        n = len(lat)
        assert n <= self.slots
        keep = []

        def arr(x, dt=np.float64):
            if x is None:
                return None
            a = np.ascontiguousarray(np.broadcast_to(np.asarray(x, dtype=dt), (n,)))
            keep.append(a)
            return a.ctypes.data

        def record(name, patch, dt):
            if not patch:
                return None
            r = self.t[name][e].cpu().numpy().astype(dt)
            for idx, v in patch.items():
                r[idx] = v
            r = np.ascontiguousarray(r)
            keep.append(r)
            return r.ctypes.data
        st = _lib.AcState(
            n=n, lat=arr(lat), lon=arr(lon), alt=arr(alt), tas=arr(tas), hdg=arr(hdg), vs=arr(vs), selspd=arr(selspd),
            selalt=arr(selalt), selvs=arr(selvs), ap_trk=arr(ap_trk), cas=arr(cas), ax=arr(ax), curlegdir=arr(curlegdir),
            swlnav=arr(None if lnav is None else np.asarray(lnav, dtype=bool), np.uint8),
            iactwp=arr(iactwp, np.int32), env_f64=record("env_f64", env_f64, np.float64),
            env_f32=record("env_f32", env_f32, np.float32), env_i32=record("env_i32", env_i32, np.int32))
        if poly is not None:
            pl = np.zeros(self.layout.poly_f64)
            pl[:len(poly)] = poly
            keep.append(pl)
            st.poly = pl.ctypes.data
        _lib.check(self._lib.bsg_load_state(self._h, int(e), C.byref(st), self._stream()))

    def render(self, env_index=0):
        """rgb_array frame (height, width, 3) uint8 of ONE env, drawn like the reference's ``_render_frame`` of that env type
        (render.py builds the draw calls from a snapshot of the env, ``bsg_render`` paints them on the device)."""
        from . import render as _render
        return _render.render_env(self, env_index)

    def close(self, **kwargs):
        if not self.closed and self._h:
            self._lib.bsg_destroy(self._h)
            self._h = C.c_void_p(0)
        self.closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
