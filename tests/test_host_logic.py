"""Host-side logic that runs without a GPU: registration ids and caps, spaces, the gymnasium shim,
perf-table sync between oracle and product, row sharding (world_size-2 gloo)."""
import os
import socket

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_register_envs_ids_and_caps():
    """bluesky_gym/__init__.py:7-46: seven ids with their max_episode_steps."""
    import bluesky_gym
    from bluesky_gym_sasha_b200.gym_compat import registry
    bluesky_gym.register_envs()
    want = {"DescentEnv-v0": 300, "PlanWaypointEnv-v0": 300, "HorizontalCREnv-v0": 300, "VerticalCREnv-v0": 300,
            "SectorCREnv-v0": 200, "StaticObstacleEnv-v0": 100, "MergeEnv-v0": 50}
    for k, v in want.items():
        assert k in registry and registry[k].max_episode_steps == v


def test_all_reference_ids_are_accelerated():
    from bluesky_gym_sasha_b200.spec import NOT_ACCELERATED, SPECS
    assert NOT_ACCELERATED == () and len(SPECS) == 7


def test_every_registered_entry_point_resolves():
    """Every id of bluesky_gym/__init__.py:6-46 resolves to a class: through the registered entry point, through
    ``import bluesky_gym.envs`` (scripts/multi_processing_example.py:17) and through the reference's own module paths
    (``bluesky_gym.envs.<name>_env:<Class>``)."""
    import importlib

    import bluesky_gym
    import bluesky_gym.envs
    from bluesky_gym_sasha_b200 import envs as penvs
    from bluesky_gym_sasha_b200.gym_compat import Env, registry
    from bluesky_gym_sasha_b200.spec import SPECS
    bluesky_gym.register_envs()
    ref_paths = {"DescentEnv-v0": "bluesky_gym.envs.descent_env:DescentEnv",
                 "PlanWaypointEnv-v0": "bluesky_gym.envs.plan_waypoint_env:PlanWaypointEnv",
                 "HorizontalCREnv-v0": "bluesky_gym.envs.horizontal_cr_env:HorizontalCREnv",
                 "VerticalCREnv-v0": "bluesky_gym.envs.vertical_cr_env:VerticalCREnv",
                 "SectorCREnv-v0": "bluesky_gym.envs.sector_cr_env:SectorCREnv",
                 "StaticObstacleEnv-v0": "bluesky_gym.envs.static_obstacle_env:StaticObstacleEnv",
                 "MergeEnv-v0": "bluesky_gym.envs.merge_env:MergeEnv"}
    assert set(ref_paths) == set(SPECS)
    for env_id, spec in SPECS.items():
        ep = registry[env_id].entry_point
        for path in (ep, ref_paths[env_id]):
            mod, cls = path.split(":")
            k = getattr(importlib.import_module(mod), cls)
            assert issubclass(k, Env) and k.ENV_ID == env_id, (env_id, path)
        assert getattr(bluesky_gym.envs, spec.entry_point.split(":")[1]).ENV_ID == env_id
    for name in penvs.__all__:
        assert hasattr(penvs, name), name
    from bluesky_gym.utils import logger          # scripts/multi_processing_example.py:19
    assert hasattr(logger, "CSVLoggerCallback")


def test_csv_logger_callback_rows(tmp_path):
    """bluesky_gym/utils/logger.py:15-35: header from infos[0]'s keys, one row per finished episode of env 0."""
    import csv

    from bluesky_gym.utils.logger import CSVLoggerCallback
    cb = CSVLoggerCallback(str(tmp_path), "log.csv")
    for t in range(1, 7):
        cb.num_timesteps = t
        cb.locals = {"infos": [{"total_reward": -float(t), "total_intrusions": t % 2}, {"total_reward": 9.0}],
                     "dones": [t % 3 == 0, True]}
        assert cb._on_step() is True
    rows = list(csv.reader(open(tmp_path / "log.csv")))
    assert rows[0] == ["timesteps", "episodes", "total_reward", "total_intrusions"]
    assert rows[1:] == [["3", "1", "-3.0", "1"], ["6", "2", "-6.0", "0"]]


def test_obs_layout_matches_reference_declarations():
    from bluesky_gym_sasha_b200.spec import SPECS
    lay, dim = SPECS["HorizontalCREnv-v0"].obs_layout(5)
    assert dim == 28 and list(lay)[:2] == ["intruder_distance", "cos_difference_pos"] and lay["cos_drift"][:2] == (26, 1)
    lay, dim = SPECS["SectorCREnv-v0"].obs_layout()
    assert dim == 31 and lay["distances"][:2] == (27, 4) and lay["airspeed"][2:] == (-1, 1)
    lay, dim = SPECS["MergeEnv-v0"].obs_layout()
    assert dim == 40 and lay["faf_reached"][2:] == (0, 1)
    assert SPECS["MergeEnv-v0"].info_keys == ("total_reward", "faf_reach", "average_drift", "total_intrusions")


def test_gym_shim_box_default_shape_and_time_limit():
    from bluesky_gym_sasha_b200 import gym_compat as g
    if g.HAVE_GYMNASIUM:
        pytest.skip("real gymnasium installed")
    b = g.spaces.Box(-np.inf, np.inf, dtype=np.float64)         # descent_env.py:55-58 -> shape (1,)
    assert b.shape == (1,) and b.dtype == np.float64 and b.contains(np.zeros(1))
    d = g.spaces.Dict({"a": b, "b": g.spaces.Box(-1, 1, shape=(3,), dtype=np.float64)})
    bd = g.batch_space(d, 5)
    assert bd["b"].shape == (5, 3) and d.contains(d.sample())

    class Dummy(g.Env):
        def reset(self, **kw):
            return 0, {}

        def step(self, a):
            return 0, 0.0, False, False, {}
    e = g.TimeLimit(Dummy(), 3)
    e.reset()
    assert [e.step(0)[3] for _ in range(3)] == [False, False, True]


def test_perf_table_in_sync_with_oracle():
    from bluesky_gym_sasha_b200.spec import A320_PERF
    from oracle.perf import A320
    assert A320_PERF == A320.as_dict()


def test_shard_rows_partition():
    from bluesky_gym_sasha_b200.cd import shard_rows
    n, w = 4096, 8
    cover = []
    for r in range(w):
        r0, nr = shard_rows(n, w, r)
        cover += list(range(r0, r0 + nr))
    assert cover == list(range(n))


def _gloo_worker(rank, world, port, q):
    """Row-sharded CD on CPU ranks: all-gather the aircraft block, evaluate own rows with the oracle."""
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from bluesky_gym_sasha_b200.cd import shard_rows
    from oracle import cbind
    from tests.common import synth_airspace
    n = 512
    full = np.stack(synth_airspace(n, box_deg=3.0, seed=9))
    r0, nr = shard_rows(n, world, rank)
    local = torch.from_numpy(np.ascontiguousarray(full[:, r0:r0 + nr]))
    gathered = [torch.empty_like(local) for _ in range(world)]
    dist.all_gather(gathered, local)
    allst = torch.cat(gathered, dim=1).numpy()
    assert np.array_equal(allst, full)
    out = cbind.detect_rows(*allst, 9260.0, 304.8, 300.0, row0=r0, nrows=nr, pair_cap=100000, nthreads=1)
    q.put((rank, out["nconf_row"].tolist(), out["confpairs"].tolist()))
    dist.destroy_process_group()


def test_row_sharding_world2_gloo():
    """SURVEY.md section 8e on CPU ranks: union of per-rank results == single-rank detection."""
    import torch.multiprocessing as mp
    from oracle import cbind
    from tests.common import synth_airspace
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted(q.get(timeout=120) for _ in range(2))
    [p.join(timeout=60) for p in procs]
    full = cbind.detect_rows(*synth_airspace(512, box_deg=3.0, seed=9), 9260.0, 304.8, 300.0, pair_cap=100000)
    assert res[0][1] + res[1][1] == full["nconf_row"].tolist()
    assert res[0][2] + res[1][2] == full["confpairs"].tolist() and len(full["confpairs"]) > 0


def test_sb3_lazy_infos_behave_like_a_list_of_dicts():
    """BlueSkySB3VecEnv's infos: built per env on first access, same content as an eager list of dicts."""
    import numpy as np
    from bluesky_gym_sasha_b200.sb3_vec_env import _LazyInfos
    E = 6
    infos = {"total_reward": np.linspace(-1, 1, E), "total_intrusions": np.arange(E), "_final_obs": np.ones(E, bool),
             "final_obs": {"a": np.arange(2 * E, dtype=np.float32).reshape(E, 2)}}
    term = np.array([1, 0, 0, 0, 0, 1], bool)
    trunc = np.array([0, 1, 0, 0, 0, 1], bool)
    lazy = _LazyInfos(infos, term, trunc, term | trunc)
    assert isinstance(lazy, list) and len(lazy) == E
    assert lazy[0]["total_reward"] == -1.0 and isinstance(lazy[3]["total_intrusions"], int)
    assert lazy[1]["TimeLimit.truncated"] is True and lazy[5]["TimeLimit.truncated"] is False      # terminated wins
    assert "terminal_observation" in lazy[0] and "terminal_observation" not in lazy[2]
    assert np.array_equal(lazy[1]["terminal_observation"]["a"], [2.0, 3.0])
    assert [d["total_intrusions"] for d in lazy] == list(range(E)) and lazy[-1]["total_intrusions"] == E - 1
    assert len(lazy[1:4]) == 3
    lazy[2] = {"replaced": 1}                    # wrappers may overwrite entries
    assert lazy[2] == {"replaced": 1}


def test_cd_records_allocator_shape_and_inert_padding(lib):
    """cd.cd_records: bsg_cd_padded(n) records as [tiles, 8, 256] float32 (at least one tile); inert=True fills every
    record with the padding record of bsg_cd_pack: x, y, sh, u, v, vs = 0, ch = 1, alt = 3e9."""
    import torch
    from bluesky_gym_sasha_b200.cd import cd_records
    for n, tiles in ((0, 1), (1, 1), (256, 1), (257, 2), (100_000, 391)):
        rec = cd_records(n, "cpu")
        assert rec.shape == (tiles, 8, 256) and rec.dtype == torch.float32 and rec.device.type == "cpu"
        inert = cd_records(n, "cpu", inert=True)
        assert inert.shape == (tiles, 8, 256) and inert.dtype == torch.float32
        want = np.zeros(8, np.float32)
        want[2], want[6] = 1.0, 3.0e9
        assert np.array_equal(inert.numpy(), np.broadcast_to(want[None, :, None], (tiles, 8, 256)))
