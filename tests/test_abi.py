"""The C-ABI library loads on a CPU-only box, exports every symbol include/bsg.h declares, answers the
pure-host queries, and fails loudly (no CPU fallback) when asked to compute without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(ROOT, "include", "bsg.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(bsg_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported(lib):
    from bluesky_gym_sasha_b200 import _lib
    names = _header_functions()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/bsg.h but not exported"
    assert set(_lib.SYMBOLS) == set(names)
    assert lib.bsg_abi_version() == 6
    for which, st in enumerate((_lib.Config, _lib.Layout, _lib.TensorTable, _lib.Wind, _lib.Perf, _lib.AcState, _lib.CdLists, _lib.TrafConfig,
                                _lib.TrafTensors)):
        assert lib.bsg_abi_struct_size(which) == C.sizeof(st), st.__name__          # the ctypes mirror of include/bsg.h
    assert lib.bsg_abi_struct_size(99) == -1


def test_cd_record_constants_match_header():
    """_lib's CD record constants (tile width, field indices) are the BSG_CD_TILE / BSG_CD_REC_* enum of include/bsg.h."""
    from bluesky_gym_sasha_b200 import _lib
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "bsg.h")).read(), flags=re.S)
    enum = dict(re.findall(r"\bBSG_(CD_TILE|CD_REC_[A-Z]+)\s*=\s*(\d+)", src))
    assert sorted(enum) == sorted(["CD_TILE", "CD_REC_FIELDS"] + ["CD_REC_" + f for f in ("X", "Y", "CH", "SH", "U", "V", "ALT", "VS")])
    for name, value in enum.items():
        assert getattr(_lib, name) == int(value), name


def test_layout_queries(lib):
    from bluesky_gym_sasha_b200 import _lib, spec
    want = {"DescentEnv-v0": (1, 4, 1, 30, 1.0), "HorizontalCREnv-v0": (8, 28, 1, 10, 5.0),
            "SectorCREnv-v0": (32, 31, 2, 5, 1.0), "MergeEnv-v0": (32, 40, 2, 10, 5.0),
            "PlanWaypointEnv-v0": (1, 20, 1, 10, 1.0), "VerticalCREnv-v0": (8, 39, 1, 30, 1.0),
            "StaticObstacleEnv-v0": (16, 43, 2, 10, 1.0)}
    for env_id, s in spec.SPECS.items():
        lay = _lib.query_layout(_lib.Config(env_type=s.env_type, num_envs=3, n_intruders=5))
        assert (lay.slots, lay.obs_dim, lay.act_dim, lay.n_sub, lay.simdt) == want[env_id]
        assert s.obs_layout(5)[1] == lay.obs_dim and lay.info_dim >= len(s.info_keys)
    lay = _lib.query_layout(_lib.Config(env_type=_lib.ENV_HORIZONTAL_CR, num_envs=1, n_intruders=20))
    assert lay.slots == 32 and lay.obs_dim == 103
    with pytest.raises(_lib.BsgError):
        _lib.query_layout(_lib.Config(env_type=_lib.ENV_HORIZONTAL_CR, num_envs=1, n_intruders=40))
    with pytest.raises(_lib.BsgError):
        _lib.query_layout(_lib.Config(env_type=17, num_envs=1))
    assert lib.bsg_cd_padded(0) == 0 and lib.bsg_cd_padded(1) == 256 and lib.bsg_cd_padded(100000) == 100096


def test_no_cpu_fallback(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from bluesky_gym_sasha_b200 import _lib
    h = C.c_void_p(0)
    cfg = _lib.Config(env_type=_lib.ENV_DESCENT, num_envs=1)
    rc = lib.bsg_create(C.byref(cfg), C.byref(h))
    assert rc == _lib.BSG_ECUDA and b"no CPU fallback" in lib.bsg_last_error()
    out = C.c_double(0)
    assert lib.bsg_probe_fp32(0, C.byref(out)) == _lib.BSG_ECUDA
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv
    with pytest.raises(_lib.BsgError):
        BlueSkyVectorEnv("HorizontalCREnv-v0", 4)
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    with pytest.raises(_lib.BsgError):
        StateBasedCD()


def test_argument_validation(lib):
    from bluesky_gym_sasha_b200 import _lib
    assert lib.bsg_cd_detect(None, 10, 5, 10, 0.0, 0.0, 0.0, 0, None, None, None, None, None, None) == _lib.BSG_EINVAL
    assert b"row range" in lib.bsg_last_error()
    assert lib.bsg_cd_pack(None, None, None, None, None, None, 4, 0.0, 0.0, None, None) == _lib.BSG_EINVAL
    assert lib.bsg_reset(None, None, None) == _lib.BSG_EINVAL


def test_product_does_not_import_oracle():
    """The product path must never route through the oracle (or any CPU fallback)."""
    pkg = os.path.join(ROOT, "bluesky_gym_sasha_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f
    for f in ("bluesky_gym/__init__.py", "bluesky_gym/envs/__init__.py"):
        assert "oracle" not in open(os.path.join(ROOT, f)).read()


def test_host_thread_copy(lib):
    """bsg_host_copy (the pooled memcpy behind bsg_step_host_copy) is byte-exact for ragged sizes and offsets."""
    import ctypes as C
    import numpy as np
    rng = np.random.default_rng(0)
    src = rng.integers(0, 256, 5_000_003, dtype=np.uint8)
    for n, off in [(0, 0), (1, 3), (4096, 1), (262_144, 0), (262_145, 7), (1_687_552, 0), (4_999_990, 13)]:
        dst = np.zeros(n + 64, dtype=np.uint8)
        assert lib.bsg_host_copy(C.c_void_p(dst.ctypes.data + 32), C.c_void_p(src.ctypes.data + off), n) == 0
        assert np.array_equal(dst[32:32 + n], src[off:off + n])
        assert not dst[:32].any() and not dst[32 + n:].any()
    for _ in range(50):                                   # repeated calls reuse the sleeping workers
        dst = np.empty(1_687_552, dtype=np.uint8)
        lib.bsg_host_copy(C.c_void_p(dst.ctypes.data), C.c_void_p(src.ctypes.data), dst.nbytes)
        assert np.array_equal(dst, src[:dst.nbytes])


def test_host_thread_widen(lib):
    """bsg_host_widen (float32 -> float64 with the host threads) equals numpy's astype for ragged sizes."""
    import ctypes as C
    import numpy as np
    rng = np.random.default_rng(1)
    src = rng.standard_normal(1_300_003).astype(np.float32)
    for n in (0, 1, 7, 16_384, 65_537, 421_888, 1_300_003):
        dst = np.full(n + 4, -7.0)
        assert lib.bsg_host_widen(C.c_void_p(dst.ctypes.data + 16), C.c_void_p(src.ctypes.data), n) == 0
        assert np.array_equal(dst[2:2 + n], src[:n].astype(np.float64)) and (dst[:2] == -7.0).all() and (dst[2 + n:] == -7.0).all()


def _build_c_host(tmp_path):
    import shutil
    import subprocess
    if shutil.which("gcc") is None or not os.path.isdir("/usr/local/cuda/include"):
        pytest.skip("needs gcc and the CUDA runtime headers")
    from bluesky_gym_sasha_b200 import build
    build.build()
    pkg = os.path.join(ROOT, "bluesky_gym_sasha_b200")
    exe = str(tmp_path / "c_abi_detect")
    cmd = ["gcc", os.path.join(ROOT, "examples", "c_abi_detect.c"), "-I" + os.path.join(ROOT, "include"), "-I/usr/local/cuda/include",
           "-L" + pkg, "-lbsg_b200", "-L/usr/local/cuda/lib64", "-lcudart", "-lm", "-Wl,-rpath," + pkg, "-Wall", "-Werror", "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_c_host_links_against_the_abi(tmp_path):
    """include/bsg.h is plain C and the library links into a C program with gcc alone (examples/c_abi_detect.c): no C++, no
    torch, no Python in the boundary.  Without a device the program reports that and exits 1."""
    import subprocess
    exe = _build_c_host(tmp_path)
    import torch
    if not torch.cuda.is_available():
        r = subprocess.run([exe, "100"], capture_output=True, text=True)
        assert r.returncode == 1 and "no CUDA device" in r.stderr


@pytest.mark.gpu
def test_c_host_runs_the_detection(cuda, tmp_path):
    """The same program on a GPU: packs 20 000 aircraft in the device-chosen order, runs the culled + symmetric and the
    all-pairs detection through the C ABI and finds the same conflicts with both."""
    import subprocess
    exe = _build_c_host(tmp_path)
    r = subprocess.run([exe, "20000"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.strip().endswith("ok") and "conflicts" in r.stdout
    print(r.stdout.strip())
