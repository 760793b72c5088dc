"""The quadtree DEVICE code (structure-plp-slam_b200/csrc/orb_quadtree.cuh) executed on the CPU: tests/cta_emu compiles the
same kernel text for the host and this test runs one (level, frame) job through each instance orb.cu launches, on random
and real FAST candidates, comparing the keypoints with the oracle's distribute_keypoints_via_tree.  Candidate counts just
below and just above each instance's shared-memory window exercise both the shared-memory and the global-scratch path.
The GPU parity runs are tests/test_orb_gpu.py and tests/test_golden.py."""
import ctypes as C
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

import oracle_api
import synth

ROOT = Path(__file__).resolve().parent.parent
_P = C.c_void_p
CELL_CAP = 1024
BORDER = 19
# (threads, node capacity, candidate window) of QtLarge, QtWide and QtNarrow in csrc/orb.cu
INSTANCES = {"large": (0, 2048, 8192), "wide": (1, 1024, 1664), "narrow": (2, 512, 2048)}


@pytest.fixture(scope="module")
def qt_emu(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    so = tmp_path_factory.mktemp("emu") / "libquadtree_emu.so"
    cmd = ["g++", "-O1", "-std=c++17", "-pthread", "-shared", "-fPIC", "-ffp-contract=off",
           f"-I{ROOT / 'structure-plp-slam_b200' / 'csrc'}", f"-I{ROOT / 'tests' / 'cta_emu'}",
           str(ROOT / "tests" / "cta_emu" / "quadtree_emu.cc"), "-o", str(so)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[:3000]
    return C.CDLL(str(so))


def _cells(rng, n):
    """Split n candidates (in gather order) into cell lists of random size, empty cells included."""
    sizes = []
    left = n
    while left > 0:
        k = 0 if rng.random() < 0.15 else int(rng.integers(1, min(left, CELL_CAP) + 1))
        sizes.append(min(k, left))
        left -= sizes[-1]
    sizes.append(0)
    return np.array(sizes, np.int32)


def _check(qt_emu, orc, instance, xs, ys, resp, w, h, budget, seed=0):
    """w, h: level size; xs, ys relative to the 19-px border, in gather order."""
    inst, nodes, _ = INSTANCES[instance]
    n = len(xs)
    cnt = _cells(np.random.default_rng(seed), n)
    assert len(cnt) <= nodes
    buf = np.zeros((len(cnt), CELL_CAP), np.uint32)
    packed = (xs.astype(np.uint32) | (ys.astype(np.uint32) << 11) | (resp.astype(np.uint32) << 21))
    off = 0
    for c, k in enumerate(cnt):
        buf[c, :k] = packed[off: off + k]
        off += k
    ox, oy = np.zeros(nodes, np.int16), np.zeros(nodes, np.int16)
    orsp, st = np.zeros(nodes, np.int32), C.c_int(0)
    got = qt_emu.emu_quadtree(C.c_int(inst), C.c_int(w), C.c_int(h), C.c_int(budget), C.c_int(nodes), C.c_int(len(cnt)),
                              cnt.ctypes.data_as(_P), buf.ctypes.data_as(_P), ox.ctypes.data_as(_P),
                              oy.ctypes.data_as(_P), orsp.ctypes.data_as(_P), C.byref(st))
    cands = np.zeros(n, oracle_api.KP_DTYPE)
    cands["x"], cands["y"], cands["response"] = xs, ys, resp
    ref = orc.orb_distribute(oracle_api.orb_params(), cands, BORDER, w - BORDER, BORDER, h - BORDER, budget)
    assert st.value == 0
    assert got == len(ref)
    assert np.array_equal(ox[:got] - BORDER, ref["x"].astype(np.int16))
    assert np.array_equal(oy[:got] - BORDER, ref["y"].astype(np.int16))
    assert np.array_equal(orsp[:got], ref["response"].astype(np.int32))


def _random(seed, n, w, h):
    rng = np.random.default_rng(seed)
    xs = rng.integers(0, w - 2 * BORDER, n)
    ys = rng.integers(0, h - 2 * BORDER, n)
    if seed % 3 == 0:  # heavy duplication -> many equal-count leaves, exercises the tie-break
        xs, ys = xs // 16 * 16, ys // 16 * 16
    return xs.astype(np.float32), ys.astype(np.float32), rng.integers(7, 255, n).astype(np.float32)


def _budgets(instance, n):
    """Budgets 5 / 60 / 217 / 1000 where the job fits the instance's node capacity: a node holds at least one
    candidate, so n <= nodes is enough, else 4 * budget + 8 <= nodes."""
    nodes = INSTANCES[instance][1]
    return [b for b in (5, 60, 217, 1000) if n <= nodes or 4 * b + 8 <= nodes]


@pytest.mark.parametrize("instance", list(INSTANCES))
@pytest.mark.parametrize("seed", range(3))
def test_random_candidates(qt_emu, orc, instance, seed):
    w, h = [(640, 480), (533, 400), (300, 700)][seed]
    n = [1300, 400, 900][seed]
    xs, ys, resp = _random(seed, n, w, h)
    for budget in _budgets(instance, n):
        _check(qt_emu, orc, instance, xs, ys, resp, w, h, budget, seed)


@pytest.mark.parametrize("instance", list(INSTANCES))
def test_window_edges(qt_emu, orc, instance):
    """Just below the shared-memory window (shared path) and just above it (global-scratch path)."""
    window = INSTANCES[instance][2]
    for n in (window, window + 1):
        xs, ys, resp = _random(n, n, 1280, 720)
        budget = max(b for b in _budgets(instance, n))
        _check(qt_emu, orc, instance, xs, ys, resp, 1280, 720, budget, n)


def test_real_fast_candidates(qt_emu, orc):
    """Every level of a real frame on each instance whose node capacity the default budgets fit."""
    img = synth.make_texture(99)
    p = oracle_api.orb_params()
    r = orc.orb_extract(p, img, debug=True)
    w, h = orc.orb_level_sizes(p, *img.shape)
    t = orc.orb_tables(p)
    off = 0
    for lvl in range(8):
        c = r["cands"][off: off + r["cands_per_level"][lvl]]
        off += r["cands_per_level"][lvl]
        budget = int(t["num_keypts_per_level"][lvl])
        for instance, (_, nodes, _) in INSTANCES.items():
            if 4 * budget + 8 <= nodes:
                _check(qt_emu, orc, instance, c["x"].copy(), c["y"].copy(), c["response"].copy(), int(w[lvl]),
                       int(h[lvl]), budget, lvl)
