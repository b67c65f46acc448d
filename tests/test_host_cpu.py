"""CPU-side checks: the C-ABI library loads and exports every declared symbol, the header and
the ctypes table agree, the sharding exchange works over gloo with world_size 2, and the
HD geometry code (host build) reproduces the golden triangulations."""
import ctypes
import importlib
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from tests.util import ROOT, compile_shared, load_golden

pkg = importlib.import_module("low-cost-mocap_b200")
_lib = importlib.import_module("low-cost-mocap_b200._lib")
sharding = importlib.import_module("low-cost-mocap_b200.sharding")


@pytest.fixture(scope="module")
def built_lib():
    build = importlib.import_module("low-cost-mocap_b200.build")
    return build.build()


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "mocap_b200.h")).read()
    return sorted(set(re.findall(r"MOCAP_API[^;(]*?\b(mocap_\w+)\s*\(", text)))


def test_header_and_binding_agree():
    assert _declared_symbols() == sorted(_lib.SYMBOLS)


def test_library_exports_every_declared_symbol(built_lib):
    lib = ctypes.CDLL(built_lib)
    for name in _declared_symbols():
        assert hasattr(lib, name), name


def test_no_cpu_fallback(built_lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(pkg.MocapError):
        pkg.MocapContext(4)


def test_status_strings(built_lib):
    lib = _lib.load()
    assert lib.mocap_status_string(0) == b"ok"
    assert b"fallback" in lib.mocap_status_string(-2)


def test_shard_indices_cover_everything():
    for n in (0, 1, 7, 16, 1001):
        for world in (1, 2, 3, 8):
            seen = np.concatenate([sharding.shard_indices(n, r, world) for r in range(world)])
            assert sorted(seen.tolist()) == list(range(n))
            assert [sharding.shard_size(n, r, world) for r in range(world)] == \
                   [len(sharding.shard_indices(n, r, world)) for r in range(world)]


_WORKER = r"""
import importlib, os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
sharding = importlib.import_module("low-cost-mocap_b200.sharding")
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % sys.argv[2], rank=int(sys.argv[3]), world_size=2)
rank, world = dist.get_rank(), 2
for n_total in (9, 10):
    R = 4
    rng = np.random.default_rng(5)
    obj = torch.from_numpy(rng.normal(size=(n_total, R, 3)))
    err = torch.from_numpy(rng.uniform(size=(n_total, R)))
    n = torch.from_numpy(rng.integers(0, R + 1, size=(n_total,)).astype(np.int32))
    mine = torch.from_numpy(sharding.shard_indices(n_total, rank, world))
    rec = sharding.pack_tracks(obj[mine], err[mine], n[mine])
    full = sharding.all_gather_tracks(rec, n_total)
    o2, e2, n2 = sharding.unpack_tracks(full, R)
    assert torch.equal(o2, obj) and torch.equal(e2, err) and torch.equal(n2, n), "gather mismatch"
    # flat-buffer form: one collective over raw bytes, views on the result
    if n_total % world == 0:
        tb = sharding.TrackBuffer(n_total // world, R, "cpu")
        tb.views["obj"].copy_(obj[mine]); tb.views["err"].copy_(err[mine]); tb.views["n"].copy_(n[mine])
        per_rank = tb.all_gather()
        for f in range(n_total):
            v = per_rank[f % world]
            assert torch.equal(v["obj"][f // world], obj[f]) and v["n"][f // world] == n[f], "flat gather mismatch"
        # pipelined form (bench.py at N > 1): two buffers in turn, the collective only enqueued, waited for
        # before its buffer is written again
        bufs = [sharding.TrackBuffer(n_total // world, R, "cpu") for _ in range(2)]
        pending = [None, None]
        for step in range(5):
            k = step % 2
            if pending[k] is not None:
                views, work = pending[k]
                work.wait()
                assert torch.equal(views[1 - rank]["obj"][0], obj[1 - rank] + (step - 2)), "pipelined gather mismatch"
            bufs[k].views["obj"].copy_(obj[mine] + step)
            pending[k] = bufs[k].all_gather(async_op=True)
        for k in range(2):
            pending[k][1].wait()
dist.destroy_process_group()
print("OK", rank)
"""


def test_track_all_gather_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    port = str(29500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, port, str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT) for r in range(2)]
    outs = [p.communicate(timeout=180)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "OK" in o


@pytest.fixture(scope="module")
def geom_host():
    src = os.path.join(ROOT, "tests", "hostcheck", "geom_host.cpp")
    out = os.path.join(ROOT, "tests", "hostcheck", "libgeom_host.so")
    if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(src), os.path.getmtime(
            os.path.join(ROOT, "low-cost-mocap_b200", "csrc", "geom.cuh"))):
        compile_shared(["g++", "-O2", "-shared", "-fPIC", "-ffp-contract=off", "-o", out, src, "-lm"])
    return ctypes.CDLL(out)


@pytest.mark.parametrize("name", ["tri_c4", "tri_c8", "tri_c16"])
def test_geometry_code_matches_golden_on_host(geom_host, name):
    """The DLT / Jacobi / projection arithmetic the kernels run (geom.cuh), compiled for the
    host: 3D points within 1e-9 of the reference (contract: 1e-7), errors bit-identical."""
    z = load_golden(name)
    obs = np.ascontiguousarray(z["obs"]); mask = np.ascontiguousarray(z["mask"])
    R = np.ascontiguousarray(z["R"]); t = np.ascontiguousarray(z["t"]); K = z["K"]
    n, C, _ = obs.shape
    Pkc = np.zeros((C, C, 12))
    for k in range(C):
        for c in range(C):
            Pkc[k, c] = (K @ np.c_[R[c], t[c]]).ravel()
    K4 = np.tile(np.array([K[0, 0], K[1, 1], K[0, 2], K[1, 2]]), (C, 1))
    X = np.zeros((n, 3)); err = np.zeros(n); valid = np.zeros(n, np.uint8)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    geom_host.hc_triangulate(p(obs), p(mask), n, C, p(Pkc), p(R), p(t), p(K4), p(X), p(err), p(valid))
    assert valid.all()
    assert np.abs(X - z["X"]).max() < 1e-9
    assert np.array_equal(err, z["err"])


def test_header_is_plain_c_and_example_links(built_lib, tmp_path):
    """include/mocap_b200.h compiles as C (not C++) and the plain-C example links against the library."""
    exe = tmp_path / "pipeline_host"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "pipeline_host.c"), "-L", os.path.dirname(built_lib),
                           "-lmocap_b200", "-Wl,-rpath," + os.path.dirname(built_lib), "-o", str(exe)])
    import torch
    if not torch.cuda.is_available():
        r = subprocess.run([str(exe)], capture_output=True, text=True)
        assert r.returncode == 1 and "no usable CUDA device" in r.stderr      # fails loudly, no CPU fallback


@pytest.fixture(scope="module")
def ba_host():
    src = os.path.join(ROOT, "tests", "hostcheck", "ba_host.cpp")
    out = os.path.join(ROOT, "tests", "hostcheck", "libba_host.so")
    compile_shared(["g++", "-O2", "-shared", "-fPIC", "-ffp-contract=off", "-o", out, src, "-lm"])
    return ctypes.CDLL(out)


def test_trust_region_control_equals_scipy_on_a_smooth_problem(ba_host):
    """The optimiser control that drives S4 (csrc/trf_core.h) is a restatement of scipy's trf_no_bounds:
    on a smooth robust fit with a dead parameter (rank-deficient Jacobian, as in the reference) it must land
    on scipy's solution with scipy's evaluation count and termination status."""
    from scipy.optimize import least_squares
    rng = np.random.default_rng(0)
    t = np.linspace(0, 4, 40)
    y = 2.5 * np.exp(-1.3 * t) + 0.5 + rng.normal(0, 0.05, 40)
    y[::7] += 3.0                                    # outliers for the Cauchy loss
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    ba_host.hc_trf_expfit.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_double, ctypes.c_void_p]
    for ftol in (1e-2, 1e-8):
        x0 = np.array([1.0, 0.5, 0.0, 7.0])
        ref = least_squares(lambda x: x[0] * np.exp(-x[1] * t) + x[2] - y, x0, loss="cauchy", ftol=ftol)
        x = x0.copy(); rep = np.zeros(7)
        assert ba_host.hc_trf_expfit(p(t), p(y), 40, p(x), ftol, p(rep)) == 0
        assert np.allclose(x, ref.x, rtol=1e-6, atol=1e-8)
        assert abs(rep[1] - ref.cost) < 1e-9 * max(1.0, ref.cost)
        assert int(rep[4]) == ref.nfev and int(rep[5]) == ref.status


def test_ba_host_model_reaches_reference_quality(ba_host):
    """Same control on the S4 problem itself (CPU stand-in of the GPU evaluators, float64 differences): from the
    golden start it reduces the reference's robust cost by orders of magnitude within scipy's evaluation budget."""
    z = load_golden("ba_c4")
    C = 4
    obs = np.ascontiguousarray(z["obs"]); mask = np.ascontiguousarray(z["mask"])
    K = np.ascontiguousarray(np.tile(z["K"].reshape(1, 9), (C, 1)))
    R = np.ascontiguousarray(z["R_start"].copy()); t = np.ascontiguousarray(z["t_start"].copy())
    rep = np.zeros(7)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    ba_host.hc_bundle_adjust.argtypes = [ctypes.c_void_p] * 2 + [ctypes.c_int] * 2 + [ctypes.c_void_p] * 3 + [ctypes.c_double, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    assert ba_host.hc_bundle_adjust(p(obs), p(mask), obs.shape[0], C, p(K), p(R), p(t), 1e-2, 0, p(rep), 1) == 0
    assert abs(rep[0] - float(z["cost0"])) < 1e-3 * float(z["cost0"])
    assert rep[1] < 0.5 * rep[0] and int(rep[5]) in (2, 3, 4)


@pytest.fixture(scope="module")
def preproc_host():
    src = os.path.join(ROOT, "tests", "hostcheck", "preproc_host.cpp")
    out = os.path.join(ROOT, "tests", "hostcheck", "libpreproc_host.so")
    compile_shared(["g++", "-O2", "-shared", "-fPIC", "-fno-strict-aliasing", "-o", out, src])
    return ctypes.CDLL(out)


@pytest.mark.parametrize("S,in_h,rot,word_stores,n_threads", [(320, 240, 0, 1, 256), (320, 240, 2, 0, 256), (200, 150, 2, 1, 96),
                                                               (90, 70, 0, 0, 256), (70, 40, 0, 0, 64)])
def test_preprocess_tile_stages_equal_cv2_chain_on_host(preproc_host, S, in_h, rot, word_stores, n_threads):
    """The tile stages the preprocessing kernel is made of (csrc/preproc_tile.cuh: packed 4-way / 2-way dot
    products, mirrored apron, transposed Q8.8 plane) stepped through on the host equal helpers.py:70-82 as
    restated by the oracle port, bit for bit: noise frames (worst case for every rounding), a saturated
    frame, sizes that are not a multiple of the tile, both rotations, both store paths."""
    import cv2
    from oracle.ref_port import RefPort
    f0 = float(S)
    K = np.array([[f0, 0, S / 2.0], [0, f0, S / 2.0], [0, 0, 1]])
    dist = np.array([-1.26372388e-01, 2.62661497e-01, 1.21306197e-03, 2.24507008e-04, -2.48534118e-01]) * (1.0 if rot == 0 else 2.5)
    m1, m2 = cv2.initUndistortRectifyMap(K, dist, np.eye(3), K, (S, S), cv2.CV_16SC2)
    m1 = np.ascontiguousarray(m1); m2 = np.ascontiguousarray(m2)
    port = RefPort([K])
    rng = np.random.default_rng(S + rot)
    frames = np.stack([rng.integers(0, 256, size=(in_h, S, 3), dtype=np.uint8), np.full((in_h, S, 3), 255, dtype=np.uint8),
                       (rng.integers(0, 2, size=(in_h, S, 3)) * 255).astype(np.uint8)])
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p) if a is not None else None
    ws = word_stores if S % 4 == 0 else 0
    want = np.stack([port.preprocess(raw, 0, dist, rot) for raw in frames])
    want_gray = np.stack([cv2.cvtColor(w, cv2.COLOR_RGB2GRAY) for w in want])        # what _find_dot thresholds (helpers.py:144)
    # the kernel handles the frames of one camera in groups: 3 frames = a full group and a ragged one (for a
    # group size of 2); then each frame on its own
    for n in (3, 1):
        for first in range(0, 3, n):
            raw = np.ascontiguousarray(frames[first:first + n])
            got = np.full((n, S, S, 3), 7, dtype=np.uint8)
            gray = np.full((n, S, S), 7, dtype=np.uint8)
            preproc_host.hc_preprocess(p(raw), n, S, in_h, S, rot, p(m1), p(m2), p(got), p(gray), ws, n_threads)
            assert np.array_equal(got, want[first:first + n]), int((got != want[first:first + n]).sum())
            assert np.array_equal(gray, want_gray[first:first + n])
            only_gray = np.zeros((n, S, S), dtype=np.uint8)
            preproc_host.hc_preprocess(p(raw), n, S, in_h, S, rot, p(m1), p(m2), None, p(only_gray), ws, n_threads)
            assert np.array_equal(only_gray, gray)


def test_preprocess_tile_stages_fuzz_on_host(preproc_host):
    """Random small geometries through the host-stepped tile stages against the cv2 chain: sizes that are not a
    multiple of 4 or of the tile, the tallest frame make_square accepts (8 pad rows), strong distortion (map
    coordinates far outside the frame), both rotations, several thread counts."""
    import cv2
    from oracle.ref_port import RefPort
    rng = np.random.default_rng(2024)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p) if a is not None else None
    for case in range(24):
        S = int(rng.integers(34, 150))
        in_h = int(rng.integers(1, S - 15)) if case % 4 else S - 16
        rot = int(rng.choice([0, 2]))
        f0 = float(rng.uniform(0.5, 1.5) * S)
        K = np.array([[f0, 0, S / 2.0 + rng.uniform(-5, 5)], [0, f0 * rng.uniform(0.9, 1.1), S / 2.0 + rng.uniform(-5, 5)], [0, 0, 1]])
        dist = np.array([-0.126, 0.263, 0.0012, 0.0002, -0.249]) * rng.uniform(-3.0, 3.0)
        m1, m2 = cv2.initUndistortRectifyMap(K, dist, np.eye(3), K, (S, S), cv2.CV_16SC2)
        m1 = np.ascontiguousarray(m1); m2 = np.ascontiguousarray(m2)
        raw = rng.integers(0, 256, size=(2, in_h, S, 3), dtype=np.uint8)
        port = RefPort([K])
        want = np.stack([port.preprocess(r, 0, dist, rot) for r in raw])
        got = np.full((2, S, S, 3), 9, dtype=np.uint8)
        gray = np.full((2, S, S), 9, dtype=np.uint8)
        preproc_host.hc_preprocess(p(raw), 2, S, in_h, S, rot, p(m1), p(m2), p(got), p(gray), 1 if S % 4 == 0 else 0,
                                   int(rng.choice([32, 96, 256])))
        assert np.array_equal(got, want), (case, S, in_h, rot, int((got != want).sum()))
        assert np.array_equal(gray, np.stack([cv2.cvtColor(w, cv2.COLOR_RGB2GRAY) for w in want])), (case, S, in_h, rot)
