"""Pins oracle/ref_port.py against the committed golden vectors that tests/golden/make_golden.py wrote by running
the real reference: its pipeline outputs (pipe_*, tri_*, ba_*) and, in reference_calls.npz, what its functions
returned for the inputs of the *_live_reference tests below.  CPU only."""
import numpy as np
import pytest

from oracle.ref_port import RefPort
from tests.util import load_golden, poses_from, obs_from, as3

PIPE_CASES = ["pipe_c2_m1", "pipe_c4_m4", "pipe_c8_m16"]


def _blobs(port, frames, b, c):
    pts = port.find_dot(as3(frames[b, c]))
    return [p for p in pts if p[0] is not None]


@pytest.mark.parametrize("name", PIPE_CASES + ["blobs_irregular"])
def test_find_dot_matches_golden(name):
    z = load_golden(name, n=12 if name == "pipe_c8_m16" else None)
    frames = z["frames"]
    B, C = frames.shape[:2]
    port = RefPort([np.eye(3)] * C)
    step = max(1, B // 12)
    for b in range(0, B, step):
        for c in range(C):
            pts = _blobs(port, frames, b, c)
            n = int(z["blob_n"][b, c])
            assert len(pts) == n
            assert np.array_equal(np.array(pts, dtype=np.int32).reshape(n, 2), z["blob_xy"][b, c, :n])


@pytest.mark.parametrize("name", PIPE_CASES)
def test_match_and_triangulate_matches_golden(name):
    z = load_golden(name, frames=False)
    C = int(z["C"])
    port = RefPort([z["K"]] * C)
    poses = poses_from(z)
    B = z["blob_n"].shape[0]
    step = max(1, B // 8)
    for b in range(0, B, step):
        pts = [[list(map(int, z["blob_xy"][b, c, i])) for i in range(z["blob_n"][b, c])] for c in range(C)]
        err, obj, _ = port.match_and_triangulate(pts, poses)
        k = int(z["nroot"][b])
        assert len(err) == k
        # same third-party routines, same order of operations -> bit-identical
        assert np.array_equal(np.asarray(obj, dtype=np.float64).reshape(k, 3), z["obj"][b, :k])
        assert np.array_equal(err, z["err"][b, :k])


@pytest.mark.parametrize("name", ["tri_c4", "tri_c8", "tri_c16"])
def test_triangulate_and_error_match_golden(name):
    z = load_golden(name)
    C = z["R"].shape[0]
    port = RefPort([z["K"]] * C)
    obs = obs_from(z)
    poses = poses_from(z)
    X = port.triangulate_many(obs, poses)
    assert np.array_equal(np.asarray(X, dtype=np.float64), z["X"])
    assert np.array_equal(port.reprojection_errors(obs, X, poses), z["err"])


def test_triangulate_needs_two_views():
    port = RefPort([np.eye(3)] * 2)
    poses = [{"R": np.eye(3), "t": np.zeros(3)}, {"R": np.eye(3), "t": np.array([-1.0, 0, 0])}]
    assert port.triangulate_one([[10, 10], [None, None]], poses) == [None, None, None]
    assert port.reprojection_error([[10, 10], [None, None]], np.zeros(3), poses) is None
    assert port.find_dot(np.zeros((480, 640, 3), np.uint8)) == [[None, None]]


def _reference_calls():
    return load_golden("reference_calls")


def test_port_equals_live_reference(synth):
    """S1-S3 of the port against what the reference returned for the same three frame-sets."""
    z = _reference_calls()
    C, M = 4, 6
    frames, truth, poses, K = synth.make_frame_pool(C, M, 3, seed=42)
    port = RefPort([K] * C)
    for b in range(3):
        ref_pts = [[list(map(int, p)) for p in z["pipe_blob_xy"][b, c, :z["pipe_blob_n"][b, c]]] or [[None, None]] for c in range(C)]
        my_pts = [port.find_dot(as3(frames[b, c])) for c in range(C)]
        assert ref_pts == my_pts
        e2, o2, _ = port.match_and_triangulate(my_pts, poses)
        k = int(z["pipe_nroot"][b])
        assert np.array_equal(z["pipe_err"][b, :k], e2)
        assert np.array_equal(z["pipe_obj"][b, :k], np.asarray(o2, dtype=np.float64).reshape(-1, 3))


def test_ba_residuals_equal_live_reference(synth):
    C = 3
    z = _reference_calls()
    obs, poses, K, _ = synth.make_tracks(C, 12, seed=2)
    start = synth.perturb_poses(poses, seed=3)
    port = RefPort([K] * C)
    r_ref = z["ba_r"]
    x0 = port.poses_to_params(start)
    r = port.ba_residuals(x0, obs)
    # poses -> rotvec -> matrix round trip in the port: equal to float32 resolution
    assert r.dtype == np.float32 and r.shape == r_ref.shape
    assert np.allclose(r, r_ref, rtol=1e-5, atol=1e-6)


def test_locate_objects_equals_live_reference(synth):
    z = _reference_calls()
    total = 0
    for seed in range(30):
        pts, errs = synth.make_drone_points(1 + seed % 3, seed % 5, seed=seed)
        mine = RefPort.locate_objects(pts.copy(), errs.copy())
        assert len(mine) == z["loc_counts"][seed]
        for i, b in enumerate(mine, start=total):
            assert np.array_equal(z["loc_pos"][i], b["pos"]) and z["loc_heading"][i] == b["heading"]
            assert z["loc_error"][i] == b["error"] and z["loc_drone"][i] == b["droneIndex"]
        total += len(mine)
    assert total >= 30


def test_preprocess_equals_live_reference():
    """RefPort.preprocess restates helpers.py:70-82; the reference only exposes that chain inside _camera_read
    (which needs camera hardware), so its pieces are compared: make_square against the digest of the reference's
    output, the cv2 calls by construction (same functions, same arguments)."""
    import hashlib
    z = _reference_calls()
    rng = np.random.default_rng(0)
    frame = rng.integers(0, 256, size=(240, 320, 3), dtype=np.uint8)
    sq = RefPort.make_square(frame)
    assert sq.dtype == np.uint8 and sq.shape == tuple(z["square_shape"])
    assert hashlib.sha256(np.ascontiguousarray(sq).tobytes()).hexdigest() == str(z["square_sha256"])


def test_calibrate_init_equals_live_reference(synth):
    """index.py:229-270: the camera chain the reference's calculate_camera_pose hands to bundle_adjustment (cv2 RNG
    seed 0) against the port's (same seed)."""
    C = 3
    z = _reference_calls()
    obs, poses, K, _ = synth.make_tracks(C, 40, seed=8, missing_frac=0.15)
    mine = RefPort([K] * C).calibrate_init(obs.tolist(), rng_seed=0)
    assert len(mine) == len(z["calib_R"]) == C
    for c, a in enumerate(mine):
        assert np.array_equal(np.asarray(a["R"], dtype=np.float64), z["calib_R"][c])
        assert np.array_equal(np.asarray(a["t"], dtype=np.float64).ravel(), z["calib_t"][c])


def _reference_shaped_modules(z):
    """Stand-ins with the layout install_into relies on: ``helpers`` holds the hot-path names the reference's helpers
    module holds and a ``Cameras`` singleton wrapper whose instance has ``camera_params``; ``index`` holds the names
    the reference's index.py imported from helpers by value."""
    import types

    class Cameras:
        def __init__(self):
            K = [[600.0, 0.0, 320.0], [0.0, 600.0, 240.0], [0.0, 0.0, 1.0]]
            self.camera_params = [{"intrinsic_matrix": np.array(K), "distortion_coef": np.zeros(5), "rotation": 0}
                                  for _ in range(4)]

        def _find_dot(self, img):
            return img, [[None, None]]

    class Singleton:                                   # instance() creates the decorated class once
        def __init__(self, decorated):
            self._decorated = decorated

        def instance(self):
            if not hasattr(self, "_instance"):
                self._instance = self._decorated()
            return self._instance

    def cpu_function(name):
        def f(*a):
            raise AssertionError(f"the CPU {name} was called")
        return f

    helpers = types.ModuleType("helpers")
    helpers.Cameras = Singleton(Cameras)
    for n in z["helpers_names"]:
        setattr(helpers, str(n), cpu_function(str(n)))
    index = types.ModuleType("index")
    for n in z["index_names"]:
        setattr(index, str(n), getattr(helpers, str(n)))
    return helpers, index


def test_install_into_rebinds_reference_shaped_modules():
    """INTEGRATION.md: install_into() must replace exactly the names the reference's callers resolve at call
    time -- the method on the class behind the Singleton wrapper, the module-level functions of helpers.py, and
    the names index.py imported from it by value (index.py:1)."""
    import importlib
    pkg = importlib.import_module("low-cost-mocap_b200")
    api = importlib.import_module("low-cost-mocap_b200.api")
    z = _reference_calls()
    assert sorted(map(str, z["helpers_names"])) == sorted(api.PATCHED_NAMES)
    assert set(map(str, z["index_names"])) == {"bundle_adjustment", "triangulate_points", "calculate_reprojection_errors"}
    helpers, index = _reference_shaped_modules(z)
    cams = helpers.Cameras.instance()
    saved = {n: getattr(helpers, n) for n in api.PATCHED_NAMES}
    saved_fd = type(cams)._find_dot
    s = pkg.install_into(helpers, index)
    assert len(s.intrinsics) == 4 and np.array_equal(s.intrinsics[0], np.asarray(cams.camera_params[0]["intrinsic_matrix"]))
    assert type(cams)._find_dot is not saved_fd
    assert cams._find_dot.__func__ is type(cams)._find_dot          # what _camera_read will call (helpers.py:87)
    for n in api.PATCHED_NAMES:
        assert getattr(helpers, n) is not saved[n] and getattr(helpers, n).__mocap_b200__
    for n in map(str, z["index_names"]):
        assert getattr(index, n) is getattr(helpers, n)
    # without a GPU the replacements fail loudly instead of falling back
    import torch
    if not torch.cuda.is_available():
        with pytest.raises(pkg.MocapError):
            helpers.triangulate_points([[[1, 2], [3, 4], [None, None], [None, None]]], [{"R": np.eye(3), "t": np.zeros(3)}] * 4)


@pytest.mark.parametrize("name", ["ba_c8", "ba_c16"])
def test_port_residuals_equal_the_reference_run_golden(name):
    """The larger S4 goldens (8 and 16 cameras) hold the start and the end state of a full bundle_adjustment run of
    the REAL reference (7 and 25 minutes of CPU time, tests/golden/make_golden.py ba8 / ba16).  The port's residual
    function must reproduce both residual vectors bit for bit."""
    z = load_golden(name)
    C = z["mask"].shape[1]
    port = RefPort([z["K"]] * C)
    obs = obs_from(z)
    for tag in ("start", "final"):
        poses = [{"R": z["R_" + tag][c], "t": z["t_" + tag][c]} for c in range(C)]
        r = port.ba_residuals(port.poses_to_params(poses), obs)
        ref = z["r0"] if tag == "start" else z["rf"]
        if tag == "start":
            assert np.array_equal(np.asarray(r, dtype=np.float32), ref)
        else:                                       # R_final went through one more rotation-vector round trip
            assert np.allclose(np.asarray(r, dtype=np.float32), ref, rtol=1e-5, atol=1e-6)
    assert float(z["costf"]) < float(z["cost0"])
