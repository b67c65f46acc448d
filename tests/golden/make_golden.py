"""Writes tests/golden/*.npz by running the REAL reference
(computer_code/api/helpers.py of a jyjblrd/Low-Cost-Mocap checkout, imported
unmodified through oracle/ref_harness.py) on seeded synthetic inputs:

    LOW_COST_MOCAP_DIR=<checkout> python tests/golden/make_golden.py

The vectors pin oracle/ref_port.py (tests/test_oracle_pinned.py) and the CUDA
path (tests/test_parity_gpu.py) on the GPU box, where the reference is absent.
"""
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.ref_harness import load_reference, NullSocket  # noqa: E402

synth = importlib.import_module("low-cost-mocap_b200.synth")
OUT = os.path.dirname(os.path.abspath(__file__))

MAXB = 64     # blobs per camera stored
MAXR = 128    # roots per frame-set stored


def pipeline_case(name, C, M, B, seed):
    helpers, cams = load_reference(C)
    clean, truth, poses, K = synth.make_frame_pool(C, M, B, seed=seed, noise_max=0)
    frames = synth.add_clutter(clean, 40, salt=seed)   # tests re-apply the same clutter
    blob_xy = np.full((B, C, MAXB, 2), -1, dtype=np.int32)
    blob_n = np.zeros((B, C), dtype=np.int32)
    obj = np.full((B, MAXR, 3), np.nan)
    err = np.full((B, MAXR), np.nan)
    nroot = np.zeros((B,), dtype=np.int32)
    for b in range(B):
        image_points = []
        for c in range(C):
            img3 = np.repeat(frames[b, c][:, :, None], 3, axis=2).copy()
            _, pts = cams._find_dot(img3)
            image_points.append(pts)
            real = [p for p in pts if p[0] is not None]
            blob_n[b, c] = len(real)
            for i, p in enumerate(real):
                blob_xy[b, c, i] = p
        e, o, _ = helpers.find_point_correspondance_and_object_points(
            [list(map(list, p)) for p in image_points], poses, [None] * C)
        k = len(e)
        nroot[b] = k
        if k:
            obj[b, :k] = np.asarray(o, dtype=np.float64)
            err[b, :k] = e
    np.savez_compressed(
        os.path.join(OUT, name + ".npz"),
        C=C, M=M, B=B, seed=seed,
        frames_clean=clean, clutter_max=40, clutter_salt=seed, truth=truth,
        R=np.stack([np.asarray(p["R"], dtype=np.float64) for p in poses]),
        t=np.stack([np.asarray(p["t"], dtype=np.float64).reshape(3) for p in poses]),
        K=K, blob_xy=blob_xy, blob_n=blob_n, obj=obj, err=err, nroot=nroot)
    print(name, "roots/frame", nroot.mean(), "blobs/cam", blob_n.mean())


def irregular_blob_case(name, n_frames, seed):
    """S1 on irregular (non-convex, touching, thin, single-pixel) solid blobs."""
    helpers, cams = load_reference(1)
    rng = np.random.default_rng(seed)
    H, W = synth.HEIGHT, synth.WIDTH
    frames = np.zeros((n_frames, H, W), dtype=np.uint8)
    for f in range(n_frames):
        img = frames[f]
        for _ in range(rng.integers(12, 40)):
            cx, cy = rng.integers(10, W - 10), rng.integers(10, H - 10)
            kind = rng.integers(0, 5)
            if kind == 0:      # random filled blob grown from random walk + dilation (solid via floodfill of holes)
                m = np.zeros((21, 21), np.uint8)
                x = y = 10
                for _ in range(rng.integers(5, 60)):
                    m[y, x] = 1
                    x = int(np.clip(x + rng.integers(-1, 2), 1, 19))
                    y = int(np.clip(y + rng.integers(-1, 2), 1, 19))
                img[cy - 10:cy + 11, cx - 10:cx + 11] |= m * 200
            elif kind == 1:    # single pixel (zero polygon area -> dropped by the reference)
                img[cy, cx] = 255
            elif kind == 2:    # 1-px line
                L = rng.integers(2, 9)
                if rng.integers(0, 2):
                    img[cy, cx:cx + L] = 180
                else:
                    img[cy:cy + L, cx] = 180
            elif kind == 3:    # rectangle
                img[cy:cy + rng.integers(2, 8), cx:cx + rng.integers(2, 8)] = 255
            else:              # diagonal staircase
                for k in range(rng.integers(2, 7)):
                    if cy + k < H and cx + k < W:
                        img[cy + k, cx + k] = 220
        # fill holes so that RETR_TREE emits no inner contours (parity contract: solid blobs)
        import cv2
        binary = (img > 51).astype(np.uint8)
        ff = binary.copy()
        mask = np.zeros((H + 2, W + 2), np.uint8)
        cv2.floodFill(ff, mask, (0, 0), 1)   # background is 4-connected from the corner
        holes = (ff == 0)
        img[holes] = 255
    clean = frames.copy()
    frames = synth.add_clutter(clean, 51, salt=seed)   # clutter up to exactly the threshold value
    blob_xy = np.full((n_frames, 1, MAXB, 2), -1, dtype=np.int32)
    blob_n = np.zeros((n_frames, 1), dtype=np.int32)
    for f in range(n_frames):
        img3 = np.repeat(frames[f][:, :, None], 3, axis=2).copy()
        _, pts = cams._find_dot(img3)
        real = [p for p in pts if p[0] is not None]
        blob_n[f, 0] = len(real)
        for i, p in enumerate(real):
            blob_xy[f, 0, i] = p
    np.savez_compressed(os.path.join(OUT, name + ".npz"), frames_clean=clean[:, None], clutter_max=51, clutter_salt=seed,
                        blob_xy=blob_xy, blob_n=blob_n)
    print(name, "blobs/frame", blob_n.mean())


def ring_blob_case(name, n_frames, seed):
    """S1 on blobs WITH holes (rings, frames, porous patches, nested blobs) next to solid ones: what the real
    _find_dot returns (one extra point per hole contour, hole-filled outer moments) and, per frame, whether cv2's
    contour hierarchy contains a hole.  The CUDA path does not reproduce RETR_TREE on such blobs; it must raise
    MOCAP_F_HOLES exactly on these frames and agree exactly on the others."""
    import cv2
    helpers, cams = load_reference(1)
    rng = np.random.default_rng(seed)
    H, W = synth.HEIGHT, synth.WIDTH
    frames = np.zeros((n_frames, H, W), dtype=np.uint8)
    has_hole = np.zeros((n_frames,), dtype=np.uint8)
    for f in range(n_frames):
        img = frames[f]
        solid_only = f % 3 == 0
        for _ in range(rng.integers(6, 20)):
            cx, cy = int(rng.integers(20, W - 40)), int(rng.integers(20, H - 30))
            kind = int(rng.integers(0, 5))
            if kind == 0 and not solid_only:
                cv2.circle(img, (cx, cy), int(rng.integers(3, 10)), 255, int(rng.integers(1, 3)))
            elif kind == 1:
                cv2.circle(img, (cx, cy), int(rng.integers(1, 7)), 230, -1)
            elif kind == 2 and not solid_only:
                w, h = int(rng.integers(3, 30)), int(rng.integers(3, 14))
                cv2.rectangle(img, (cx, cy), (cx + w, cy + h), 255, 1)
                if rng.integers(0, 2):
                    cv2.circle(img, (cx + w // 2, cy + h // 2), 1, 255, -1)
            elif kind == 3 and not solid_only:
                m = (rng.uniform(size=(9, 14)) < 0.75).astype(np.uint8) * 200
                img[cy:cy + 9, cx:cx + 14] = np.maximum(img[cy:cy + 9, cx:cx + 14], m)
            else:
                img[cy - 2:cy + 3, cx - 2:cx + 3] = 255
    clean = frames.copy()
    frames = synth.add_clutter(clean, 40, salt=seed)
    blob_xy = np.full((n_frames, 1, 4 * MAXB, 2), -1, dtype=np.int32)
    blob_n = np.zeros((n_frames, 1), dtype=np.int32)
    for f in range(n_frames):
        img3 = np.repeat(frames[f][:, :, None], 3, axis=2).copy()
        _, pts = cams._find_dot(img3)
        real = [p for p in pts if p[0] is not None]
        blob_n[f, 0] = len(real)
        for i, p in enumerate(real):
            blob_xy[f, 0, i] = p
        _, hier = cv2.findContours((frames[f] > 51).astype(np.uint8), cv2.RETR_TREE, cv2.CHAIN_APPROX_SIMPLE)
        if hier is not None:
            depth = lambda i: 0 if hier[0][i][3] < 0 else 1 + depth(hier[0][i][3])
            has_hole[f] = any(depth(i) % 2 == 1 for i in range(hier.shape[1]))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), frames_clean=clean[:, None], clutter_max=40, clutter_salt=seed,
                        blob_xy=blob_xy, blob_n=blob_n, has_hole=has_hole)
    print(name, "blobs/frame", blob_n.mean(), "frames with holes", int(has_hole.sum()), "of", n_frames)


def triangulate_case(name, C, F, seed):
    helpers, cams = load_reference(C)
    obs, poses, K, pts = synth.make_tracks(C, F, seed=seed)
    X = helpers.triangulate_points(obs, poses)
    errs = helpers.calculate_reprojection_errors(obs, X, poses)
    np.savez_compressed(
        os.path.join(OUT, name + ".npz"),
        obs=np.array([[[-1 if v is None else v for v in cam] for cam in fr] for fr in obs], dtype=np.float64),
        mask=np.array([[cam[0] is not None for cam in fr] for fr in obs], dtype=np.uint8),
        R=np.stack([np.asarray(p["R"], dtype=np.float64) for p in poses]),
        t=np.stack([np.asarray(p["t"], dtype=np.float64).reshape(3) for p in poses]),
        K=K, X=np.asarray(X, dtype=np.float64), err=errs, truth=pts)
    print(name, "max |X-truth|", np.abs(np.asarray(X, dtype=np.float64) - pts).max())


def ba_case(name, C, F, seed):
    helpers, cams = load_reference(C)
    obs, poses, K, pts = synth.make_tracks(C, F, seed=seed, missing_frac=0.1)
    start = synth.perturb_poses(poses, seed=seed + 1)
    # residual vector at the start point (tight parity target)
    from oracle.ref_port import RefPort
    port = RefPort([K] * C)
    x0 = port.poses_to_params(start)
    X0 = helpers.triangulate_points(obs, start)
    r0 = helpers.calculate_reprojection_errors(obs, X0, start).astype(np.float32)
    out = helpers.bundle_adjustment(obs, [dict(R=np.asarray(p["R"]), t=np.asarray(p["t"])) for p in start], NullSocket())
    Xf = helpers.triangulate_points(obs, out)
    rf = helpers.calculate_reprojection_errors(obs, Xf, out).astype(np.float32)
    cost = lambda r: 0.5 * np.sum(np.log1p(r.astype(np.float64) ** 2))
    np.savez_compressed(
        os.path.join(OUT, name + ".npz"),
        obs=np.array([[[-1 if v is None else v for v in cam] for cam in fr] for fr in obs], dtype=np.float64),
        mask=np.array([[cam[0] is not None for cam in fr] for fr in obs], dtype=np.uint8),
        K=K,
        R_true=np.stack([np.asarray(p["R"], dtype=np.float64) for p in poses]),
        t_true=np.stack([np.asarray(p["t"], dtype=np.float64).reshape(3) for p in poses]),
        R_start=np.stack([np.asarray(p["R"], dtype=np.float64) for p in start]),
        t_start=np.stack([np.asarray(p["t"], dtype=np.float64).reshape(3) for p in start]),
        R_final=np.stack([np.asarray(p["R"], dtype=np.float64) for p in out]),
        t_final=np.stack([np.asarray(p["t"], dtype=np.float64).reshape(3) for p in out]),
        x0=x0, r0=r0, rf=rf, cost0=cost(r0), costf=cost(rf), X_final=np.asarray(Xf, dtype=np.float64))
    print(name, "cost", cost(r0), "->", cost(rf))


def reference_calls_case(name):
    """What the reference returns for the inputs of the port-versus-reference tests in tests/test_oracle_pinned.py:
    S1-S3 on three frame-sets, one S4 residual vector, locate_objects, make_square, the camera chain that index.py's
    calculate_camera_pose hands to bundle_adjustment, and which hot-path names its two modules hold."""
    import hashlib
    import cv2
    from oracle.ref_harness import load_reference_index
    api = importlib.import_module("low-cost-mocap_b200.api")
    z = {}
    # S1-S3: 4 cameras, 6 markers, 3 frame-sets of the synthetic stream (seed 42)
    C, M, B = 4, 6, 3
    helpers, cams = load_reference(C)
    frames, _, poses, _ = synth.make_frame_pool(C, M, B, seed=42)
    blob_xy = np.full((B, C, MAXB, 2), -1, dtype=np.int32)
    blob_n = np.zeros((B, C), dtype=np.int32)             # 0: _find_dot returned [[None, None]]
    obj = np.full((B, MAXR, 3), np.nan)
    err = np.full((B, MAXR), np.nan)
    nroot = np.zeros((B,), dtype=np.int32)
    for b in range(B):
        pts = [cams._find_dot(np.repeat(frames[b, c][:, :, None], 3, axis=2).copy())[1] for c in range(C)]
        for c, p in enumerate(pts):
            real = [q for q in p if q[0] is not None]
            assert len(real) == len(p) or p == [[None, None]]
            blob_n[b, c] = len(real)
            for i, q in enumerate(real):
                blob_xy[b, c, i] = q
        e, o, _ = helpers.find_point_correspondance_and_object_points([list(map(list, p)) for p in pts], poses, [None] * C)
        nroot[b] = len(e)
        obj[b, :len(e)] = np.asarray(o, dtype=np.float64).reshape(-1, 3)
        err[b, :len(e)] = e
    z.update(pipe_blob_xy=blob_xy, pipe_blob_n=blob_n, pipe_obj=obj, pipe_err=err, pipe_nroot=nroot)
    # S4 residual vector: 3 cameras, 12 points (seed 2), start perturbed with seed 3
    helpers, cams = load_reference(3)
    obs, poses, K, _ = synth.make_tracks(3, 12, seed=2)
    start = synth.perturb_poses(poses, seed=3)
    X = helpers.triangulate_points(obs, start)
    z["ba_r"] = helpers.calculate_reprojection_errors(obs, X, start).astype(np.float32)
    # locate_objects on 30 seeded drone layouts
    helpers, _ = load_reference(2)
    counts, pos, heading, error, drone = [], [], [], [], []
    for seed in range(30):
        pts, errs = synth.make_drone_points(1 + seed % 3, seed % 5, seed=seed)
        found = helpers.locate_objects(pts.copy(), errs.copy())
        counts.append(len(found))
        for f in found:
            pos.append(f["pos"]); heading.append(f["heading"]); error.append(f["error"]); drone.append(f["droneIndex"])
    z.update(loc_counts=np.array(counts, dtype=np.int32), loc_pos=np.array(pos, dtype=np.float64).reshape(-1, 3),
             loc_heading=np.array(heading, dtype=np.float64), loc_error=np.array(error, dtype=np.float64),
             loc_drone=np.array(drone, dtype=np.int32))
    # make_square of a 240x320 noise frame (seed 0): the output is incompressible noise, so its digest is stored
    helpers, _ = load_reference(1)
    sq = helpers.make_square(np.random.default_rng(0).integers(0, 256, size=(240, 320, 3), dtype=np.uint8))
    z.update(square_shape=np.array(sq.shape), square_sha256=np.array(hashlib.sha256(np.ascontiguousarray(sq).tobytes()).hexdigest()))
    # index.py calculate_camera_pose: 3 cameras, 40 frames (seed 8), cv2 RNG seed 0; bundle_adjustment intercepted
    index, helpers, cams = load_reference_index(3)
    obs, poses, K, _ = synth.make_tracks(3, 40, seed=8, missing_frac=0.15)
    captured = {}

    def fake_ba(image_points, camera_poses, sio):
        captured["poses"] = camera_poses
        return camera_poses
    real_ba, real_ser = index.bundle_adjustment, index.camera_pose_to_serializable
    index.bundle_adjustment = fake_ba
    index.camera_pose_to_serializable = lambda p: p
    try:
        cv2.setRNGSeed(0)
        index.calculate_camera_pose({"cameraPoints": obs.tolist()})
    finally:
        index.bundle_adjustment, index.camera_pose_to_serializable = real_ba, real_ser
    z.update(calib_R=np.stack([np.array(p["R"], dtype=np.float64) for p in captured["poses"]]),
             calib_t=np.stack([np.array(p["t"], dtype=np.float64).reshape(3) for p in captured["poses"]]))
    z.update(helpers_names=np.array([n for n in api.PATCHED_NAMES if hasattr(helpers, n)]),
             index_names=np.array([n for n in api.PATCHED_NAMES if hasattr(index, n)]))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **z)
    print(name, "roots", nroot.tolist(), "objects", int(sum(counts)), "index holds", z["index_names"].tolist())


if __name__ == "__main__":
    which = sys.argv[1:] or ["pipe", "blobs", "rings", "tri", "ba", "calls"]
    if "calls" in which:
        reference_calls_case("reference_calls")
    if "pipe8" in which:
        pipeline_case("pipe_c8_m16", 8, 16, 100, seed=0)
    if "pipe" in which:
        pipeline_case("pipe_c2_m1", 2, 1, 100, seed=0)      # BASELINE config 1 shape
        pipeline_case("pipe_c4_m4", 4, 4, 40, seed=0)      # config 2 shape
        pipeline_case("pipe_c8_m16", 8, 16, 100, seed=0)   # config 3/4 shape (the first 10 frame-sets are those of the 10-set round-1 file)
    if "blobs" in which:
        irregular_blob_case("blobs_irregular", 30, seed=3)
    if "rings" in which:
        ring_blob_case("blobs_rings", 18, seed=4)
    if "tri" in which:
        triangulate_case("tri_c4", 4, 200, seed=5)
        triangulate_case("tri_c8", 8, 200, seed=6)
        triangulate_case("tri_c16", 16, 200, seed=7)
    if "ba" in which:
        ba_case("ba_c4", 4, 40, seed=11)
    if "ba8" in which:      # config-3 batch shape (about half an hour of reference CPU time)
        ba_case("ba_c8", 8, 60, seed=12)
    if "ba16" in which:     # reduced config-5 shape (16 cameras)
        ba_case("ba_c16", 16, 96, seed=13)
