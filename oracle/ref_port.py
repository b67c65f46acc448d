"""CPU restatement of the reference's per-frame marker pipeline.  TEST INFRASTRUCTURE.

Only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` may import this file -- as the
checker or as the timed CPU baseline, never as a product path.

The reference is plain Python on top of cv2 / numpy / scipy
(computer_code/api/helpers.py of jyjblrd/Low-Cost-Mocap).  It is not part of this
repository, so this file restates, stage by stage, what it computes, calling the SAME
third-party routines at the same precision (cv2.findContours/moments,
cv2.computeCorrespondEpilines, cv2.projectPoints, scipy.linalg.svd,
scipy.optimize.least_squares) so both the numbers and the CPU cost are those of
the reference.  Pinning: ``tests/test_oracle_pinned.py`` checks every function
here against the committed vectors in ``tests/golden/*.npz`` that
``tests/golden/make_golden.py`` wrote by running the real reference (imported via
``oracle/ref_harness.py``).  The three ``cv2.sfm`` calls are restated in
``oracle/sfm_shim.py`` -- that boundary alone is parity-UNPINNED.

Stage map (reference file:line):
  S1 find_dot                  helpers.py:143-163   Cameras._find_dot
  S2 match_and_triangulate     helpers.py:339-421   find_point_correspondance_and_object_points
  S3 triangulate_one/_many     helpers.py:293-336   triangulate_point(s)
     reprojection_error(s)     helpers.py:203-241   calculate_reprojection_error(s)
  S4 bundle_adjust             helpers.py:244-290   bundle_adjustment
     locate_objects            helpers.py:424-480   locate_objects (tracking hand-off, SURVEY §8(f) #3)
"""
from __future__ import annotations

import numpy as np
import cv2
from scipy import linalg, optimize
from scipy.spatial.transform import Rotation

from . import sfm_shim

MISSING2 = [None, None]


class RefPort:
    """Holds what the reference keeps in its ``Cameras`` singleton for this path:
    one 3x3 intrinsic matrix per camera (helpers.py:19-22, 188-193)."""

    def __init__(self, intrinsics):
        self.K = [np.asarray(k, dtype=np.float64) for k in intrinsics]

    # ------------------------------------------------- capture-side preprocessing (SURVEY §8(f) #2)
    @staticmethod
    def make_square(img):
        """helpers.py:507-523: centre the frame in a zero square, fade 8 rows above and below."""
        rows, cols, _ = img.shape
        size = max(rows, cols)
        out = np.zeros((size, size, 3), dtype=np.uint8)
        ax, ay = (size - cols) // 2, (size - rows) // 2
        out[ay:ay + rows, ax:ax + cols] = img
        for i in range(8):
            alpha = (i + 1) / 8
            out[ay - i - 1, :] = img[0, :] * (1 - alpha)
            out[ay + rows + i, :] = img[-1, :] * (1 - alpha)
        return out

    def preprocess(self, frame, cam, distortion, rotation=0):
        """helpers.py:70-82 for one camera frame (HxWx3 uint8)."""
        f = np.rot90(frame, k=rotation)
        f = self.make_square(f)
        f = cv2.undistort(f, self.K[cam], np.asarray(distortion, dtype=np.float64))
        f = cv2.GaussianBlur(f, (9, 9), 0)
        sharpen = np.array([[-2, -1, -1, -1, -2], [-1, 1, 3, 1, -1], [-1, 3, 4, 3, -1], [-1, 1, 3, 1, -1], [-2, -1, -1, -1, -2]])
        f = cv2.filter2D(f, -1, sharpen)
        return cv2.cvtColor(f, cv2.COLOR_RGB2BGR)

    # ------------------------------------------------------------------ S1
    def find_dot(self, img):
        """helpers.py:143-163.  img: HxWx3 uint8.  Returns list of [cx, cy]
        (or [[None, None]] when no contour has non-zero area).  The drawing side
        effects (helpers.py:148,156-157) are not restated: they do not feed S2-S4."""
        grey = cv2.cvtColor(img, cv2.COLOR_RGB2GRAY)
        binary = cv2.threshold(grey, 255 * 0.2, 255, cv2.THRESH_BINARY)[1]
        contours, _ = cv2.findContours(binary, cv2.RETR_TREE, cv2.CHAIN_APPROX_SIMPLE)
        out = []
        for cnt in contours:
            mo = cv2.moments(cnt)
            if mo["m00"] != 0:
                out.append([int(mo["m10"] / mo["m00"]), int(mo["m01"] / mo["m00"])])
        return out if out else [list(MISSING2)]

    # ------------------------------------------------------------------ S3
    def projection(self, k_index, pose):
        """K[k_index] @ [R|t]  (helpers.py:305-308, 351-355)."""
        Rt = np.c_[np.asarray(pose["R"], dtype=np.float64), np.asarray(pose["t"], dtype=np.float64).reshape(3)]
        return self.K[k_index] @ Rt

    @staticmethod
    def _present(views):
        """Rows of an (n,2) observation list that are not [None, None]
        (helpers.py:295-298, 217-220)."""
        return [i for i, v in enumerate(views) if not (v[0] is None and v[1] is None)]

    def triangulate_one(self, views, poses):
        """helpers.py:293-327.  NOTE the reference's quirk, kept on purpose: the
        k-th PRESENT view uses K[k], not K[camera index] (helpers.py:305-307)."""
        keep = self._present(views)
        if len(keep) <= 1:
            return [None, None, None]
        rows = []
        for k, cam in enumerate(keep):
            P = self.projection(k, poses[cam])
            x, y = views[cam][0], views[cam][1]
            rows.append(y * P[2, :] - P[1, :])
            rows.append(P[0, :] - x * P[2, :])
        A = np.array(rows).reshape((2 * len(keep), 4))
        B = A.transpose() @ A
        _, _, Vh = linalg.svd(B, full_matrices=False)
        return Vh[3, 0:3] / Vh[3, 3]

    def triangulate_many(self, observations, poses):
        """helpers.py:330-336."""
        return np.array([self.triangulate_one(v, poses) for v in observations])

    def reprojection_error(self, views, point, poses):
        """helpers.py:214-241: mean squared pixel residual; the 3D point is cast to
        float32, cv.projectPoints returns float32 pixels, the rest is float64."""
        keep = self._present(views)
        if len(keep) <= 1:
            return None
        sq = []
        X32 = np.expand_dims(np.asarray(point), axis=0).astype(np.float32)
        for k, cam in enumerate(keep):
            proj, _ = cv2.projectPoints(
                X32,
                np.array(poses[cam]["R"], dtype=np.float64),
                np.array(poses[cam]["t"], dtype=np.float64),
                self.K[k],
                np.array([]),
            )
            px = proj[0, 0]
            sq.append((views[cam][0] - float(px[0])) ** 2)
            sq.append((views[cam][1] - float(px[1])) ** 2)
        # the reference reduces an object array left to right (helpers.py:239-241)
        acc = 0.0
        for v in sq:
            acc = acc + v
        return acc / len(sq)

    def reprojection_errors(self, observations, points, poses):
        """helpers.py:203-211 (entries that yield None are skipped)."""
        out = []
        for views, pt in zip(observations, points):
            e = self.reprojection_error(views, pt, poses)
            if e is not None:
                out.append(e)
        return np.array(out, dtype=np.float64)

    # ------------------------------------------------------------------ S2
    def epipolar_line(self, root_cam, cam, point, poses):
        """helpers.py:362-364: F from the two projection matrices (cv.sfm, see
        sfm_shim), then cv.computeCorrespondEpilines on a float32 point; the line
        comes back as three float32 values widened to Python floats."""
        F = sfm_shim.fundamentalFromProjections(self.projection(root_cam, poses[root_cam]),
                                                self.projection(cam, poses[cam]))
        line = cv2.computeCorrespondEpilines(np.array([point], dtype=np.float32), 1, F)
        return line[0, 0].tolist()

    def match_and_triangulate(self, image_points, poses):
        """helpers.py:339-421 without the frame drawing.  ``image_points`` is the
        per-camera list of [x, y] lists ([None, None] sentinels are removed
        first, helpers.py:342-346).  Returns (errors (K,), object_points (K,3),
        chosen_groups) -- the third item (the winning correspondence of every
        kept root) is extra, exposed for parity tests."""
        pts = [[list(p) for p in cam_pts if not (p[0] is None and p[1] is None)] for cam_pts in image_points]
        C = len(poses)
        roots = [(0, p) for p in pts[0]]                 # helpers.py:357
        groups = [[[p]] for p in pts[0]]                 # helpers.py:349

        for cam in range(1, C):
            lines = [self.epipolar_line(rc, cam, rp, poses) for rc, rp in roots]
            here = np.array(pts[cam])
            unmatched = [list(p) for p in pts[cam]]
            for j, (a, b, c) in enumerate(lines):
                if len(here) != 0:
                    dist = np.abs(a * here[:, 0] + b * here[:, 1] + c) / np.sqrt(a ** 2 + b ** 2)
                    near = dist < 5                       # helpers.py:375
                    order = dist[near].argsort()          # helpers.py:383-385
                    cands = here[near][order].tolist()
                else:
                    cands = []
                if not cands:
                    for g in groups[j]:                   # helpers.py:387-389
                        g.append(list(MISSING2))
                    continue
                unmatched = [p for p in unmatched if p != cands[0]]      # helpers.py:391
                groups[j] = [g + [cand] for cand in cands for g in groups[j]]   # helpers.py:394-400
            for p in unmatched:                           # helpers.py:402-406
                roots.append((cam, p))
                groups.append([[list(MISSING2)] * cam + [p]])

        errors, points, chosen = [], [], []
        for root_groups in groups:                        # helpers.py:408-419
            cand_pts = self.triangulate_many(root_groups, poses)
            if np.all(cand_pts == None):                  # noqa: E711 (object-array compare, as the reference)
                continue
            errs = self.reprojection_errors(root_groups, cand_pts, poses)
            best = int(np.argmin(errs))
            points.append(cand_pts[best])
            errors.append(errs[best])
            chosen.append(root_groups[best])
        return np.array(errors), np.array(points), chosen

    # ------------------------------------------------------- tracking hand-off (SURVEY §8(f) #3)
    @staticmethod
    def locate_objects(object_points, errors):
        """helpers.py:424-480: marker triplets -> [{pos, heading, error, droneIndex}]."""
        pts = np.asarray(object_points, dtype=np.float64)
        n = pts.shape[0]
        dist = np.zeros((n, n))
        for i in range(n):
            for j in range(n):
                dist[i, j] = np.sqrt(np.sum((pts[i] - pts[j]) ** 2))
        used, found = [], []
        for i in range(n):
            if i in used:
                continue
            near = np.where(np.abs(dist[i] - 0.095) < 0.025)[0]
            if len(near) < 2:
                continue
            for a in near:
                hit = False
                for b in near:
                    if np.abs(np.sqrt(np.sum((pts[a] - pts[b]) ** 2)) - 0.15) > 0.025:
                        continue
                    used += [i, a, b]
                    centre = (pts[a] + pts[b]) / 2
                    axis = pts[a] - pts[b]
                    axis /= linalg.norm(axis)
                    heading = np.arctan2(axis[1], axis[0])
                    heading = heading - np.pi if heading > np.pi / 2 else heading
                    heading = heading + np.pi if heading < -np.pi / 2 else heading
                    found.append({"pos": centre, "heading": -heading,
                                  "error": np.mean([errors[i], errors[a], errors[b]]),
                                  "droneIndex": 0 if (pts[i] - centre)[1] > 0 else 1})
                    hit = True
                    break
                if hit:
                    break
        return found

    # --------------------------------------------------- cold-start extrinsics (SURVEY §8(f) #4)
    def calibrate_init(self, image_points, rng_seed=0, return_F=False):
        """index.py:229-270: chain of relative poses from adjacent camera pairs.  cv.findFundamentalMat is
        randomised; cv2.setRNGSeed makes this restatement repeatable (the reference never seeds it)."""
        pts = np.array(image_points)
        by_cam = pts.transpose((1, 0, 2))
        n_cam = by_cam.shape[0]
        poses = [{"R": np.eye(3), "t": np.array([[0], [0], [0]], dtype=np.float32)}]
        Fs = []
        cv2.setRNGSeed(rng_seed)
        for c in range(n_cam - 1):
            a, b = by_cam[c], by_cam[c + 1]
            both = np.where(np.all(a != None, axis=1) & np.all(b != None, axis=1))[0]      # noqa: E711
            a = np.take(a, both, axis=0).astype(np.float32)
            b = np.take(b, both, axis=0).astype(np.float32)
            F, _ = cv2.findFundamentalMat(a, b, cv2.FM_RANSAC, 1, 0.99999)
            Fs.append(F)
            E = sfm_shim.essentialFromFundamental(F, self.K[0], self.K[1])
            Rs, ts = sfm_shim.motionFromEssential(E)
            best_R, best_t, best = None, None, 0
            for i in range(4):
                X = self.triangulate_many(np.hstack([np.expand_dims(a, axis=1), np.expand_dims(b, axis=1)]),
                                          [poses[-1], {"R": Rs[i], "t": ts[i]}])
                Xc = np.array([Rs[i].T @ x for x in X])
                front = np.sum(X[:, 2] > 0) + np.sum(Xc[:, 2] > 0)
                if front > best:
                    best, best_R, best_t = front, Rs[i], ts[i]
            poses.append({"R": best_R @ poses[-1]["R"], "t": poses[-1]["t"] + (poses[-1]["R"] @ best_t)})
        return (poses, Fs) if return_F else poses

    # ------------------------------------------------------------------ S4
    @staticmethod
    def params_to_poses(params):
        """helpers.py:247-262: x = [f0, (f_i, rotvec_i, t_i) ...]; camera 0 = (I, 0)."""
        n_cam = int((params.size - 1) / 7) + 1
        poses = [{"R": np.eye(3), "t": np.array([0, 0, 0], dtype=np.float32)}]
        for i in range(n_cam - 1):
            base = 1 + 7 * i
            poses.append({
                "R": Rotation.from_rotvec(params[base + 1: base + 4]).as_matrix(),
                "t": params[base + 4: base + 7],
            })
        return poses

    def poses_to_params(self, poses):
        """helpers.py:278-285 (the focal entries are dead parameters, helpers.py:267-270;
        note the reference reads K[i] with i enumerating poses[1:], i.e. K[i-1])."""
        x = [self.K[0][0, 0]]
        for i, pose in enumerate(poses[1:]):
            x.append(self.K[i][0, 0])
            x.extend(Rotation.from_matrix(np.asarray(pose["R"], dtype=np.float64)).as_rotvec().flatten())
            x.extend(np.asarray(pose["t"], dtype=np.float64).flatten())
        return np.array(x, dtype=np.float64)

    def ba_residuals(self, params, observations):
        """helpers.py:264-276: re-triangulate every point with the trial poses, then
        the per-point mean squared reprojection error, cast to float32."""
        poses = self.params_to_poses(params)
        pts = self.triangulate_many(observations, poses)
        return self.reprojection_errors(observations, pts, poses).astype(np.float32)

    def bundle_adjust(self, observations, poses, verbose=0, return_result=False):
        """helpers.py:287-290: scipy TRF, Cauchy loss, ftol 1e-2, 2-point FD Jacobian."""
        x0 = self.poses_to_params(poses)
        res = optimize.least_squares(lambda p: self.ba_residuals(p, observations), x0,
                                     verbose=verbose, loss="cauchy", ftol=1e-2)
        out = self.params_to_poses(res.x)
        return (out, res) if return_result else out
