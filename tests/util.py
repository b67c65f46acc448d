"""Helpers shared by the CPU and GPU test files."""
import importlib
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
synth = importlib.import_module("low-cost-mocap_b200.synth")


def load_golden(name, n=None, frames=True):
    """Golden vectors written by tests/golden/make_golden.py from the real reference.  ``n``: only the first n
    frame-sets / frames (every per-frame-set array is cut; the deterministic clutter of a pixel depends on its flat
    index only, so the first n frames get the same clutter as in the full set).  ``frames=False``: skip rebuilding
    the frames (tests that start from the blob lists)."""
    z = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    if n is not None and "frames_clean" in z:
        full = z["frames_clean"].shape[0]
        for k, v in list(z.items()):
            if isinstance(v, np.ndarray) and v.ndim >= 1 and v.shape[0] == full:
                z[k] = v[:n]
    if "frames_clean" in z and frames:
        z["frames"] = synth.add_clutter(z["frames_clean"], int(z["clutter_max"]), salt=int(z["clutter_salt"]))
    return z


def poses_from(z, prefix=""):
    R, t = z["R" + prefix], z["t" + prefix]
    return [{"R": R[i], "t": t[i]} for i in range(len(R))]


def obs_from(z):
    """(F,C,2) float array + (F,C) mask  ->  object array with None for missing views."""
    obs, mask = z["obs"], z["mask"]
    F, C, _ = obs.shape
    out = np.empty((F, C, 2), dtype=object)
    for f in range(F):
        for c in range(C):
            if mask[f, c]:
                v0, v1 = obs[f, c]
                out[f, c, 0] = int(v0) if float(v0).is_integer() else float(v0)
                out[f, c, 1] = int(v1) if float(v1).is_integer() else float(v1)
            else:
                out[f, c, 0] = None
                out[f, c, 1] = None
    return out


def as3(img):
    return np.repeat(img[:, :, None], 3, axis=2).copy()


def compile_shared(cmd):
    """Run a compiler command ``cmd`` (which names its output with "-o", path) so that the library appears at that
    path only once it is complete: test processes running side by side (pytest -n) never load a half-written one."""
    out = cmd[cmd.index("-o") + 1]
    tmp = f"{out[:-len('.so')]}.{os.getpid()}.tmp.so"
    subprocess.check_call([tmp if a == out else a for a in cmd])
    os.replace(tmp, out)
    return out
