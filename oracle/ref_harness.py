"""Loader for the UNMODIFIED reference implementation (test infrastructure only).

This module imports ``computer_code/api/helpers.py`` of a jyjblrd/Low-Cost-Mocap
checkout named by the ``LOW_COST_MOCAP_DIR`` environment variable, as it lies,
with the three shims SURVEY.md §8(c) lists:

* a one-class ``pseyepy`` stub (the module is imported at helpers.py:12 and a
  ``Camera`` is constructed at helpers.py:24-25),
* ``helpers.drawlines`` replaced by a no-op (pure drawing, helpers.py:497-504;
  it overflows on near-vertical lines and eats the global numpy RNG),
* ``cv2.sfm`` provided by :mod:`oracle.sfm_shim` (opencv_contrib is not
  installed; that boundary is parity-UNPINNED, see DESIGN.md).

The reference is not part of this repository, so nothing here may be imported
by the tests, ``smoke()`` or ``bench.py``.  It is used only by
``tests/golden/make_golden.py``, which writes the committed golden vectors that
the tests compare against.
"""
import os
import sys
import types

REFERENCE_API_DIR = os.path.join(os.environ.get("LOW_COST_MOCAP_DIR", ""), "computer_code", "api")


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_API_DIR, "helpers.py"))


_cached = None


def load_reference(num_cameras: int, intrinsic_matrix=None):
    """Return (helpers_module, cameras_singleton) of the real reference.

    ``num_cameras`` entries of identical intrinsics are installed in
    ``Cameras.instance().camera_params`` (the shipped JSON has 4 entries only,
    helpers.py:19-22 / camera-params.json).
    """
    global _cached
    import cv2
    import numpy as np
    from . import sfm_shim

    if not reference_available():
        raise RuntimeError("reference tree not found: set LOW_COST_MOCAP_DIR to a jyjblrd/Low-Cost-Mocap checkout")

    if _cached is None:
        stub = types.ModuleType("pseyepy")

        class Camera:  # stands in for the USB camera driver (helpers.py:24)
            RES_SMALL = 0

            def __init__(self, **kw):
                self.exposure = [100] * 4
                self.gain = [10] * 4

            def read(self):
                raise RuntimeError("no camera hardware in the oracle harness")

        stub.Camera = Camera
        sys.modules["pseyepy"] = stub
        if REFERENCE_API_DIR not in sys.path:
            sys.path.insert(0, REFERENCE_API_DIR)
        if not hasattr(cv2, "sfm"):
            cv2.sfm = sfm_shim.namespace()
        import helpers  # the reference module, unmodified

        helpers.drawlines = lambda img, lines: img
        _cached = helpers

    helpers = _cached
    cams = helpers.Cameras.instance()
    if intrinsic_matrix is None:
        intrinsic_matrix = [[600.0, 0.0, 320.0], [0.0, 600.0, 240.0], [0.0, 0.0, 1.0]]
    K = np.asarray(intrinsic_matrix, dtype=np.float64)
    cams.camera_params = [
        {"intrinsic_matrix": K.copy(), "distortion_coef": np.zeros(5), "rotation": 0}
        for _ in range(num_cameras)
    ]
    cams.num_cameras = num_cameras
    return helpers, cams


class NullSocket:
    """``socketio`` stand-in for bundle_adjustment (helpers.py:274)."""

    def __init__(self):
        self.count = 0

    def emit(self, *a, **k):
        self.count += 1


_index_cached = None


def load_reference_index(num_cameras: int, intrinsic_matrix=None):
    """Import the reference's index.py (the Socket.IO handlers) with pass-through stubs for the web /
    serial / trajectory packages it needs at import time (flask, flask_socketio, flask_cors, serial,
    ruckig: none installed here, none on the hot path).  Returns (index_module, helpers, cameras)."""
    global _index_cached
    helpers, cams = load_reference(num_cameras, intrinsic_matrix)
    if _index_cached is None:
        def passthrough_decorator(*a, **k):
            def deco(fn):
                return fn
            return deco

        flask = types.ModuleType("flask")

        class Flask:
            def __init__(self, *a, **k):
                pass
            route = staticmethod(passthrough_decorator)

        flask.Flask = Flask
        flask.Response = object
        flask.request = types.SimpleNamespace()
        fsio = types.ModuleType("flask_socketio")

        class SocketIO:
            def __init__(self, *a, **k):
                self.events = []
            on = staticmethod(passthrough_decorator)

            def emit(self, *a, **k):
                self.events.append((a, k))

            def run(self, *a, **k):
                pass

        fsio.SocketIO = SocketIO
        fcors = types.ModuleType("flask_cors")
        fcors.CORS = lambda *a, **k: None
        serial = types.ModuleType("serial")
        serial.Serial = lambda *a, **k: types.SimpleNamespace(write=lambda *a, **k: None)
        ruckig = types.ModuleType("ruckig")
        for name in ("InputParameter", "OutputParameter", "Result", "Ruckig"):
            setattr(ruckig, name, object)
        for name, mod in (("flask", flask), ("flask_socketio", fsio), ("flask_cors", fcors), ("serial", serial), ("ruckig", ruckig)):
            sys.modules.setdefault(name, mod)
        import index  # the reference module, unmodified
        _index_cached = index
    return _index_cached, helpers, cams
