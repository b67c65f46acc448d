"""The DEVICE code of the hot path, run unchanged on the host: tests/hostcheck/simt_emu.h gives every CUDA
thread a std::thread (barriers and warp collectives are rendezvous points), so the warp-synchronous S1 code
of csrc/blob_device.cuh -- packed threshold, radix / rank / bitonic sort, lock-free union-find, 2x2-cell
moments, ranking -- is checked against the reference's golden vectors and cv2 on a machine without a GPU.
(The GPU parity tests in test_parity_gpu.py run the same code on the device through the C ABI.)"""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from tests.util import ROOT, compile_shared, load_golden

PIPE_CASES = ["pipe_c2_m1", "pipe_c4_m4", "pipe_c8_m16"]

pytestmark = pytest.mark.timeout(300)        # a divergent barrier in the device code shows up as a deadlock here

HC = os.path.join(ROOT, "tests", "hostcheck")
CUDA_INC = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")


@pytest.fixture(scope="module")
def blob_emu():
    src = os.path.join(HC, "blob_emu_host.cpp")
    out = os.path.join(HC, "libblob_emu.so")
    compile_shared(["g++", "-std=c++20", "-O2", "-shared", "-fPIC", "-pthread", "-I" + CUDA_INC, "-Wno-attributes",
                           "-fno-strict-aliasing", "-o", out, src])
    lib = ctypes.CDLL(out)

    def detect(img, threshold=51, max_blobs=64, E=1024, force_cta=0, seed=1):
        img = np.ascontiguousarray(img, dtype=np.uint8)
        H, W = img.shape
        xy = np.zeros((max_blobs, 2), np.int32); n = np.zeros(1, np.int32)
        mom = np.zeros((max_blobs, 4), np.int64); fl = np.zeros(1, np.int32)
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        rc = lib.hc_blob_detect(p(img), W, H, int(threshold), max_blobs, E, force_cta, seed, p(xy), p(n), p(mom), p(fl))
        assert rc >= 0, rc
        return {"path": rc, "n": int(n[0]), "xy": xy[:n[0]].copy(), "mom": mom[:n[0]].copy(), "flags": int(fl[0])}
    return detect


@pytest.mark.parametrize("name", PIPE_CASES + ["blobs_irregular"])
def test_blob_device_code_vs_reference_golden(blob_emu, name):
    """Exact blob count, centres and order (helpers.py:143-163) on the reference's golden frames, through the
    one-warp-per-image variant and through the 128-thread variant of the same device function."""
    z = load_golden(name, n=12 if name.startswith("pipe_") else None)
    frames = z["frames"]
    B, C = frames.shape[:2]
    step = max(1, (B * C) // 16)                         # a spread of ~24 images per case keeps the CPU suite short
    for idx in range(0, B * C, step):
        b, c = divmod(idx, C)
        k = int(z["blob_n"][b, c])
        for force_cta in (0, 1):
            d = blob_emu(frames[b, c], force_cta=force_cta, seed=idx)
            assert d["flags"] == 0 and d["n"] == k, (b, c, force_cta)
            assert np.array_equal(d["xy"], z["blob_xy"][b, c, :k]), (b, c, force_cta)


def test_blob_device_code_moments_and_pixel_counts_vs_cv2(blob_emu):
    """A2 / SX6 / SY6 are the integers cv.moments accumulates for the contour; the pixel count equals
    cv2.connectedComponentsWithStats (8-connectivity)."""
    import cv2
    z = load_golden("blobs_irregular")
    for f, frame in enumerate(z["frames"][:, 0]):
        binary = (frame > 51).astype(np.uint8)
        contours, _ = cv2.findContours(binary * 255, cv2.RETR_TREE, cv2.CHAIN_APPROX_SIMPLE)
        _, lab, stats, _ = cv2.connectedComponentsWithStats(binary, connectivity=8)
        kept = []
        for cnt in contours:
            m = cv2.moments(cnt)
            if m["m00"] != 0:
                x0, y0 = cnt[0, 0]
                kept.append((round(m["m00"] * 2), round(m["m10"] * 6), round(m["m01"] * 6), stats[lab[y0, x0], cv2.CC_STAT_AREA]))
        d = blob_emu(frame, seed=f)
        assert d["n"] == len(kept)
        for i, ref in enumerate(kept):
            assert tuple(int(v) for v in d["mom"][i]) == ref, (f, i)


@pytest.mark.parametrize("threshold", [0, 1, 50, 51, 52, 127, 128, 129, 200, 254, 255])
def test_packed_threshold_is_strictly_greater(blob_emu, threshold):
    """pix > threshold for every byte value: the packed compare has two regimes around 128, and the cheap
    "any byte above?" test of the stream loop must agree with the per-pixel mask (checked inside the harness)."""
    img = np.zeros((480, 640), np.uint8)
    for v in range(256):                       # 256 isolated 2x2 squares, one per grey value
        y, x = 8 + 12 * (v // 32), 8 + 12 * (v % 32)
        img[y:y + 2, x:x + 2] = v
    d = blob_emu(img, threshold=threshold, E=1024)
    expect = 255 - threshold
    assert d["n"] == min(expect, 64) and ((d["flags"] & 2) != 0) == (expect > 64)


def test_capacity_paths_of_the_blob_code(blob_emu):
    """More segments than a warp's slab, more blobs than a warp accumulates, a blob wider than a row index span,
    a frame full of set pixels: the warp variant must decline (uniformly) and the CTA variant must finish; both
    agree with the oracle's _find_dot."""
    from oracle.ref_port import RefPort
    port = RefPort([np.eye(3)])
    rng = np.random.default_rng(3)
    cases = []
    a = np.zeros((480, 640), np.uint8)                     # 70 small blobs: > 64 warp accumulators
    for k in range(70):
        y, x = 10 + 6 * (k // 35), 20 + 16 * (k % 35)
        a[y:y + 3, x:x + 3] = 255
    cases.append(a)
    b = np.zeros((480, 640), np.uint8); b[300:304, 100:400] = 255          # long thin blob
    cases.append(b)
    c = np.zeros((480, 640), np.uint8); c[40:440, 300:330] = 200           # tall blob: 400 rows, 800+ segments
    cases.append(c)
    d = np.zeros((480, 640), np.uint8)                     # irregular blobs grown by random walks
    for _ in range(12):
        y, x = int(rng.integers(40, 440)), int(rng.integers(40, 600))
        for _ in range(150):
            d[y - 1:y + 2, x - 1:x + 2] = 255
            y = int(np.clip(y + rng.integers(-2, 3), 2, 477)); x = int(np.clip(x + rng.integers(-2, 3), 2, 637))
    import cv2
    d = cv2.morphologyEx(d, cv2.MORPH_CLOSE, np.ones((5, 5), np.uint8))   # solid blobs (no holes): the S1 contract
    filled = d.copy()
    contours, _ = cv2.findContours(d, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_NONE)
    cv2.drawContours(filled, contours, -1, 255, thickness=cv2.FILLED)
    cases.append(filled)
    for i, img in enumerate(cases):
        ref = [q for q in port.find_dot(np.repeat(img[:, :, None], 3, axis=2)) if q[0] is not None]
        got = blob_emu(img, max_blobs=64, E=4096, seed=i)
        assert got["xy"].tolist() == ref[:64], i
        assert got["n"] == min(len(ref), 64)
        forced = blob_emu(img, max_blobs=64, E=4096, force_cta=1, seed=i)
        assert forced["xy"].tolist() == got["xy"].tolist() and forced["n"] == got["n"]
    assert blob_emu(cases[0], E=4096)["path"] == 2          # the warp variant declined 70 blobs
    assert blob_emu(cases[2], E=4096)["path"] == 2          # and 800 segments
    assert blob_emu(cases[1], E=4096)["path"] == 1


# ------------------------------------------------------------------------------------------------ S2 + S3
X_TOL = 1e-7          # pose units (BASELINE north_star)
ERR_RTOL = 1e-9


@pytest.fixture(scope="module")
def match_emu():
    src = os.path.join(HC, "match_emu_host.cpp")
    out = os.path.join(HC, "libmatch_emu.so")
    compile_shared(["g++", "-std=c++20", "-O2", "-shared", "-fPIC", "-pthread", "-I" + CUDA_INC, "-Wno-attributes",
                           "-fno-strict-aliasing", "-o", out, src])
    lib = ctypes.CDLL(out)

    def match(K, R, t, blob_xy, blob_n, max_roots=128, max_cands=8, max_groups=4096):
        C = len(R)
        B = blob_n.shape[0]
        MB = blob_xy.shape[2]
        K = np.ascontiguousarray(np.stack([K] * C) if np.ndim(K) == 2 else K, dtype=np.float64)
        R = np.ascontiguousarray(R, dtype=np.float64); t = np.ascontiguousarray(np.reshape(t, (C, 3)), dtype=np.float64)
        xy = np.ascontiguousarray(blob_xy, dtype=np.int32); n = np.ascontiguousarray(blob_n, dtype=np.int32)
        obj = np.zeros((B, max_roots, 3)); err = np.zeros((B, max_roots))
        k = np.zeros(B, np.int32); fl = np.zeros(B, np.int32)
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        assert lib.hc_match_triangulate(p(K), p(R), p(t), C, p(xy), p(n), B, MB, max_roots, max_cands, ctypes.c_uint(max_groups),
                                        p(obj), p(err), p(k), p(fl)) == 0
        return {"obj": obj, "err": err, "n": k, "flags": fl}

    def chunked(K, R, t, blob_xy, blob_n, chunk, item_cap, n_ctas=3, max_roots=128, max_cands=8, max_groups=4096):
        """k_match_triangulate + k_match_chunks on an emulated grid: frame-sets of more than ``chunk`` groups go to several warps"""
        C = len(R)
        B = blob_n.shape[0]
        MB = blob_xy.shape[2]
        K = np.ascontiguousarray(np.stack([K] * C) if np.ndim(K) == 2 else K, dtype=np.float64)
        R = np.ascontiguousarray(R, dtype=np.float64); t = np.ascontiguousarray(np.reshape(t, (C, 3)), dtype=np.float64)
        xy = np.ascontiguousarray(blob_xy, dtype=np.int32); n = np.ascontiguousarray(blob_n, dtype=np.int32)
        obj = np.zeros((B, max_roots, 3)); err = np.zeros((B, max_roots))
        k = np.zeros(B, np.int32); fl = np.zeros(B, np.int32); txy = np.zeros((B, max_roots, C, 2), np.int32); stats = np.zeros(3, np.int64)
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        assert lib.hc_match_triangulate_chunked(p(K), p(R), p(t), C, p(xy), p(n), B, MB, max_roots, max_cands, ctypes.c_uint(max_groups),
                                                ctypes.c_uint(chunk), ctypes.c_uint(item_cap), n_ctas,
                                                p(obj), p(err), p(k), p(fl), p(txy), p(stats)) == 0
        return {"obj": obj, "err": err, "n": k, "flags": fl, "track_xy": txy, "items": int(stats[0]), "claimed": int(stats[1]), "armed": int(stats[2])}
    match.chunked = chunked
    return match


@pytest.mark.parametrize("name", PIPE_CASES)
def test_matcher_device_code_vs_reference_golden(match_emu, name):
    """find_point_correspondance_and_object_points (helpers.py:339-421) as the device code computes it, one
    emulated warp per frame-set: same kept roots, 3D points within 1e-7 pose units, reprojection errors equal."""
    z = load_golden(name, frames=False)
    B = min(len(z["nroot"]), 20)                        # 100 heavy frame-sets take a while one emulated warp at a time
    d = match_emu(z["K"], z["R"], z["t"], z["blob_xy"][:B], z["blob_n"][:B])
    k = d["n"]
    assert np.array_equal(k, z["nroot"][:B]) and not d["flags"].any()
    for b in range(len(k)):
        if k[b]:
            assert np.abs(d["obj"][b, :k[b]] - z["obj"][b, :k[b]]).max() <= X_TOL
            assert np.allclose(d["err"][b, :k[b]], z["err"][b, :k[b]], rtol=ERR_RTOL, atol=1e-12)


def test_chunked_matcher_equals_one_warp_per_frame_set(match_emu):
    """Frame-sets cut into items of `chunk` candidate groups and folded back together (k_match_chunks) give bit for bit what
    one warp walking the whole frame-set gives -- points, errors, counts, flags, the winners' pixels -- for chunks of one
    round (32 groups, every root spans several items), for larger chunks (frame-sets on both sides of the threshold), with
    an item list that is too short (the frame-sets that do not fit are finished by the claiming warp), and with ties
    between groups in different items (duplicated blobs: np.argmin keeps the first group)."""
    z = load_golden("pipe_c8_m16", frames=False)
    B = 10
    xy, nb = z["blob_xy"][:B].copy(), z["blob_n"][:B].copy()
    # ties across items: frame-set 1 sees the same blob twice in cameras 2 and 5
    for c in (2, 5):
        k = int(nb[1, c])
        xy[1, c, k] = xy[1, c, 0]; nb[1, c] = k + 1
    one = match_emu.chunked(z["K"], z["R"], z["t"], xy, nb, chunk=0, item_cap=0)
    ref = match_emu(z["K"], z["R"], z["t"], xy, nb)
    assert one["items"] == 0 and np.array_equal(one["n"], ref["n"]) and np.array_equal(one["flags"], ref["flags"])

    def same(a, b):
        if not (np.array_equal(a["n"], b["n"]) and np.array_equal(a["flags"], b["flags"])):
            return False
        for s in range(B):
            k = a["n"][s]
            if not (np.array_equal(a["obj"][s, :k], b["obj"][s, :k]) and np.array_equal(a["err"][s, :k], b["err"][s, :k])
                    and np.array_equal(a["track_xy"][s, :k], b["track_xy"][s, :k])):
                return False
        return True
    for s in range(B):
        k = ref["n"][s]
        assert np.array_equal(one["obj"][s, :k], ref["obj"][s, :k]) and np.array_equal(one["err"][s, :k], ref["err"][s, :k])
    many = match_emu.chunked(z["K"], z["R"], z["t"], xy, nb, chunk=32, item_cap=4096)
    assert many["items"] > 5 * B and many["claimed"] >= many["items"] and many["armed"] == 0 and same(many, one)
    some = match_emu.chunked(z["K"], z["R"], z["t"], xy, nb, chunk=256, item_cap=4096, n_ctas=2)
    assert 0 < some["items"] < many["items"] and some["armed"] == 0 and same(some, one)
    short = match_emu.chunked(z["K"], z["R"], z["t"], xy, nb, chunk=32, item_cap=many["items"] // 3)
    assert short["items"] == many["items"] and short["armed"] == 0 and same(short, one)
    # the capacity flags travel with the frame-set through the items
    tight = match_emu.chunked(z["K"], z["R"], z["t"], xy, nb, chunk=32, item_cap=4096, max_roots=8, max_groups=40)
    tight1 = match_emu.chunked(z["K"], z["R"], z["t"], xy, nb, chunk=0, item_cap=0, max_roots=8, max_groups=40)
    assert tight1["flags"].any() and same(tight, tight1)


@pytest.mark.parametrize("name", ["pipe_c2_m1", "pipe_c4_m4"])
def test_pixels_to_points_through_the_device_code_on_host(blob_emu, match_emu, name):
    """The whole S1 -> S2 -> S3 chain of the kernels, from the golden FRAMES to 3D points, without a GPU."""
    z = load_golden(name, n=8)
    frames = z["frames"][:8]
    B, C = frames.shape[:2]
    xy = np.zeros((B, C, 64, 2), np.int32); n = np.zeros((B, C), np.int32)
    for b in range(B):
        for c in range(C):
            d = blob_emu(frames[b, c], seed=b * C + c)
            n[b, c] = d["n"]; xy[b, c, :d["n"]] = d["xy"]
    assert np.array_equal(n, z["blob_n"][:B])
    m = match_emu(z["K"], z["R"], z["t"], xy, n)
    assert np.array_equal(m["n"], z["nroot"][:B])
    for b in range(B):
        k = m["n"][b]
        if k:
            assert np.abs(m["obj"][b, :k] - z["obj"][b, :k]).max() <= X_TOL


def test_matcher_device_code_capacity_flags(match_emu):
    """More roots than max_roots: the warp reports the overflow flag and keeps the first max_roots roots; a
    frame-set without blobs yields no points."""
    z = load_golden("pipe_c8_m16", frames=False)
    full = match_emu(z["K"], z["R"], z["t"], z["blob_xy"][:2], z["blob_n"][:2])
    small = match_emu(z["K"], z["R"], z["t"], z["blob_xy"][:2], z["blob_n"][:2], max_roots=8)
    assert (small["flags"] != 0).all() and (small["n"] <= 8).all() and (full["flags"] == 0).all()
    empty = match_emu(z["K"], z["R"], z["t"], z["blob_xy"][:1], np.zeros((1, 8), np.int32))
    assert empty["n"][0] == 0


# ------------------------------------------------------------------------- the single-pass pipeline kernel
@pytest.fixture(scope="module")
def fused_emu():
    src = os.path.join(HC, "fused_emu_host.cpp")
    out = os.path.join(HC, "libfused_emu.so")
    compile_shared(["g++", "-std=c++20", "-O2", "-shared", "-fPIC", "-pthread", "-I" + CUDA_INC, "-Wno-attributes",
                           "-fno-strict-aliasing", "-o", out, src])
    lib = ctypes.CDLL(out)

    def run(frames, K, R, t, threshold=51, max_blobs=64, E=1024, max_roots=128, max_cands=8, max_groups=4096, n_warps=8, runs=2, phased=0):
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        channels = 3 if frames.ndim == 5 else 1                 # [B, C, H, W, 3]: the interleaved layout _find_dot receives
        B, C, H, W = frames.shape[:4]
        K = np.ascontiguousarray(np.stack([K] * C) if np.ndim(K) == 2 else K, dtype=np.float64)
        R = np.ascontiguousarray(R, dtype=np.float64); t = np.ascontiguousarray(np.reshape(t, (C, 3)), dtype=np.float64)
        obj = np.zeros((B, max_roots, 3)); err = np.zeros((B, max_roots)); k = np.zeros(B, np.int32); fl = np.zeros(B, np.int32)
        bxy = np.zeros((B * C, max_blobs, 2), np.int32); bn = np.zeros(B * C, np.int32)
        iw = np.zeros(B * C, np.uint32); sw = np.zeros(B, np.uint32); cnt = np.zeros(4, np.int64)
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        rc = lib.hc_pipeline_fused(p(frames), B, C, W, H, int(threshold), p(K), p(R), p(t), max_blobs, E, max_roots, max_cands,
                                   ctypes.c_uint(max_groups), n_warps, runs, phased, p(obj), p(err), p(k), p(fl), p(bxy), p(bn), p(iw), p(sw), p(cnt), channels)
        assert rc == 0
        return {"obj": obj, "err": err, "n": k, "flags": fl, "blob_xy": bxy.reshape(B, C, max_blobs, 2), "blob_n": bn.reshape(B, C),
                "deferred_images": iw[:cnt[0]].tolist(), "deferred_sets": sw[:cnt[1]].tolist(), "dirty_scratch": int(cnt[2])}
    return run


@pytest.mark.parametrize("name,n_warps", [("pipe_c2_m1", 4), ("pipe_c4_m4", 8), ("pipe_c4_m4", 16), ("pipe_c8_m16", 8)])
def test_single_pass_kernel_on_host_vs_reference_golden(fused_emu, name, n_warps):
    """k_pipeline_fused itself, every CUDA thread a host thread racing for units and for the last-arriver roles,
    run twice on the same scratch (every counter must re-arm itself): golden blob lists and 3D points."""
    B = 10 if name != "pipe_c8_m16" else 5
    z = load_golden(name, n=B)
    d = fused_emu(z["frames"][:B], z["K"], z["R"], z["t"], n_warps=n_warps, runs=2)
    assert d["deferred_images"] == [] and d["deferred_sets"] == [] and d["dirty_scratch"] == 0
    assert np.array_equal(d["blob_n"], z["blob_n"][:B])
    assert np.array_equal(d["n"], z["nroot"][:B]) and not d["flags"].any()
    for b in range(B):
        for c in range(d["blob_n"].shape[1]):
            k = d["blob_n"][b, c]
            assert np.array_equal(d["blob_xy"][b, c, :k], z["blob_xy"][b, c, :k])
        k = d["n"][b]
        if k:
            assert np.abs(d["obj"][b, :k] - z["obj"][b, :k]).max() <= X_TOL
            assert np.allclose(d["err"][b, :k], z["err"][b, :k], rtol=ERR_RTOL, atol=1e-12)


@pytest.mark.parametrize("shape,threshold", [((48, 32, 2), 51), ((320, 320, 3), 51), ((1024, 768, 1), 51), ((640, 480, 2), 180)])
def test_single_pass_kernel_on_host_other_geometries(fused_emu, blob_emu, match_emu, shape, threshold):
    """Image sizes whose segment count is not a multiple of a warp iteration (ragged slices), the 64-bit
    accumulator variant (1024x768), tiny frames, the AND regime of the packed threshold: the single-pass kernel
    agrees with the separately driven blob and matcher device code, and S1 with the oracle's _find_dot."""
    from oracle.ref_port import RefPort
    W, H, C = shape
    rng = np.random.default_rng(W + H + C)
    B = 3
    frames = rng.integers(0, 40, size=(B, C, H, W), dtype=np.uint8)
    yy, xx = np.mgrid[:H, :W]
    for b in range(B):
        for c in range(C):
            for _ in range(4):
                cy, cx, sg = rng.uniform(4, H - 4), rng.uniform(4, W - 4), rng.uniform(1.0, 2.5)
                frames[b, c] = np.maximum(frames[b, c], (255 * np.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / (2 * sg * sg))).astype(np.uint8))
    K = np.array([[W * 1.0, 0, W / 2.0], [0, W * 1.0, H / 2.0], [0, 0, 1]])
    R = np.stack([np.eye(3)] * C); t = np.array([[-0.3 * c, 0.0, 0.0] for c in range(C)])
    d = fused_emu(frames, K, R, t, threshold=threshold, max_roots=32, n_warps=8, runs=2)
    assert d["dirty_scratch"] == 0 and d["deferred_images"] == [] and d["deferred_sets"] == []
    port = RefPort([K] * C)
    xy = np.zeros((B, C, 64, 2), np.int32); n = np.zeros((B, C), np.int32)
    for b in range(B):
        for c in range(C):
            s1 = blob_emu(frames[b, c], threshold=threshold, seed=b)
            n[b, c] = s1["n"]; xy[b, c, :s1["n"]] = s1["xy"]
            if threshold == 51:
                ref = [q for q in port.find_dot(np.repeat(frames[b, c][:, :, None], 3, axis=2)) if q[0] is not None]
                assert s1["xy"].tolist() == ref
    assert np.array_equal(d["blob_n"], n) and np.array_equal(d["blob_xy"], xy)
    m = match_emu(K, R, t, xy, n, max_roots=32)
    assert np.array_equal(d["n"], m["n"]) and np.array_equal(d["flags"], m["flags"])
    for b in range(B):
        k = m["n"][b]
        assert np.array_equal(d["obj"][b, :k], m["obj"][b, :k]) and np.array_equal(d["err"][b, :k], m["err"][b, :k])


def test_single_pass_kernel_on_host_defers_what_a_warp_cannot_hold(fused_emu):
    """An image with 70 blobs exceeds a warp's accumulators: the kernel must put the image and its frame-set on
    the worklists (for k_blob_reduce / k_match_triangulate), finish every other frame-set, and leave no counter
    behind except the deferred image's segment list."""
    z = load_golden("pipe_c4_m4", n=6)
    frames = z["frames"][:6].copy()
    for k in range(70):
        y, x = 10 + 6 * (k // 35), 20 + 16 * (k % 35)
        frames[2, 1, y:y + 3, x:x + 3] = 255
    d = fused_emu(frames, z["K"], z["R"], z["t"], runs=1)
    assert d["deferred_images"] == [2 * 4 + 1] and d["deferred_sets"] == [2] and d["dirty_scratch"] == 0
    for b in (0, 1, 3, 4, 5):
        k = d["n"][b]
        assert k == z["nroot"][b] and np.abs(d["obj"][b, :k] - z["obj"][b, :k]).max() <= X_TOL


def test_device_code_has_no_unintended_data_races(tmp_path):
    """ThreadSanitizer over the emulated kernel: every CUDA thread is a host thread, so a missing barrier or
    fence between warps (or lanes) is a reportable data race.  The union-find of the blob reduce races BY DESIGN
    (lock-free path halving + atomicMin, blob_device.cuh) and is suppressed; nothing else may be reported, on
    light frame-sets and on the deferral path."""
    import shutil
    tsan = subprocess.run(["gcc", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not tsan or not os.path.isabs(tsan) or not os.path.exists(tsan):
        pytest.skip("libtsan not available")
    libs = {}
    for name in ("fused", "blob", "match"):
        libs[name] = str(tmp_path / f"lib{name}_tsan.so")
        subprocess.check_call(["g++", "-std=c++20", "-O1", "-g", "-fsanitize=thread", "-shared", "-fPIC", "-pthread", "-I" + CUDA_INC,
                               "-Wno-attributes", "-Wno-tsan", "-fno-strict-aliasing", "-o", libs[name], os.path.join(HC, f"{name}_emu_host.cpp")])
    lib = libs["fused"]
    supp = tmp_path / "supp.txt"
    supp.write_text("race:uf_find\nrace:uf_unite\nrace:atomicMin\n")
    env = dict(os.environ, LD_PRELOAD=tsan, TSAN_OPTIONS=f"report_signal_unsafe=0 history_size=4 exitcode=0 suppressions={supp}")
    for extra in ([], ["crowded"], ["phased", "crowded"]):
        r = subprocess.run([shutil.which("python") or "python", os.path.join(HC, "tsan_fused_run.py"), ROOT, lib, "pipe_c4_m4"] + extra,
                           capture_output=True, text=True, env=env, timeout=280)
        out = r.stdout + r.stderr
        assert "RESULT 0" in out, out[-2000:]
        assert "WARNING: ThreadSanitizer" not in out, out[:4000]
    # the blob code on its own (one-warp and 128-thread variants, light and crowded image) and the matcher
    r = subprocess.run([shutil.which("python") or "python", os.path.join(HC, "tsan_blob_match_run.py"), ROOT, libs["blob"], libs["match"]],
                       capture_output=True, text=True, env=env, timeout=280)
    out = r.stdout + r.stderr
    assert out.count("BLOB") == 4 and "MATCH True" in out and "CHUNKED True" in out, out[-2000:]
    assert "WARNING: ThreadSanitizer" not in out, out[:4000]


def test_blob_device_code_fuzz_vs_cv2(blob_emu):
    """Random solid shapes (random walks of squares, filled; touching, on the border, in images as small as 16x2)
    through both variants of the blob code: centres, count and order identical to cv2's findContours + moments."""
    import cv2
    from oracle.ref_port import RefPort
    port = RefPort([np.eye(3)])
    rng = np.random.default_rng(11)
    done = blobs = 0
    while done < 150:
        W = int(rng.choice([16, 32, 48, 64, 160, 320])); H = int(rng.integers(2, 160))
        img = np.zeros((H, W), np.uint8)
        for _ in range(int(rng.integers(0, 10))):
            y, x, r = int(rng.integers(0, H)), int(rng.integers(0, W)), int(rng.integers(0, 3))
            for _ in range(int(rng.integers(1, 50))):
                img[max(0, y - r):y + r + 1, max(0, x - r):x + r + 1] = 255
                y = int(np.clip(y + rng.integers(-2, 3), 0, H - 1)); x = int(np.clip(x + rng.integers(-2, 3), 0, W - 1))
        contours, _ = cv2.findContours(img, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_NONE)
        cv2.drawContours(img, contours, -1, 255, thickness=cv2.FILLED)
        _, hier = cv2.findContours(img, cv2.RETR_CCOMP, cv2.CHAIN_APPROX_NONE)
        if hier is not None and (hier[0][:, 3] >= 0).any():
            continue                                          # a hole survived: outside the S1 contract (DESIGN.md section 7)
        grey = (img > 0).astype(np.uint8) * int(rng.integers(60, 256))
        ref = [q for q in port.find_dot(np.repeat(grey[:, :, None], 3, axis=2)) if q[0] is not None]
        for force_cta in (0, 1):
            d = blob_emu(grey, E=4096, force_cta=force_cta, seed=done)
            assert d["xy"].tolist() == ref[:64], (done, W, H, force_cta)
        blobs += len(ref)
        done += 1
    assert blobs > 300


def test_matcher_device_code_fuzz_vs_oracle(match_emu):
    """Random blob constellations that do not come from any scene (many wrong correspondences, ragged counts,
    near-threshold distances to epipolar lines): kept roots, their order and the chosen points equal the oracle's."""
    import importlib
    from oracle.ref_port import RefPort
    synth = importlib.import_module("low-cost-mocap_b200.synth")
    rng = np.random.default_rng(78)
    for C in (3, 5):
        poses, K = synth.make_rig(C)
        port = RefPort([K] * C)
        B, MB = 25, 16
        xy = np.zeros((B, C, MB, 2), np.int32); n = np.zeros((B, C), np.int32)
        for b in range(B):
            pts3 = rng.uniform(-0.5, 0.5, size=(int(rng.integers(0, 5)), 3)) + np.array([0, 0, 3.0])
            for c in range(C):
                lst = [list(map(int, synth.project(p[None], poses[c], K)[0])) for p in pts3 if rng.uniform() < 0.85]
                lst += [[int(rng.integers(100, 540)), int(rng.integers(100, 380))] for _ in range(int(rng.integers(0, 4)))]
                uniq = [list(q) for q in dict.fromkeys(tuple(q) for q in lst)]
                uniq = [uniq[i] for i in rng.permutation(len(uniq))][:MB]
                n[b, c] = len(uniq)
                if uniq:
                    xy[b, c, :len(uniq)] = uniq
        R = np.stack([np.asarray(p["R"], dtype=np.float64) for p in poses]); t = np.stack([np.asarray(p["t"], dtype=np.float64).reshape(3) for p in poses])
        d = match_emu(K, R, t, xy, n, max_roots=64, max_cands=16)
        assert not d["flags"].any()
        for b in range(B):
            lists = [[list(map(int, xy[b, c, i])) for i in range(n[b, c])] for c in range(C)]
            e, o, _ = port.match_and_triangulate(lists, poses)
            assert d["n"][b] == len(e), (C, b)
            if len(e):
                ref = np.asarray(o, dtype=np.float64)
                scale = np.maximum(1.0, np.abs(ref).max(axis=1, keepdims=True))      # wrong correspondences are ill-conditioned
                assert (np.abs(d["obj"][b, :len(e)] - ref) / scale).max() <= 1e-6, (C, b)
                assert np.allclose(d["err"][b, :len(e)], e, rtol=1e-6, atol=1e-9)


# ------------------------------------------------- the phase-synchronous variant (MOCAP_PIPELINE=phased, opt-in)
@pytest.mark.parametrize("name", PIPE_CASES)
def test_phased_kernel_on_host_vs_reference_golden(fused_emu, name):
    """k_pipeline_phased (csrc/fused_phased.cuh): images and frame-sets are queued per CTA and the CTA changes
    phase as a whole.  Same golden results as the single-pass kernel, every counter re-armed after a run."""
    B = 12 if name != "pipe_c8_m16" else 6
    z = load_golden(name, n=B)
    d = fused_emu(z["frames"][:B], z["K"], z["R"], z["t"], runs=2, phased=1)
    assert d["deferred_images"] == [] and d["deferred_sets"] == [] and d["dirty_scratch"] == 0
    assert np.array_equal(d["blob_n"], z["blob_n"][:B])
    assert np.array_equal(d["n"], z["nroot"][:B]) and not d["flags"].any()
    for b in range(B):
        for c in range(d["blob_n"].shape[1]):
            k = d["blob_n"][b, c]
            assert np.array_equal(d["blob_xy"][b, c, :k], z["blob_xy"][b, c, :k])
        k = d["n"][b]
        if k:
            assert np.abs(d["obj"][b, :k] - z["obj"][b, :k]).max() <= X_TOL
            assert np.allclose(d["err"][b, :k], z["err"][b, :k], rtol=ERR_RTOL, atol=1e-12)


def test_phased_kernel_on_host_equals_single_pass_kernel(fused_emu):
    """Bit-identical outputs of the two kernels on ragged geometry, many small frame-sets (the queues wrap several
    times) and a crowded image (deferral to the worklists)."""
    rng = np.random.default_rng(5)
    W, H, C, B = 48, 32, 3, 40
    frames = rng.integers(0, 40, size=(B, C, H, W), dtype=np.uint8)
    yy, xx = np.mgrid[:H, :W]
    for b in range(B):
        for c in range(C):
            for _ in range(3):
                cy, cx, sg = rng.uniform(3, H - 3), rng.uniform(3, W - 3), rng.uniform(0.8, 1.8)
                frames[b, c] = np.maximum(frames[b, c], (255 * np.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / (2 * sg * sg))).astype(np.uint8))
    K = np.array([[W * 1.0, 0, W / 2.0], [0, W * 1.0, H / 2.0], [0, 0, 1]])
    R = np.stack([np.eye(3)] * C); t = np.array([[-0.3 * c, 0.0, 0.0] for c in range(C)])
    a = fused_emu(frames, K, R, t, max_roots=32, runs=2, phased=0)
    b = fused_emu(frames, K, R, t, max_roots=32, runs=2, phased=1)
    # the only images that may leave the fast path are the ones holding a blob with a hole (RETR_TREE work, blob_holes.cuh)
    import cv2
    holed = []
    for i, img in enumerate(frames.reshape(B * C, H, W)):
        _, hier = cv2.findContours(cv2.threshold(img, 255 * 0.2, 255, cv2.THRESH_BINARY)[1], cv2.RETR_TREE, cv2.CHAIN_APPROX_SIMPLE)
        if hier is not None and (hier[0, :, 3] >= 0).any():
            holed.append(i)
    assert b["dirty_scratch"] == 0 and b["deferred_images"] == holed and b["deferred_sets"] == sorted({i // C for i in holed})
    assert np.array_equal(a["blob_n"], b["blob_n"]) and np.array_equal(a["blob_xy"], b["blob_xy"])
    assert np.array_equal(a["n"], b["n"]) and np.array_equal(a["flags"], b["flags"])
    for s in range(B):
        k = a["n"][s]
        assert np.array_equal(a["obj"][s, :k], b["obj"][s, :k]) and np.array_equal(a["err"][s, :k], b["err"][s, :k])
    z = load_golden("pipe_c4_m4", n=6)
    crowded = z["frames"][:6].copy()
    for k in range(70):
        y, x = 10 + 6 * (k // 35), 20 + 16 * (k % 35)
        crowded[2, 1, y:y + 3, x:x + 3] = 255
    d = fused_emu(crowded, z["K"], z["R"], z["t"], runs=1, phased=1)
    assert d["deferred_images"] == [2 * 4 + 1] and d["deferred_sets"] == [2] and d["dirty_scratch"] == 0
    for s in (0, 1, 3, 4, 5):
        k = d["n"][s]
        assert k == z["nroot"][s] and np.abs(d["obj"][s, :k] - z["obj"][s, :k]).max() <= X_TOL


# ---------------------------------------------------------------------------------------------------------------
# S4: the persistent, grid-synchronous bundle adjustment kernel (csrc/ba_device.cuh) on the host
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ba_emu():
    out = os.path.join(HC, "libba_dev_emu.so")
    compile_shared(["g++", "-std=c++20", "-O2", "-shared", "-fPIC", "-pthread", "-I" + CUDA_INC, "-Wno-attributes",
                           "-fno-strict-aliasing", "-o", out, os.path.join(HC, "ba_dev_emu_host.cpp")])
    model = os.path.join(HC, "libba_host.so")
    compile_shared(["g++", "-O2", "-shared", "-fPIC", "-o", model, os.path.join(HC, "ba_host.cpp"), "-lm"])
    emu, host = ctypes.CDLL(out), ctypes.CDLL(model)
    emu.hc_ba_solve_dev.argtypes = [ctypes.c_void_p] * 2 + [ctypes.c_int] * 2 + [ctypes.c_void_p] * 3 + [ctypes.c_double] + [ctypes.c_int] * 6 + [ctypes.c_void_p]
    host.hc_bundle_adjust.argtypes = [ctypes.c_void_p] * 2 + [ctypes.c_int] * 2 + [ctypes.c_void_p] * 3 + [ctypes.c_double, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)

    def solve(obs, mask, K, R, t, prefit, n_ctas, n_threads, jac_mode=1, max_nfev=0):
        C = mask.shape[1]
        obs = np.ascontiguousarray(obs, np.float64); mask = np.ascontiguousarray(mask, np.uint8)
        Ks = np.ascontiguousarray(np.stack([K] * C)); R = np.ascontiguousarray(R.copy()); t = np.ascontiguousarray(t.copy())
        rep = np.zeros(13)
        assert emu.hc_ba_solve_dev(p(obs), p(mask), obs.shape[0], C, p(Ks), p(R), p(t), 1e-2, max_nfev, jac_mode, int(prefit), 50, n_ctas, n_threads, p(rep)) == 0
        keys = ["cost_initial", "cost_final", "optimality", "n_iterations", "n_fev", "status", "n_residuals", "prefit_cost_initial",
                "prefit_cost_final", "prefit_iterations", "smem", "n_tr_solves", "n_tr_newton"]
        return R, t, dict(zip(keys, rep))

    def model_solve(obs, mask, K, R, t, jac_mode=1):
        C = mask.shape[1]
        obs = np.ascontiguousarray(obs, np.float64); mask = np.ascontiguousarray(mask, np.uint8)
        Ks = np.ascontiguousarray(np.stack([K] * C)); R = np.ascontiguousarray(R.copy()); t = np.ascontiguousarray(t.copy())
        rep = np.zeros(7)
        assert host.hc_bundle_adjust(p(obs), p(mask), obs.shape[0], C, p(Ks), p(R), p(t), 1e-2, 0, p(rep), jac_mode) == 0
        return R, t, dict(zip(["cost_initial", "cost_final", "optimality", "n_iterations", "n_fev", "status", "n_jev"], rep))
    return solve, model_solve


def test_ba_kernel_on_host_equals_the_host_stepped_model(ba_emu):
    """k_ba_solve without the prefit is scipy's trust-region iteration; its sub-problem runs on Cholesky factors of
    A + alpha I where the host-stepped model (trf_core.h, itself checked against scipy) uses an eigen-decomposition.
    Several CTAs of real threads: same iterations, evaluations, status, cost and poses."""
    solve, model_solve = ba_emu
    z = np.load(os.path.join(ROOT, "tests", "golden", "ba_c4.npz"))
    Rm, tm, rm = model_solve(z["obs"], z["mask"], z["K"], z["R_start"], z["t_start"])
    for n_ctas, n_threads in ((1, 64), (3, 64)):
        R, t, r = solve(z["obs"], z["mask"], z["K"], z["R_start"], z["t_start"], False, n_ctas, n_threads)
        assert (r["n_iterations"], r["n_fev"], r["status"]) == (rm["n_iterations"], rm["n_fev"], rm["status"])
        assert abs(r["cost_final"] - rm["cost_final"]) <= 1e-9 * rm["cost_final"] and abs(r["cost_initial"] - float(z["cost0"])) < 1e-6 * float(z["cost0"])
        assert np.abs(R - Rm).max() < 1e-10 and np.abs(t - tm).max() < 1e-10
        assert r["n_residuals"] == z["mask"].shape[0]


def test_ba_kernel_on_host_with_prefit_beats_the_reference(ba_emu):
    """The default path (Levenberg-Marquardt prefit with the tile-wise Schur complement, then the polish) ends below
    the robust cost the real reference reaches from the same start (golden ba_c4), for any grid shape, and a
    different grid shape changes only the rounding of the sums."""
    solve, _ = ba_emu
    z = np.load(os.path.join(ROOT, "tests", "golden", "ba_c4.npz"))
    R1, t1, r1 = solve(z["obs"], z["mask"], z["K"], z["R_start"], z["t_start"], True, 3, 64)
    R2, t2, r2 = solve(z["obs"], z["mask"], z["K"], z["R_start"], z["t_start"], True, 2, 32)
    assert r1["cost_final"] <= float(z["costf"]) and r1["prefit_cost_final"] < 1e-3 * r1["prefit_cost_initial"]
    assert r1["status"] in (1, 2, 3, 4) and r1["smem"] < 227 * 1024
    assert abs(r1["cost_final"] - r2["cost_final"]) < 1e-6 and np.abs(R1 - R2).max() < 1e-7 and np.abs(t1 - t2).max() < 1e-7
    assert np.allclose(R1[0], np.eye(3)) and np.allclose(t1[0], 0)


def test_blob_device_code_reproduces_retr_tree_on_blobs_with_holes(blob_emu):
    """cv.findContours(RETR_TREE) (helpers.py:147) emits a contour per hole, takes the outer contour's moments over the
    FILLED blob and orders the contours along its hierarchy.  The one-warp path hands an image whose Euler numbers show
    a hole to the full-size reduction, which runs the RETR_TREE slow path (csrc/blob_holes.cuh): the emitted points
    -- count, values and order -- equal cv2's on random images with rings, frames, porous patches, blobs inside holes,
    rings inside rings, holes touching diagonally, 1-px walls, blobs across the 16-px segment boundaries and at the
    image border; no flag is left.  A holed blob too large for the slow path's window keeps MOCAP_F_HOLES."""
    import cv2
    rng = np.random.default_rng(31)
    H, W = 96, 128

    def reference(img):
        contours, hier = cv2.findContours((img > 51).astype(np.uint8), cv2.RETR_TREE, cv2.CHAIN_APPROX_SIMPLE)
        out = []
        for cnt in contours:
            m = cv2.moments(cnt)
            if m["m00"] != 0:
                out.append([int(m["m10"] / m["m00"]), int(m["m01"] / m["m00"])])
        has_hole = hier is not None and any(h[3] >= 0 for h in hier[0])
        return out, has_hole
    seen = {True: 0, False: 0}
    for trial in range(50):
        img = np.zeros((H, W), np.uint8)
        for _ in range(rng.integers(1, 7)):
            cx, cy = int(rng.integers(0, W)), int(rng.integers(0, H))
            kind = rng.integers(0, 6)
            if kind == 0:
                cv2.circle(img, (cx, cy), int(rng.integers(2, 10)), 255, int(rng.integers(1, 3)))          # ring
            elif kind == 1:
                cv2.circle(img, (cx, cy), int(rng.integers(1, 7)), 255, -1)                                # disc
            elif kind == 2:
                w, h = int(rng.integers(3, 24)), int(rng.integers(3, 12))
                cv2.rectangle(img, (cx, cy), (cx + w, cy + h), 255, 1)                                     # frame (may cross segments)
                if rng.integers(0, 2):
                    cv2.circle(img, (cx + w // 2, cy + h // 2), 1, 255, -1)                                # blob inside the hole
            elif kind == 3:
                m = (rng.uniform(size=(9, 14)) < 0.72).astype(np.uint8) * 255                              # porous patch
                y0, x0 = min(cy, H - 9), min(cx, W - 14)
                img[y0:y0 + 9, x0:x0 + 14] = np.maximum(img[y0:y0 + 9, x0:x0 + 14], m)
            elif kind == 4:
                cv2.circle(img, (cx, cy), int(rng.integers(6, 12)), 255, 1)                                # ring inside a ring
                cv2.circle(img, (cx, cy), int(rng.integers(2, 4)), 255, 1)
            else:
                img[max(cy - 2, 0):cy + 3, max(cx - 2, 0):cx + 3] = 255
                img[cy, cx] = 0 if rng.integers(0, 2) else 255                                            # 1-px hole
        ref, has_hole = reference(img)
        seen[has_hole] += 1
        for force_cta in (0, 1):
            d = blob_emu(img, force_cta=force_cta, seed=trial)
            assert d["flags"] == 0 and d["xy"].tolist() == ref, (trial, force_cta, d["flags"])
            if has_hole:
                assert d["path"] == 2                    # the slow path lives in the full-size reduction
    assert seen[True] >= 15                           # (solid-only images are what every other blob test covers)
    big = np.zeros((H, W), np.uint8)
    cv2.circle(big, (64, 48), 40, 255, 2)                # an 84-px ring: wider than the 62-px window
    d = blob_emu(big)
    assert d["flags"] == 32 and d["n"] == 1


def test_single_pass_kernel_on_host_three_channel_layout(fused_emu):
    """The H x W x 3 interleaved layout (helpers.py:143-145) through the single-pass kernel: a 16-pixel segment is three
    streamed words, the first word of a segment that passes the byte test computes the grey mask (cv2's 8-bit
    RGB2GRAY), later words of the same segment stand down.  Checked against cv2 on coloured frames (blobs whose
    brightest CHANNEL exceeds the threshold while the grey value does not, blobs across word and segment borders)."""
    import cv2
    rng = np.random.default_rng(8)
    B, C, H, W = 3, 2, 48, 96
    frames = rng.integers(0, 45, size=(B, C, H, W, 3), dtype=np.uint8)
    for b in range(B):
        for c in range(C):
            for _ in range(6):
                x, y = int(rng.integers(2, W - 8)), int(rng.integers(2, H - 6))
                colour = rng.integers(30, 256, size=3)
                if rng.integers(0, 3) == 0:
                    colour = np.array([0, 0, 255]) if rng.integers(0, 2) else np.array([250, 20, 20])     # one bright channel only
                frames[b, c, y:y + int(rng.integers(2, 5)), x:x + int(rng.integers(2, 7))] = colour
    K = np.array([[60.0, 0, 48], [0, 60.0, 24], [0, 0, 1]])
    R = np.stack([np.eye(3)] * C); t = np.array([[0.0, 0, 0], [-0.3, 0, 0]])
    d = fused_emu(frames, K, R, t, n_warps=4, runs=2)
    assert d["dirty_scratch"] == 0 and d["deferred_images"] == []
    some = 0
    for b in range(B):
        for c in range(C):
            grey = cv2.cvtColor(frames[b, c], cv2.COLOR_RGB2GRAY)
            contours, _ = cv2.findContours((grey > 51).astype(np.uint8), cv2.RETR_TREE, cv2.CHAIN_APPROX_SIMPLE)
            ref = []
            for cnt in contours:
                m = cv2.moments(cnt)
                if m["m00"] != 0:
                    ref.append([int(m["m10"] / m["m00"]), int(m["m01"] / m["m00"])])
            k = d["blob_n"][b, c]
            assert k == len(ref) and np.array_equal(d["blob_xy"][b, c, :k], np.array(ref, np.int32).reshape(k, 2)), (b, c)
            some += k
    assert some >= 10
