"""GPU parity tests of the surfel rasteriser's backward on each of its four routes, against the CPU oracle.

ga_raster_backward_ex picks one of four routes, depending on the forward's list_k and on the scratch buffer it is
given:
  R1  split kernels (A: per-pixel records, B: per-instance reduction) walking the forward's per-pixel lists (list_k > 0)
  R2  the same split kernels recomputing every (pixel, surfel) pair (list_k == 0)
  R3  the fused shared-memory kernel, chosen on the host: the scratch holds little more than the accumulators
  R4  the same fused kernel, chosen on the device: the scratch holds record lists, but fewer than the scene needs
Every test below forces a route through the C ABI with a chosen scratch size, proves which route ran with
ga_raster_backward_records (the record total against the capacity), and compares the gradient with the sum of the
oracle's per-view backward.  Bar: rel-L2 <= 1e-3 per gradient group, as in test_raster_gpu.py.

The scenes cover what the headline workload does not: image sizes that are not multiples of the 16-pixel tile, a
single surfel, a batch of two different scenes (the per-surfel backward sums views per batch item), surfels culled
in every view, a tile above the shared-memory sort limit, and a scene whose record total exceeds 2^32.
"""
import ctypes as C
import time
import zlib

import numpy as np
import pytest
import torch

from tests.helpers import cameras, oracle_view, rel_l2, scene

pytestmark = pytest.mark.gpu

TOL = 1e-3
GRAD_COLS = [("means3D", slice(0, 3)), ("opacity", slice(3, 4)), ("scales", slice(4, 6)),
             ("rotations", slice(6, 10)), ("colors", slice(10, 13))]
SATURATED = 0xffffffff

# (route, forward list_k)
ROUTES = [("R1", 32), ("R2", 0), ("R3", 0), ("R4", 0), ("R4", 32)]
ROUTE_IDS = ["R1-lists", "R2-recompute", "R3-fused-host", "R4-fused-device-k0", "R4-fused-device-k32"]


# ---------------------------------------------------------------------------------------------------------------
# scenes
# ---------------------------------------------------------------------------------------------------------------
def _look(vs):
    """Camera axes in world coordinates (right, down, forward) of a row-vector view matrix."""
    return vs[:3, 0].astype(np.float64), vs[:3, 1].astype(np.float64), vs[:3, 2].astype(np.float64)


def _quat_from_rotmat(R):
    """(w, x, y, z) of a proper rotation matrix (the inverse of the rasteriser's quat_to_rotmat)."""
    w = np.sqrt(max(0.0, 1.0 + R[0, 0] + R[1, 1] + R[2, 2])) / 2.0
    x = np.copysign(np.sqrt(max(0.0, 1.0 + R[0, 0] - R[1, 1] - R[2, 2])) / 2.0, R[2, 1] - R[1, 2])
    y = np.copysign(np.sqrt(max(0.0, 1.0 - R[0, 0] + R[1, 1] - R[2, 2])) / 2.0, R[0, 2] - R[2, 0])
    z = np.copysign(np.sqrt(max(0.0, 1.0 - R[0, 0] - R[1, 1] + R[2, 2])) / 2.0, R[1, 0] - R[0, 1])
    return np.array([w, x, y, z])


def _facing_surfels(P, vs, seed, scale, opacity, depth_spread):
    """P surfels at the image centre, parallel to the image plane, spread in depth along the optical axis."""
    rng = np.random.default_rng(seed)
    right, down, fwd = _look(vs)
    q = _quat_from_rotmat(np.stack([right, down, fwd], 1))
    g = np.zeros((P, 13), np.float32)
    g[:, 0:3] = (fwd[None] * rng.uniform(-depth_spread, depth_spread, (P, 1))
                 + right[None] * rng.uniform(-0.01, 0.01, (P, 1)) + down[None] * rng.uniform(-0.01, 0.01, (P, 1)))
    g[:, 3] = rng.uniform(*opacity, P)
    g[:, 4:6] = rng.uniform(*scale, (P, 2))
    g[:, 6:10] = q[None]
    g[:, 10:13] = rng.uniform(0.0, 1.0, (P, 3))
    return g


def _make_scene(name):
    sm, B = 1.0, 1
    if name == "ragged_250x300":
        P, H, W, V = 3000, 250, 300, 2
        g = scene(P, 90, 8.0)[None]
    elif name == "ragged_33x47":
        P, H, W, V = 400, 33, 47, 1                    # 3 x 2 tiles, 5 of the 6 partial
        g = scene(P, 91, 20.0)[None]
    elif name == "tiny_17x17":
        # one surfel covering the whole 17 x 17 image: 2 x 2 tiles, three of them partial
        P, H, W, V = 1, 17, 17, 1
        vs, _, _, _ = cameras(1, start=92)
        g = _facing_surfels(1, vs[0], 92, (0.3, 0.3), (0.8, 0.8), 0.0)[None]
    elif name == "batch2_ragged":
        P, H, W, V, B = 1500, 90, 70, 3, 2
        g = np.stack([scene(P, 93, 6.0), scene(P, 94, 3.0)])
    elif name == "culled_lowopacity_sm1.7":
        P, H, W, V = 2000, 100, 84, 2
        sm = 1.7
        g = scene(P, 95, 10.0)
        g[::3, 3] = 0.001                               # below 1/255: binned, never contributes
        g[1::20, 0:3] = 100.0                           # behind every camera
        g[11::20, 0:3] = np.array([0.0, 0.0, 5.0], np.float32)       # in front, far outside the frustum
        g = g[None]
    elif name == "dense_32x32":
        # the scene of test_sort_fallback_large_tile: tiles above 4096 instances
        P, H, W, V = 6000, 32, 32, 1
        g = scene(P, 7, 1.0)
        g[:, 0:3] *= 0.02
        g = g[None]
    else:
        raise KeyError(name)
    start = {"tiny_17x17": 92}.get(name, 0)
    vs, ps, _, _ = cameras(B * V, start=start)
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    gc = rng.standard_normal((B * V, 3, H, W)).astype(np.float32)
    ga = rng.standard_normal((B * V, 7, H, W)).astype(np.float32)
    return dict(name=name, g=np.ascontiguousarray(g, dtype=np.float32), vs=vs, ps=ps, bg=[1.0, 0.5, 0.2], H=H, W=W,
                B=B, V=V, P=P, sm=sm, gc=gc, ga=ga)


SCENES = ["ragged_250x300", "ragged_33x47", "tiny_17x17", "batch2_ragged", "culled_lowopacity_sm1.7", "dense_32x32"]
_SCENE_CACHE, _ORACLE_CACHE = {}, {}


@pytest.fixture(params=SCENES)
def sc(request):
    name = request.param
    if name not in _SCENE_CACHE:
        _SCENE_CACHE[name] = _make_scene(name)
    return _SCENE_CACHE[name]


def _oracle_grads(sc):
    """[B, P, 13] float64: per batch item, the oracle's backward summed over that item's views."""
    if sc["name"] in _ORACLE_CACHE:
        return _ORACLE_CACHE[sc["name"]]
    want = _oracle_grad_sum(sc["g"], sc["vs"], sc["ps"], sc["bg"], sc["H"], sc["W"], sc["gc"], sc["ga"],
                            sc["B"], sc["V"], sc["sm"])
    _ORACLE_CACHE[sc["name"]] = want
    return want


def _oracle_grad_sum(g, vs, ps, bg, H, W, gc, ga, B, V, sm=1.0):
    from oracle import surfel_oracle as so
    P = g.shape[1]
    want = np.zeros((B, P, 13))
    for b in range(B):
        for v in range(V):
            nv = b * V + v
            o = oracle_view(g[b], vs[nv], ps[nv], bg, H, W, scale_modifier=sm)
            r = so.rasterize_backward(o, gc[nv], ga[nv])
            want[b, :, 0:3] += r["means3D"]; want[b, :, 3:4] += r["opacities"]; want[b, :, 4:6] += r["scales"]
            want[b, :, 6:10] += r["rotations"]; want[b, :, 10:13] += r["colors"]
    return want


def _check_grads(got, want, tag, tol=TOL):
    for b in range(want.shape[0]):
        for name, sl in GRAD_COLS:
            r = rel_l2(got[b][:, sl], want[b][:, sl])
            assert r <= tol, (tag, "batch item %d" % b, name, r)


# ---------------------------------------------------------------------------------------------------------------
# the C ABI with a chosen scratch size
# ---------------------------------------------------------------------------------------------------------------
def _ptr(t):
    return C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _align(x):
    return (x + 255) // 256 * 256


def _acc_bytes(B, P, V):
    return _align(B * V * P * 18 * 4)


def _fixed_bytes(B, P, V):
    """Scratch in front of the record lists: accumulators | tile slice starts (255 x 255 per image) | flag."""
    return _acc_bytes(B, P, V) + _align((B * V * 255 * 255 + 1) * 4) + 256


def _route_scratch_bytes(route, B, P, V):
    from gaussiananything_b200 import _lib
    if route in ("R1", "R2"):
        return int(_lib.lib().ga_raster_backward_scratch_bytes(B, P, V))
    if route == "R3":
        return _acc_bytes(B, P, V)
    return _fixed_bytes(B, P, V) + 4096 + 16           # the smallest record buffer there is: 257 records


def _forward(sc, list_k):
    from gaussiananything_b200 import raster
    dev = torch.device("cuda:0")
    B, V, H, W = sc["B"], sc["V"], sc["H"], sc["W"]
    g13 = torch.tensor(sc["g"], device=dev)
    vm = torch.tensor(sc["vs"], device=dev).reshape(B, V, 4, 4)
    pm = torch.tensor(sc["ps"], device=dev).reshape(B, V, 4, 4)
    bg = torch.tensor(sc["bg"], dtype=torch.float32, device=dev)
    return raster.forward_raw(g13, vm, pm, bg, H, W, sc["sm"], list_k=list_k)


def _records(st, scratch, nbytes):
    """(record total, capacity) from ga_raster_backward_records."""
    from gaussiananything_b200 import _lib
    B, P, V, H, W = st["dims"]
    total, cap = C.c_uint64(0), C.c_uint64(0)
    rc = _lib.lib().ga_raster_backward_records(B, P, V, H, W, _ptr(st["ws"]), st["L"].total_bytes, st["max_instances"],
                                               st["list_k"], _ptr(scratch), nbytes, C.byref(total), C.byref(cap),
                                               _stream())
    _lib.check(rc, "ga_raster_backward_records")
    return total.value, cap.value


def _backward(st, gc, ga, scratch, nbytes):
    from gaussiananything_b200 import _lib
    B, P, V, H, W = st["dims"]
    dev = st["ws"].device
    dgc = torch.tensor(gc, device=dev).reshape(B, V, 3, H, W).contiguous()
    dga = torch.tensor(ga, device=dev).reshape(B, V, 7, H, W).contiguous()
    grad = torch.full((B, P, 13), float("nan"), device=dev)
    rc = _lib.lib().ga_raster_backward_ex(
        _ptr(st["gauss13"]), B, P, V, _ptr(st["viewmats"]), _ptr(st["projmats"]), _ptr(st["bg"]), H, W,
        st["scale_modifier"], _ptr(st["radii"]), _ptr(dgc), _ptr(dga), _ptr(st["ws"]), st["L"].total_bytes,
        st["max_instances"], st["list_k"], _ptr(scratch), nbytes, _ptr(grad), _stream())
    _lib.check(rc, "ga_raster_backward_ex")
    torch.cuda.synchronize()
    return grad.cpu().numpy().astype(np.float64)


def _run_route(sc, route, list_k):
    """Forward with list_k, backward forced onto `route`; asserts that the route is the one that ran."""
    B, P, V = sc["B"], sc["P"], sc["V"]
    c, a, radii, st = _forward(sc, list_k)
    nbytes = _route_scratch_bytes(route, B, P, V)
    boundary = _fixed_bytes(B, P, V) + 4096            # the largest scratch that still gets the fused kernel on the host
    scratch = torch.empty(max(nbytes, boundary + 16), dtype=torch.uint8, device=st["ws"].device)
    if route in ("R1", "R2"):
        # ga_raster_backward_scratch_bytes budgets 64 records per surfel and view, which large splats exceed (and a
        # budget under 4 KB enables no lists at all): size the buffer from the probe, as a caller would
        need = _records(st, scratch, nbytes)[0]
        nbytes = max(nbytes, boundary + 16 * (need + 1))
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=st["ws"].device)
    if route == "R3":
        assert nbytes <= boundary
        assert _records(st, scratch, boundary)[1] == 0, "a scratch of accumulators + tile table + 4 KB enables lists"
        assert _records(st, scratch, boundary + 16)[1] == 257
    else:
        total, cap = _records(st, scratch, nbytes)
        if route == "R4":
            assert cap == 257 and total > cap, ("R4 not forced", total, cap)
        else:
            assert 0 < total <= cap, (route, "split kernels not chosen", total, cap)
    grad = _backward(st, sc["gc"], sc["ga"], scratch, nbytes)
    return grad, st, radii


# ---------------------------------------------------------------------------------------------------------------
# every route on every scene against the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("route,list_k", ROUTES, ids=ROUTE_IDS)
def test_backward_route_vs_oracle(sc, route, list_k):
    from gaussiananything_b200 import raster
    grad, st, radii = _run_route(sc, route, list_k)
    assert np.isfinite(grad).all()
    _check_grads(grad, _oracle_grads(sc), "%s/%s k=%d" % (sc["name"], route, list_k))
    B, P, V, H, W = st["dims"]
    if sc["name"].startswith("culled"):
        # a surfel culled in every view of its batch item receives no gradient at all: exact zeros, not small values
        dead = (radii.cpu().numpy() == 0).all(axis=1)              # [B, P]
        assert dead.sum() >= 0.09 * P, dead.sum()
        assert (grad[dead] == 0.0).all(), np.abs(grad[dead]).max()
    if sc["name"] == "dense_32x32":
        wsv = raster.workspace_views(st["ws"], st["L"], B, P, V, H, W, st["max_instances"])
        assert int(wsv["status"][2]) >= 1, "expected a tile sorted in global memory (> 4096 instances)"
        T = ((W + 15) // 16) * ((H + 15) // 16)
        counts = np.diff(wsv["tile_start"].cpu().numpy().astype(np.int64))
        assert counts.max() > 4096
        if list_k:
            L = st["L"]
            flags = st["ws"][L.tile_flag:L.tile_flag + 4 * B * V * T].view(torch.int32)
            assert int(flags.sum()) >= 1, "expected a tile whose per-pixel lists overflowed list_k"


def test_fused_routes_agree(sc):
    """R3 and R4 run the same fused kernel (R4 after the split kernels found the buffer too small and exited): the
    gradients differ only by the order of float atomics, whether or not the forward recorded lists."""
    g3 = _run_route(sc, "R3", 0)[0]
    for list_k in (0, 32):
        g4 = _run_route(sc, "R4", list_k)[0]
        _check_grads(g4, g3, "%s R4 k=%d vs R3" % (sc["name"], list_k), tol=1e-5)


def test_batch2_autograd_per_item():
    """rasterize_surfels_batched with B = 2: each batch item's gradient is the sum over its own views only."""
    from gaussiananything_b200 import raster
    sc = _SCENE_CACHE.setdefault("batch2_ragged", _make_scene("batch2_ragged"))
    B, V, P, H, W = sc["B"], sc["V"], sc["P"], sc["H"], sc["W"]
    dev = torch.device("cuda:0")
    g13 = torch.tensor(sc["g"], device=dev).requires_grad_(True)
    vm = torch.tensor(sc["vs"], device=dev).reshape(B, V, 4, 4)
    pm = torch.tensor(sc["ps"], device=dev).reshape(B, V, 4, 4)
    color, allmap, radii = raster.rasterize_surfels_batched(g13, vm, pm, torch.tensor(sc["bg"], device=dev), H, W, 1.0)
    loss = ((color * torch.tensor(sc["gc"], device=dev).reshape(B, V, 3, H, W)).sum()
            + (allmap * torch.tensor(sc["ga"], device=dev).reshape(B, V, 7, H, W)).sum())
    loss.backward()
    got = g13.grad.cpu().numpy().astype(np.float64)
    want = _oracle_grads(sc)
    _check_grads(got, want, "autograd B=2")
    # the two items really differ: a kernel that mixed them up could not pass the check above by accident
    assert rel_l2(want[0], want[1]) > 0.5


# ---------------------------------------------------------------------------------------------------------------
# the record total against a host replica
# ---------------------------------------------------------------------------------------------------------------
def _host_record_areas(wsv, NV, H, W, tiles=None):
    """Yields (view, tile, int64 areas of the tile's instances): the pixels of each instance's cull box inside its
    tile, as raster_render.cu's clipped_box_area computes them (float32 box and tile bounds, floor / ceil to pixel
    centres).  An empty cull box (a surfel too transparent to reach alpha 1/255 anywhere) covers no pixel."""
    gx, gy = (W + 15) // 16, (H + 15) // 16
    T = gx * gy
    ts = wsv["tile_start"].cpu().numpy().astype(np.int64)
    ids = wsv["ids"].cpu().numpy().view(np.uint32)
    rec = wsv["rec"].cpu().numpy()
    for v in range(NV):
        for t in (range(T) if tiles is None else tiles):
            s, e = ts[v * T + t], ts[v * T + t + 1]
            bb = rec[v, ids[s:e], 16:20]
            ox, oy = np.float32((t % gx) * 16), np.float32((t // gx) * 16)
            x0, x1 = np.maximum(bb[:, 0], ox), np.minimum(bb[:, 1], ox + np.float32(15))
            y0, y1 = np.maximum(bb[:, 2], oy), np.minimum(bb[:, 3], oy + np.float32(15))
            ok = (x0 <= x1) & (y0 <= y1)
            x0, x1, y0, y1 = (np.where(ok, a, ox) for a in (x0, x1, y0, y1))
            wx = np.maximum(0, np.floor(x1).astype(np.int64) - np.ceil(x0).astype(np.int64) + 1)
            wy = np.maximum(0, np.floor(y1).astype(np.int64) - np.ceil(y0).astype(np.int64) + 1)
            yield v, t, np.where(ok, wx * wy, 0)


@pytest.mark.parametrize("name", ["c1_256", "culled_lowopacity_sm1.7"])
def test_record_total_matches_host_replica(name):
    """list_k = 0: the probe's record total == the sum over instances of the clipped cull-box area, in int64."""
    from gaussiananything_b200 import _lib, raster
    if name == "c1_256":
        P, H, W = 10000, 256, 256
        vs, ps, _, _ = cameras(1)
        sc = dict(name=name, g=scene(P, 0, 1.0)[None], vs=vs, ps=ps, bg=[1.0, 1.0, 1.0], H=H, W=W, B=1, V=1, P=P, sm=1.0)
    else:
        sc = _SCENE_CACHE.setdefault(name, _make_scene(name))
    B, V, P, H, W = sc["B"], sc["V"], sc["P"], sc["H"], sc["W"]
    c, a, radii, st = _forward(sc, 0)
    nbytes = int(_lib.lib().ga_raster_backward_scratch_bytes(B, P, V))
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=st["ws"].device)
    total, cap = _records(st, scratch, nbytes)
    wsv = raster.workspace_views(st["ws"], st["L"], B, P, V, H, W, st["max_instances"])
    want = sum(int(ar.sum()) for _, _, ar in _host_record_areas(wsv, B * V, H, W))
    assert want > 0
    assert total == want, (total, want)
    assert cap == (nbytes - _fixed_bytes(B, P, V)) // 16


def test_whole_image_record_total_saturates_and_falls_back():
    """65 560 surfels that each cover all 256 tiles of a 256 x 256 view: 16.8 M instances of 256 records each, a
    record total of 2^32 + 1 572 864.  The total must not wrap to 1 572 864 (which fits the default buffer and would
    send kernel A to wrapped offsets): it saturates at 2^32 - 1, above every capacity, so the fused kernel runs.  With
    list_k = 32 the forward counts only the chunk of 256 instances per tile it staged, 2^24 records: above the default
    capacity too, and within a buffer sized from the probe, where the split kernels run.  All match the oracle."""
    from gaussiananything_b200 import _lib, raster
    t0 = time.time()
    P, H, W = 65560, 256, 256
    vs, ps, _, _ = cameras(1)
    g = _facing_surfels(P, vs[0], 96, (0.8, 1.2), (0.03, 0.1), 0.3)
    rng = np.random.default_rng(96)
    sc = dict(name="whole_image", g=g[None], vs=vs, ps=ps, bg=[0.2, 0.3, 0.4], H=H, W=W, B=1, V=1, P=P, sm=1.0,
              gc=rng.standard_normal((1, 3, H, W)).astype(np.float32),
              ga=rng.standard_normal((1, 7, H, W)).astype(np.float32))
    c, a, radii, st = _forward(sc, 0)
    assert st["num_rendered"] == P * 256
    wsv = raster.workspace_views(st["ws"], st["L"], 1, P, 1, H, W, st["max_instances"])
    # precondition, from the host replica: every instance covers its whole tile
    for _, t, ar in _host_record_areas(wsv, 1, H, W):
        assert ar.size == P and (ar == 256).all(), (t, ar.size, int(ar.min()))
    assert P * 256 * 256 == 2 ** 32 + 1572864
    nbytes = int(_lib.lib().ga_raster_backward_scratch_bytes(1, P, 1))
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=st["ws"].device)
    total, cap = _records(st, scratch, nbytes)
    assert cap == P * 64
    assert total == SATURATED, ("record total", total, "capacity", cap)
    assert total > cap
    # only now, with the fallback decision known to be right, run the backward
    want = _oracle_grads(sc)
    got0 = _backward(st, sc["gc"], sc["ga"], scratch, nbytes)
    _check_grads(got0, want, "whole image, k=0 (fused kernel)")
    c, a, radii, st = _forward(sc, 32)
    total32, cap32 = _records(st, scratch, nbytes)
    assert total32 == 256 * 256 * 256 and total32 > cap32, (total32, cap32)
    got32 = _backward(st, sc["gc"], sc["ga"], scratch, nbytes)
    _check_grads(got32, want, "whole image, k=32 (fused kernel)")
    nbytes = _fixed_bytes(1, P, 1) + 4096 + 16 * total32
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=st["ws"].device)
    total32, cap32 = _records(st, scratch, nbytes)
    assert total32 <= cap32, (total32, cap32)
    got32 = _backward(st, sc["gc"], sc["ga"], scratch, nbytes)
    _check_grads(got32, want, "whole image, k=32 (split kernels, lists)")
    print("whole-image scene: %.1f s" % (time.time() - t0))
