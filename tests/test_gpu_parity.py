"""GPU parity tests: the CUDA library, called through its C ABI (vidu4d_b200.rasterizer._C -> ctypes ->
libsurfel_raster.so), against
  (1) the committed golden fixtures = outputs of the unmodified reference extension (tests/golden/),
  (2) the CPU oracle on seeded inputs at sizes it finishes in seconds,
  (3) digests of the reference extension's outputs at config C2 (100 K surfels, 512^2; tests/golden/ref_*.npz),
  (4) size-independent properties at BASELINE.json's full size (300 K surfels, 512^2).
Bar: integer/index work bit-exact; float buffers and gradients within 1e-4 relative (north_star), with the
tolerance written at each assert.  Nothing here reads /root/reference.
"""
import os

import numpy as np
import pytest
import torch

from .conftest import GOLDEN_CASES, load_golden

pytestmark = pytest.mark.gpu
TOL = 1e-4
GRADS = ("dL_dmeans2D", "dL_dcolors", "dL_dopacity", "dL_dmeans3D", "dL_dtransMat", "dL_dsh", "dL_dscales", "dL_drotations")


@pytest.fixture(scope="module")
def dev(built):
    from vidu4d_b200 import _capi
    _capi.load()
    return torch.device("cuda:0")


def _run_ours(inp, dev, debug=False, with_grads=True):
    """inp: dict of numpy arrays as in the golden files (in_* keys without prefix)."""
    from vidu4d_b200 import debug as dbg, rasterizer as R
    P, W, H, deg, pre = [int(v) for v in inp["meta"]]
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in inp.items() if k != "meta"}
    e = torch.empty((0,), device=dev)
    shs = e if pre else t["shs"]
    col = t["colors_precomp"] if pre else e
    tx, ty = float(inp["tanfov"][0]), float(inp["tanfov"][1])
    out = R._C.rasterize_gaussians(t["bg"], t["means3D"], col, t["opacities"], t["scales"], t["rotations"], 1.0, e,
                                   t["viewmatrix"], t["projmatrix"], tx, ty, H, W, shs, deg, t["campos"], False, debug)
    nr, color, allmap, radii, gb, bb, ib = out
    res = dict(num_rendered=nr, color=color, allmap=allmap, radii=radii, bufs=(gb, bb, ib))
    res.update(dbg.decode(gb, bb, ib, P, W, H, nr))
    if with_grads:
        g = R._C.rasterize_gaussians_backward(t["bg"], t["means3D"], radii, col, t["scales"], t["rotations"], 1.0, e,
                                              t["viewmatrix"], t["projmatrix"], tx, ty, t["dL_dcolor"], t["dL_dallmap"], shs,
                                              deg, t["campos"], gb, nr, bb, ib, debug)
        res["grads"] = dict(zip(GRADS, g))
    return res


def _golden_inputs(g):
    return {k[3:]: v for k, v in g.items() if k.startswith("in_")}


def _np(x):
    return x.detach().cpu().numpy()


def _assert_n_contrib(mine, ref, ranges, W, H):
    """Plane 0 (last contributor) must match everywhere.  Plane 1 (median contributor) is compared only in tiles
    whose instance list is non-empty: for an empty tile the reference stores `(uint32_t)(-1.0f)`
    (forward.cu:326,452) -- undefined behaviour in C++, and its sm_100a build leaves garbage there (never read by
    its backward, which does nothing for an empty range)."""
    mine = np.asarray(mine).astype(np.int64) & 0xFFFFFFFF
    ref = np.asarray(ref).astype(np.int64) & 0xFFFFFFFF
    np.testing.assert_array_equal(mine[0], ref[0])
    tx = (W + 15) // 16
    ys, xs = np.mgrid[0:H, 0:W]
    t = (ys // 16) * tx + xs // 16
    rg = np.asarray(ranges).astype(np.int64)
    nonempty = (rg[:, 1] - rg[:, 0])[t] > 0
    np.testing.assert_array_equal(mine[1][nonempty], ref[1][nonempty])
    assert (mine[1][~nonempty] == 0).all()


def _assert_close_robust(mine, ref, tol, what, outlier_frac=2e-4, outlier_tol=5e-2):
    """CPU-oracle comparisons only: libm expf / 1/sqrtf differ from MUFU.EX2 / MUFU.RSQ in the last ulp, so a
    (pixel, surfel) pair sitting exactly on a discrete threshold (alpha = 1/255, T = 1e-4, rho3d = rho2d) can fall
    on the other side.  Require `tol` for all but a vanishing fraction of elements and a loose bound on those."""
    mine = np.asarray(mine, np.float64).reshape(-1)
    ref = np.asarray(ref, np.float64).reshape(-1)
    scale = np.abs(ref).max() + 1e-30
    err = np.abs(mine - ref) / scale
    bad = err > tol
    assert bad.mean() <= outlier_frac, (what, bad.mean(), err.max())
    assert err.max() <= outlier_tol, (what, err.max())


# ----------------------------------------------------------------------------------------------- (1) goldens
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_against_reference_golden(name, dev):
    g = load_golden(name)
    r = _run_ours(_golden_inputs(g), dev, debug=True)
    R = int(g["ref_num_rendered"][0])
    # ---- tile assignment / sort: bit-exact
    assert r["num_rendered"] == R
    np.testing.assert_array_equal(_np(r["radii"]), g["ref_radii"])
    np.testing.assert_array_equal(_np(r["tiles_touched"]), g["ref_geom_tiles_touched"])
    vis = g["ref_radii"] > 0
    np.testing.assert_array_equal(_np(r["depths"])[vis].view(np.int32), g["ref_geom_depths"][vis].view(np.int32))
    np.testing.assert_array_equal(_np(r["keys"]), g["ref_bin_keys"])
    np.testing.assert_array_equal(_np(r["point_list"]), g["ref_bin_point_list"])
    np.testing.assert_array_equal(_np(r["ranges"]), g["ref_img_ranges"])
    P_, W_, H_ = [int(v) for v in g["in_meta"][:3]]
    _assert_n_contrib(_np(r["n_contrib"]), g["ref_img_n_contrib"], g["ref_img_ranges"], W_, H_)
    # ---- per-surfel projected geometry: same FMA map as the reference build => identical bits
    rec = _np(r["surfel_rec"])
    np.testing.assert_array_equal(rec[vis][:, 0:9].view(np.int32), g["ref_geom_transMat"][vis].view(np.int32))
    np.testing.assert_array_equal(rec[vis][:, 9:11].view(np.int32), g["ref_geom_means2D"][vis].view(np.int32))
    # ---- rendered buffers: tolerance 1e-4 relative (in fact bit-identical on this hardware)
    for mine, ref in ((_np(r["color"]), g["ref_color"]), (_np(r["allmap"]), g["ref_allmap"]),
                      (_np(r["final_T"]), g["ref_img_final_T"])):
        assert np.abs(mine - ref).max() <= TOL * max(1.0, np.abs(ref).max())
    assert np.array_equal(_np(r["color"]), g["ref_color"]), "colour planes are expected to be bit-identical to the reference"
    # ---- gradients: 1e-4 of the tensor's max magnitude (the reference itself is atomics-ordered)
    for k in GRADS:
        ref = g["ref_grad_" + k]
        if ref.size == 0:
            continue
        mine = _np(r["grads"][k]).reshape(ref.shape)
        assert np.abs(mine - ref).max() <= TOL * (np.abs(ref).max() + 1e-30), k


# ----------------------------------------------------------------------------------------------- (2) CPU oracle
@pytest.mark.parametrize("P,W,H,seed,rigid", [(20000, 256, 256, 21, False), (8000, 200, 120, 22, True)])
def test_against_cpu_oracle(P, W, H, seed, rigid, dev):
    from oracle import surfel_oracle as so
    from tests.golden.make_golden import build_case
    inp = build_case(P, W, H, seed, rigid=rigid, bg=(0.3, 0.1, 0.6))
    r = _run_ours(inp, dev)
    st = so.forward(inp["means3D"], inp["opacities"], inp["scales"], inp["rotations"], shs=inp["shs"], sh_degree=3, W=W, H=H,
                    tanfovx=0.5, tanfovy=0.5, bg=inp["bg"], viewmatrix=inp["viewmatrix"], projmatrix=inp["projmatrix"],
                    campos=inp["campos"])
    og = so.backward(st, inp["dL_dcolor"], inp["dL_dallmap"])
    # index work: exact (the oracle reproduces the GPU's arithmetic except MUFU.RSQ/EX2; a knife-edge surfel
    # could legitimately differ -- none does for these seeds)
    assert r["num_rendered"] == st.num_rendered
    np.testing.assert_array_equal(_np(r["radii"]), st.radii)
    np.testing.assert_array_equal(_np(r["keys"]).astype(np.uint64), st.keys)
    np.testing.assert_array_equal(_np(r["point_list"]).astype(np.uint32), st.point_list)
    np.testing.assert_array_equal(_np(r["ranges"]).astype(np.uint32), st.ranges)
    _assert_close_robust(_np(r["color"]), st.color, TOL, "color")
    for i in range(8):
        _assert_close_robust(_np(r["allmap"][i]), st.allmap[i], TOL, f"allmap[{i}]")
    for k in GRADS:
        _assert_close_robust(_np(r["grads"][k]), og[k], TOL, k)


# ----------------------------------------------------------------------------------------------- (3) reference digests
def _assert_index_work_matches_digest(r, g):
    """Instance count, radii, sorted keys / surfel ids, tile ranges and both contributor planes bit-exact against a
    digest of tests/golden/make_golden.py (the median plane is zero in tiles with an empty list)."""
    from tests.golden.make_golden import array_sha
    assert r["num_rendered"] == int(g["num_rendered"][0])
    for a, key in ((r["radii"], "radii"), (r["keys"], "keys"), (r["point_list"], "point_list"), (r["ranges"], "ranges")):
        assert np.array_equal(array_sha(_np(a)), g["sha_" + key]), f"{key} differ from the reference's"
    nc = _np(r["n_contrib"]).astype(np.int64) & 0xFFFFFFFF
    assert np.array_equal(array_sha(nc[0]), g["sha_n_contrib0"]), "last-contributor plane differs from the reference's"
    assert np.array_equal(array_sha(nc[1]), g["sha_n_contrib1"]), "median-contributor plane differs from the reference's"


def _assert_close_to_digest(mine, idx, ref_at_idx, ref_absmax, tol, what, axis=-1):
    """Within `tol` of the reference at the digest's sample `idx` (along `axis`), and in the largest magnitude over the
    whole array, which a difference beyond `tol` at the element where it is reached would change."""
    err = np.abs(np.take(mine, idx, axis=axis) - ref_at_idx).max()
    assert err <= tol, (what, float(err), tol)
    assert abs(float(np.abs(mine).max()) - float(ref_absmax)) <= tol, (what, "largest magnitude", float(np.abs(mine).max()), float(ref_absmax))


def _assert_grads_close_to_digest(r, g):
    """All eight gradient tensors within 1e-4 of the tensor's max magnitude."""
    for k in GRADS:
        shape = tuple(int(v) for v in g["shape_" + k])
        if np.prod(shape) == 0:
            continue
        _assert_close_to_digest(_np(r["grads"][k]).reshape(shape), g["surf"], g["grad_" + k], g["absmax_" + k],
                                TOL * (float(g["absmax_" + k]) + 1e-30), k, axis=0)


def test_against_live_reference_c2(dev):
    """Config C2 (100 K surfels, 512^2) against the digest of the reference's outputs (tests/golden/ref_c2_100k_512.npz)."""
    from tests.golden.make_golden import BIG_CASES, array_sha, inputs_sha
    g = load_golden("ref_c2_100k_512")
    inp = BIG_CASES["ref_c2_100k_512"]()
    assert np.array_equal(inputs_sha(inp), g["inputs_sha"]), "the seeded inputs differ from the ones the digest was made of"
    r = _run_ours(inp, dev)
    _assert_index_work_matches_digest(r, g)
    assert np.array_equal(array_sha(_np(r["color"])), g["sha_color"]), "colour planes are expected to be bit-identical to the reference"
    am, amax = _np(r["allmap"]), float(g["absmax_allmap"].max())
    _assert_close_to_digest(am.reshape(8, -1), g["pix"], g["allmap_at_pix"], amax, TOL * amax, "allmap")
    _assert_grads_close_to_digest(r, g)


# ----------------------------------------------------------------------------------------------- (4) full size
@pytest.fixture(scope="module")
def headline(dev):
    from tests.golden.make_golden import build_case
    inp = build_case(300_000, 512, 512, 41)
    return inp, _run_ours(inp, dev)


def test_full_size_structure(headline):
    inp, r = headline
    R = r["num_rendered"]
    keys = r["keys"]
    assert R == int(r["tiles_touched"].sum().item())
    assert bool((keys[1:] >= keys[:-1]).all()), "sorted by (tile, depth)"
    rg = r["ranges"].long()
    nz = rg[(rg[:, 1] - rg[:, 0]) > 0]
    assert int((nz[:, 1] - nz[:, 0]).sum().item()) == R and int(nz[0, 0]) == 0 and int(nz[-1, 1]) == R
    assert bool((nz[1:, 0] == nz[:-1, 1]).all()), "tile ranges tile [0, R) without gaps"
    # every surfel appears exactly tiles_touched times in the sorted list
    cnt = torch.bincount(r["point_list"].long(), minlength=300_000)
    assert torch.equal(cnt, r["tiles_touched"].long())
    # stable sort: equal keys keep emission order = ascending surfel id
    same = keys[1:] == keys[:-1]
    assert bool((r["point_list"][1:][same] > r["point_list"][:-1][same]).all())
    # alpha plane = 1 - final T, contributors bounded by the tile list length
    assert torch.equal(r["allmap"][1], 1.0 - r["final_T"][0])
    assert float(r["allmap"][1].min()) >= 0.0 and float(r["allmap"][1].max()) <= 1.0
    assert torch.isfinite(r["color"]).all() and torch.isfinite(r["allmap"]).all()
    assert bool((r["radii"] >= 0).all())
    for k in GRADS:
        assert torch.isfinite(r["grads"][k]).all(), k
    inv = r["radii"] == 0
    assert float(r["grads"]["dL_dmeans3D"][inv].abs().sum()) == 0.0


def test_full_size_forward_is_deterministic(headline, dev):
    inp, r = headline
    r2 = _run_ours(inp, dev, with_grads=False)
    assert torch.equal(r["color"], r2["color"]) and torch.equal(r["allmap"], r2["allmap"])
    assert torch.equal(r["keys"], r2["keys"]) and torch.equal(r["point_list"], r2["point_list"])


def test_full_size_backward_is_linear(headline, dev):
    """Backward is linear in (dL_dcolor, dL_dallmap): bwd(2a - 3b) == 2 bwd(a) - 3 bwd(b) up to fp32 summation."""
    from vidu4d_b200 import rasterizer as R
    inp, r = headline
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in inp.items() if k != "meta"}
    e = torch.empty((0,), device=dev)
    gb, bb, ib = r["bufs"]
    g = torch.Generator(device=dev).manual_seed(3)
    a = (torch.randn((3, 512, 512), device=dev, generator=g), torch.randn((8, 512, 512), device=dev, generator=g))
    b = (torch.randn((3, 512, 512), device=dev, generator=g), torch.randn((8, 512, 512), device=dev, generator=g))

    def bwd(dc, do):
        return R._C.rasterize_gaussians_backward(t["bg"], t["means3D"], r["radii"], e, t["scales"], t["rotations"], 1.0, e,
                                                 t["viewmatrix"], t["projmatrix"], 0.5, 0.5, dc, do, t["shs"], 3, t["campos"],
                                                 gb, r["num_rendered"], bb, ib, False)
    ga, gb_, gc = bwd(*a), bwd(*b), bwd(2 * a[0] - 3 * b[0], 2 * a[1] - 3 * b[1])
    for x, y, z, k in zip(ga, gb_, gc, GRADS):
        lin = 2 * x - 3 * y
        assert float((lin - z).abs().max()) <= 1e-4 * float(z.abs().max() + 1e-30), k


# ----------------------------------------------------------------------------------------------- API level
def _cloud(P, dev, seed=0):
    from vidu4d_b200.synthetic import SurfelCloud, object_scene
    return SurfelCloud(object_scene(P, seed=seed), dev)


def test_render_api_autograd_and_inplace_edit(dev):
    """render() returns the reference's dict; the caller edits `render` IN PLACE before backward
    (lab4d/nnutils/deformable_gaussian.py:188-190) -- must not trip autograd's version counter."""
    from vidu4d_b200.renderer import PipelineParams, make_camera, render
    cloud = _cloud(5000, dev, seed=3)
    cam = make_camera(128, 96, 2 * np.arctan(0.5), 2 * np.arctan(0.375), device=dev)
    bg = torch.zeros(3, device=dev)
    out = render(cam, cloud, PipelineParams(), bg)
    assert set(out) == {"render", "viewspace_points", "visibility_filter", "radii", "acc", "rend_normal", "rend_dist",
                        "surf_depth", "render_depth_median", "render_depth_expected", "surf_normal"}
    assert out["render"].shape == (3, 96, 128) and out["surf_depth"].shape == (3, 96, 128)
    learnable_bg = torch.full((3, 1, 1), 0.5, device=dev, requires_grad=True)
    out["render"][:3] = out["render"][:3] + (1 - out["acc"]) * learnable_bg
    loss = out["render"].mean() + 0.1 * out["rend_dist"].mean() + 0.1 * (out["rend_normal"] * out["surf_normal"]).sum(0).mean()
    loss.backward()
    for p in cloud.flat_params():
        assert p.grad is not None and torch.isfinite(p.grad).all() and float(p.grad.abs().sum()) > 0
    vp = out["viewspace_points"]
    assert vp.grad is not None and vp.grad.shape == (5000, 3) and float(vp.grad[:, 2].abs().sum()) == 0.0
    assert int(out["visibility_filter"].sum()) == int((out["radii"] > 0).sum()) > 0
    with pytest.raises(Exception, match="excatly one of either SHs or precomputed colors"):
        render(cam, cloud, PipelineParams(), bg, override_color=torch.rand(5000, 3, device=dev))


def test_nosync_mode_overflow_is_detected_and_recovered(dev):
    from vidu4d_b200 import _capi, rasterizer as R
    from tests.golden.make_golden import build_case
    inp = build_case(3000, 128, 128, 51)
    base = _run_ours(inp, dev, with_grads=False)
    key = (dev.index, 128, 128)
    try:
        R.set_sync_mode(False)
        R._cap_hint[key] = 64                       # force a capacity far below num_rendered
        bad = _run_ours(inp, dev, with_grads=False)
        assert bad["num_rendered"] == -1
        with pytest.raises(_capi.SurfelRasterError, match="overflow"):
            R.check_overflow()
        assert R._cap_hint[key] == base["num_rendered"]      # hint refreshed from the device word
        good = _run_ours(inp, dev, with_grads=False)           # same call now fits
        R.check_overflow()
        assert torch.equal(good["color"], base["color"])
    finally:
        R.set_sync_mode(True)
        R._pending.clear()
    # sync mode recovers transparently from a too-small hint
    R._cap_hint[key] = 64
    again = _run_ours(inp, dev, with_grads=False)
    assert again["num_rendered"] == base["num_rendered"] and torch.equal(again["color"], base["color"])


def test_empty_inputs_and_mark_visible(dev):
    from vidu4d_b200 import rasterizer as R
    e = torch.empty((0,), device=dev)
    z3 = torch.zeros((0, 3), device=dev)
    out = R._C.rasterize_gaussians(torch.ones(3, device=dev), z3, z3, torch.zeros((0, 1), device=dev),
                                   torch.zeros((0, 2), device=dev), torch.zeros((0, 4), device=dev), 1.0, e,
                                   torch.eye(4, device=dev), torch.eye(4, device=dev), 0.5, 0.5, 32, 48, e, 0,
                                   torch.zeros(3, device=dev), False, False)
    assert out[0] == 0 and out[1].shape == (3, 32, 48) and float(out[1].abs().sum()) == 0.0   # P == 0 -> zeros, not bg
    pts = torch.tensor([[0.0, 0.0, 0.1], [0.0, 0.0, 0.2], [0.0, 0.0, 0.21], [1.0, 1.0, 5.0]], device=dev)
    rs = R.GaussianRasterizationSettings(8, 8, 0.5, 0.5, torch.zeros(3, device=dev), 1.0, torch.eye(4, device=dev),
                                         torch.eye(4, device=dev), 0, torch.zeros(3, device=dev), False, False)
    vis = R.GaussianRasterizer(rs).markVisible(pts)
    assert vis.dtype == torch.bool and vis.tolist() == [False, False, True, True]


def test_non_default_stream_and_noncontiguous_inputs(dev):
    from tests.golden.make_golden import build_case
    inp = build_case(4000, 96, 96, 61)
    base = _run_ours(inp, dev, with_grads=True)
    s = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(s):
        other = _run_ours(inp, dev, with_grads=True)
    s.synchronize()
    assert torch.equal(base["color"], other["color"])
    # non-contiguous means3D / scales (the binding makes them contiguous like the reference's .contiguous())
    from vidu4d_b200 import rasterizer as R
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in inp.items() if k != "meta"}
    big = torch.zeros((4000, 6), device=dev)
    big[:, ::2] = t["means3D"]
    e = torch.empty((0,), device=dev)
    out = R._C.rasterize_gaussians(t["bg"], big[:, ::2], e, t["opacities"], t["scales"], t["rotations"], 1.0, e, t["viewmatrix"],
                                   t["projmatrix"], 0.5, 0.5, 96, 96, t["shs"], 3, t["campos"], False, False)
    assert torch.equal(out[1], base["color"])


def test_very_long_tile_lists_against_oracle(dev):
    """50 K surfels on a 32x32 image: 4 tiles of > 8 K instances each (dozens of ring chunks per tile, look-back over
    many sort tiles): sorted list bit-exact and colour within tolerance of the CPU oracle."""
    from oracle import surfel_oracle as so
    from tests.golden.make_golden import build_case
    inp = build_case(50000, 32, 32, 72)
    r = _run_ours(inp, dev)
    st = so.forward(inp["means3D"], inp["opacities"], inp["scales"], inp["rotations"], shs=inp["shs"], sh_degree=3, W=32, H=32,
                    tanfovx=0.5, tanfovy=0.5, bg=inp["bg"], viewmatrix=inp["viewmatrix"], projmatrix=inp["projmatrix"],
                    campos=inp["campos"])
    og = so.backward(st, inp["dL_dcolor"], inp["dL_dallmap"])
    assert r["num_rendered"] == st.num_rendered and int(_np(r["ranges"]).max()) > 8192
    np.testing.assert_array_equal(_np(r["point_list"]).astype(np.uint32), st.point_list)
    _assert_close_robust(_np(r["color"]), st.color, TOL, "color")
    for k in GRADS:
        _assert_close_robust(_np(r["grads"][k]), og[k], TOL, k)


def test_render_fused_matches_render(dev):
    """render_fused() (one CUDA kernel each way for the allmap post-processing) == render() (the reference's torch
    expressions, gaussian_renderer/__init__.py:121-162 + point_utils.py:9-37): values and parameter gradients."""
    from vidu4d_b200.renderer import PipelineParams, make_camera, render, render_fused
    from vidu4d_b200.synthetic import random_rotation
    rng = np.random.default_rng(5)
    Rc = random_rotation(rng)
    # camera looking at the object from a rotated frame: camera-to-world rotation Rc, object kept at distance ~1
    T = -Rc.T @ np.array([0.0, 0.0, 0.0]) + np.array([0.05, -0.03, 0.0])
    cam = make_camera(160, 112, 2 * np.arctan(0.5), 2 * np.arctan(0.35), device=dev)
    bg = torch.tensor([0.1, 0.3, 0.2], device=dev)
    g = torch.Generator(device=dev).manual_seed(9)
    wts = {k: torch.randn((c, 112, 160), device=dev, generator=g) for k, c in
           (("render", 3), ("acc", 1), ("rend_normal", 3), ("rend_dist", 1), ("surf_depth", 3), ("render_depth_median", 3),
            ("render_depth_expected", 3), ("surf_normal", 3))}
    for depth_ratio in (0.0, 0.3):
        grads = []
        outs = []
        for fn in (render, render_fused):
            cloud = _cloud(6000, dev, seed=11)
            out = fn(cam, cloud, PipelineParams(depth_ratio=depth_ratio), bg)
            loss = sum((out[k] * w).sum() for k, w in wts.items())
            loss.backward()
            outs.append(out)
            grads.append([p.grad.clone() for p in cloud.flat_params()])
        for k in wts:
            a, b = outs[0][k], outs[1][k]
            assert a.shape == b.shape, k
            # surf_normal normalises a cross product of central differences: ill-conditioned on silhouettes, so two
            # correct fp32 evaluation orders differ by ~1e-5 there; everything else agrees to the last bits
            tol = 1e-4 if k == "surf_normal" else 1e-5
            assert float((a.detach() - b.detach()).abs().max()) <= tol * float(a.detach().abs().max() + 1e-6), (k, depth_ratio)
        for ga, gb in zip(*grads):
            assert float((ga - gb).abs().max()) <= 1e-3 * float(ga.abs().max() + 1e-30), depth_ratio


def test_stage3_standin_loss_decreases(dev):
    """configs[2] in miniature: bob-skinning warp (PyTorch) -> render_fused -> loss -> Adam, non-leaf rasterizer inputs,
    in-place learnable-background edit of the render before backward.  The loss must go down."""
    import importlib.util
    import os
    from .conftest import ROOT
    spec = importlib.util.spec_from_file_location("stage3_standin", os.path.join(ROOT, "examples", "stage3_standin.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    r = m.run(surfels=20000, res=128, frames=8, steps=60, bones=12, log_every=10, quiet=True)
    first, last = r["losses"][0][1], r["losses"][-1][1]
    assert np.isfinite(last) and last < 0.8 * first, r["losses"]


@pytest.mark.parametrize("M,deg", [(1, 0), (4, 1), (9, 2), (16, 1)])
def test_sh_coefficient_counts_against_oracle(M, deg, dev):
    """shs with fewer than 16 coefficients per surfel (M = sh.size(1)) and an active degree below the stored one:
    exercises the generic (non-float4) staging paths of preprocess_fwd / surfel_bwd."""
    from oracle import surfel_oracle as so
    from tests.golden.make_golden import build_case
    inp = build_case(3000, 96, 80, 80 + M, sh_degree=deg)
    inp["shs"] = np.ascontiguousarray(inp["shs"][:, :M])
    r = _run_ours(inp, dev)
    st = so.forward(inp["means3D"], inp["opacities"], inp["scales"], inp["rotations"], shs=inp["shs"], sh_degree=deg, W=96, H=80,
                    tanfovx=0.5, tanfovy=0.5, bg=inp["bg"], viewmatrix=inp["viewmatrix"], projmatrix=inp["projmatrix"],
                    campos=inp["campos"])
    og = so.backward(st, inp["dL_dcolor"], inp["dL_dallmap"])
    np.testing.assert_array_equal(_np(r["point_list"]).astype(np.uint32), st.point_list)
    _assert_close_robust(_np(r["color"]), st.color, TOL, "color")
    assert r["grads"]["dL_dsh"].shape == (3000, M, 3)
    for k in GRADS:
        _assert_close_robust(_np(r["grads"][k]), og[k], TOL, k)
    used = (deg + 1) ** 2
    assert float(r["grads"]["dL_dsh"][:, used:].abs().sum()) == 0.0     # coefficients above the active degree get no gradient


def test_prefiltered_flag_reports_culled_surfels(dev):
    """The reference __trap()s when `prefiltered` is set and a surfel is culled (auxiliary.h:175-183); we raise."""
    from tests.golden.make_golden import build_case
    from vidu4d_b200 import rasterizer as R
    inp = build_case(600, 64, 64, 16, center=(0.0, 0.0, 0.45), sh_degree=0)       # part of the cloud is behind z = 0.2
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in inp.items() if k != "meta"}
    e = torch.empty((0,), device=dev)
    with pytest.raises(RuntimeError, match="prefiltered"):
        R._C.rasterize_gaussians(t["bg"], t["means3D"], e, t["opacities"], t["scales"], t["rotations"], 1.0, e, t["viewmatrix"],
                                 t["projmatrix"], 0.5, 0.5, 64, 64, t["shs"], 0, t["campos"], True, False)


_GROUP_CHILD = r'''
import sys, numpy as np, torch
sys.path.insert(0, sys.argv[1])
from tests.test_gpu_parity import _run_ours
from tests.golden.make_golden import build_case
inp = build_case(6000, 112, 80, 77)
r = _run_ours(inp, torch.device("cuda:0"), with_grads=True)
np.savez(sys.argv[2], color=r["color"].cpu().numpy(), allmap=r["allmap"].cpu().numpy(),
         n_contrib=r["n_contrib"].cpu().numpy(), **{"g_" + k: v.cpu().numpy() for k, v in r["grads"].items()})
'''


@pytest.mark.gpu
@pytest.mark.parametrize("fwd_g,bwd_g", [(8, 8), (16, 16), (4, 32), (32, 8)])
def test_alternative_group_sizes_agree_with_default(fwd_g, bwd_g, dev, tmp_path):
    """The pixel-block size of the composite kernels is a tuning switch read once per process
    (SURFEL_FWD_GROUPS / SURFEL_BWD_GROUPS): every combination must give the forward planes bit for bit (per-pixel
    arithmetic and instance order do not depend on it) and the same gradients up to summation order."""
    import subprocess, sys
    from tests.golden.make_golden import build_case
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    base = _run_ours(build_case(6000, 112, 80, 77), dev, with_grads=True)
    out = str(tmp_path / "alt.npz")
    env = dict(os.environ, SURFEL_FWD_GROUPS=str(fwd_g), SURFEL_BWD_GROUPS=str(bwd_g))
    r = subprocess.run([sys.executable, "-c", _GROUP_CHILD, root, out], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    alt = np.load(out)
    np.testing.assert_array_equal(alt["color"], _np(base["color"]))
    np.testing.assert_array_equal(alt["allmap"], _np(base["allmap"]))
    np.testing.assert_array_equal(alt["n_contrib"][0], _np(base["n_contrib"])[0])
    for k, v in base["grads"].items():
        a, b = alt["g_" + k], _np(v)
        scale = max(float(np.abs(b).max()), 1e-20)
        assert float(np.abs(a - b).max()) <= 2e-5 * scale, k
