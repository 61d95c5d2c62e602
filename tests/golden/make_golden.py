"""Generate the golden fixtures that pin the CPU oracle (and the CUDA path) to the REFERENCE ITSELF.

The reference (yikaiw/Vidu4D, gs/submodules/diff-surfel-rasterization) has no tests or golden vectors for
this path (SURVEY.md section 4), and it has no CPU implementation, so its outputs can only be produced on a
GPU.  This script runs the UNMODIFIED reference extension (oracle/_ref/_C.so, built by oracle/build_ref.sh
for sm_100a) on seeded scenes on the B200 box and stores inputs + every output / intermediate buffer:

    python tests/golden/make_golden.py             # writes tests/golden/<case>.npz
    python tests/golden/make_golden.py --digests   # writes tests/golden/ref_<case>.npz

Fixtures are small (<= ~1.5K surfels, <= 96x64 px).  tests/test_oracle_golden.py (CPU) checks the oracle
against them; tests/test_gpu_parity.py (GPU) checks the CUDA library against them.

The full-size cases (BIG_CASES: 100 K and 300 K surfels at 512x512) have tens of MB of reference outputs, so
--digests stores a digest of each instead (digest_reference): SHA-256 of every array the GPU tests require to be
bit-exact, the largest magnitude of every array they compare within a tolerance, and the values of those arrays
at a fixed, seeded sample of pixels and visible surfels.  tests/test_gpu_headline.py and
tests/test_gpu_parity.py::test_against_live_reference_c2 check the CUDA library against them.
"""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_ext  # noqa: E402
from vidu4d_b200.synthetic import object_scene, orbit_view, projection_matrix, random_rotation, rigid_view  # noqa: E402

CASES = {
    # name: (P, W, H, seed, options)
    "id_deg3_64": dict(P=1000, W=64, H=64, seed=11),
    "rigid_bg_96x64": dict(P=1200, W=96, H=64, seed=12, rigid=True, bg=(0.2, 0.5, 0.7)),
    "ragged_80x48_deg1": dict(P=900, W=80, H=48, seed=13, sh_degree=1, rigid=True),
    "precomp_init_70x50": dict(P=800, W=70, H=50, seed=14, colors_precomp=True, opacity="init"),
    "big_surfels_64": dict(P=300, W=64, H=64, seed=15, scale_mul=6.0, sh_degree=2),
    "near_cull_64": dict(P=600, W=64, H=64, seed=16, center=(0.0, 0.0, 0.45), sh_degree=0),
    "single_32": dict(P=1, W=32, H=32, seed=17),
}


def build_case(P, W, H, seed, rigid=False, bg=(0.0, 0.0, 0.0), sh_degree=3, colors_precomp=False, opacity="trained",
               scale_mul=1.0, center=(0.0, 0.0, 1.0)):
    sc = object_scene(P, seed=seed, opacity=opacity, sh_degree=sh_degree, center=center)
    sc.scales = (sc.scales * scale_mul).astype(np.float32)
    vm = np.eye(4, dtype=np.float32)
    campos = np.zeros(3, np.float32)
    if rigid:
        rng = np.random.default_rng(seed + 100)
        sc, vm, campos = rigid_view(sc, random_rotation(rng), np.array([0.3, -0.2, 0.5]))
    tan = 0.5
    pm = (vm.astype(np.float64) @ projection_matrix(tan, tan).astype(np.float64)).astype(np.float32)
    rng = np.random.default_rng(seed + 7)
    inp = dict(
        means3D=sc.means3D, scales=sc.scales, rotations=sc.rotations, opacities=sc.opacities,
        shs=sc.shs if not colors_precomp else np.zeros((0,), np.float32),
        colors_precomp=rng.uniform(0, 1, size=(P, 3)).astype(np.float32) if colors_precomp else np.zeros((0,), np.float32),
        viewmatrix=vm, projmatrix=pm, campos=campos, bg=np.asarray(bg, np.float32),
        dL_dcolor=rng.normal(size=(3, H, W)).astype(np.float32),
        dL_dallmap=rng.normal(size=(8, H, W)).astype(np.float32),
        meta=np.array([P, W, H, sh_degree, int(colors_precomp)], np.int64),
        tanfov=np.array([tan, tan], np.float32),
    )
    return inp


def bench_inputs(view, P=300_000, res=512):
    """The exact inputs bench.py renders: object_scene(seed 0, trained opacities) at the world origin, orbit camera
    `view` of 64 (view=None: the Stage-3 identity camera with the object at z = 1)."""
    tan = 0.5
    Pm = projection_matrix(tan, tan).astype(np.float64)
    if view is None:
        sc = object_scene(P, seed=0, opacity="trained", center=(0.0, 0.0, 1.0))
        vm = np.eye(4, dtype=np.float32); cp = np.zeros(3, np.float32)
    else:
        sc = object_scene(P, seed=0, opacity="trained", center=(0.0, 0.0, 0.0))
        R, t = orbit_view(view, 64)
        W2C = np.eye(4); W2C[:3, :3] = R; W2C[:3, 3] = t
        vm = W2C.T.astype(np.float32); cp = (-R.T @ t).astype(np.float32)
    pm = (vm.astype(np.float64) @ Pm).astype(np.float32)
    rng = np.random.default_rng(1234)
    return dict(means3D=sc.means3D, scales=sc.scales, rotations=sc.rotations, opacities=sc.opacities, shs=sc.shs,
                colors_precomp=np.zeros((0,), np.float32), viewmatrix=vm, projmatrix=pm, campos=cp,
                bg=np.zeros(3, np.float32), dL_dcolor=rng.normal(size=(3, res, res)).astype(np.float32),
                dL_dallmap=(0.1 * rng.normal(size=(8, res, res))).astype(np.float32),
                meta=np.array([P, res, res, 3, 0], np.int64), tanfov=np.array([tan, tan], np.float32))


BIG_CASES = {
    "ref_headline_identity": lambda: bench_inputs(None),
    "ref_headline_orbit0": lambda: bench_inputs(0),
    "ref_headline_orbit17": lambda: bench_inputs(17),
    "ref_c2_100k_512": lambda: build_case(100_000, 512, 512, 31, rigid=True),     # BASELINE config[1]
}
DIGEST_PIXELS, DIGEST_SURFELS = 512, 64


def array_sha(a) -> np.ndarray:
    """SHA-256 (32 uint8) of an array's shape and values: integers as int64, floats as float32 with -0.0 folded into
    +0.0, so that two arrays have the same digest exactly when np.array_equal holds for them."""
    a = np.asarray(a)
    a = a.astype("<i8") if a.dtype.kind in "biu" else a.astype("<f4") + np.float32(0.0)
    h = hashlib.sha256(repr(a.shape).encode())
    h.update(np.ascontiguousarray(a).tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def inputs_sha(inp) -> np.ndarray:
    return array_sha(np.concatenate([array_sha(inp[k]) for k in sorted(inp)]))


def digest_reference(inp, ref) -> dict:
    """What the full-size GPU tests compare against, small enough to commit (see the module docstring)."""
    P, W, H = [int(v) for v in inp["meta"][:3]]
    rng = np.random.default_rng(0)
    pix = np.sort(rng.choice(W * H, DIGEST_PIXELS, replace=False)).astype(np.int32)
    vis = np.flatnonzero(ref["radii"] > 0)
    surf = np.sort(rng.choice(vis, min(DIGEST_SURFELS, vis.size), replace=False)).astype(np.int32)
    # contributor planes: the median plane only in tiles whose list is non-empty (the reference leaves garbage in
    # the others), zero elsewhere, which is what the CUDA library writes there
    nc = ref["img_n_contrib"].astype(np.int64) & 0xFFFFFFFF
    rg = ref["img_ranges"].astype(np.int64)
    tile = (np.arange(H)[:, None] // 16) * ((W + 15) // 16) + np.arange(W)[None, :] // 16
    nc1 = np.where((rg[:, 1] - rg[:, 0])[tile] > 0, nc[1], 0)
    color, allmap = ref["color"], ref["allmap"]
    d = dict(inputs_sha=inputs_sha(inp), num_rendered=ref["num_rendered"], pix=pix, surf=surf,
             sha_radii=array_sha(ref["radii"]), sha_keys=array_sha(ref["bin_keys"]),
             sha_point_list=array_sha(ref["bin_point_list"]), sha_ranges=array_sha(ref["img_ranges"]),
             sha_n_contrib0=array_sha(nc[0]), sha_n_contrib1=array_sha(nc1),
             sha_color=array_sha(color), sha_allmap=np.stack([array_sha(c) for c in allmap]),
             absmax_color=np.float64(np.abs(color).max()), absmax_allmap=np.abs(allmap).reshape(8, -1).max(1).astype(np.float64),
             color_at_pix=color.reshape(3, -1)[:, pix], allmap_at_pix=allmap.reshape(8, -1)[:, pix])
    for k in (k[5:] for k in ref if k.startswith("grad_")):
        g = ref["grad_" + k]
        d["shape_" + k] = np.array(g.shape, np.int64)
        if g.size:
            assert g.shape[0] == P, (k, g.shape)
            d["absmax_" + k] = np.float64(np.abs(g).max())
            d["grad_" + k] = g[surf]
    return d


def run_reference(inp, dev):
    P, W, H, deg, pre = [int(v) for v in inp["meta"]]
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in inp.items() if k not in ("meta",)}
    shs = None if pre else t["shs"]
    col = t["colors_precomp"] if pre else None
    kw = dict(sh_degree=deg, tanfovx=float(inp["tanfov"][0]), tanfovy=float(inp["tanfov"][1]), bg=t["bg"],
              viewmatrix=t["viewmatrix"], projmatrix=t["projmatrix"], campos=t["campos"])
    fw = ref_ext.forward(t["means3D"], t["opacities"], t["scales"], t["rotations"], shs=shs, colors_precomp=col,
                         W=W, H=H, **kw)
    gb = ref_ext.backward(fw, t["means3D"], t["scales"], t["rotations"], shs=shs, colors_precomp=col,
                          dL_dcolor=t["dL_dcolor"], dL_dallmap=t["dL_dallmap"], **kw)
    R = int(fw["num_rendered"])
    out = dict(num_rendered=np.array([R], np.int64), color=ref_ext.to_np(fw["color"]), allmap=ref_ext.to_np(fw["allmap"]),
               radii=ref_ext.to_np(fw["radii"]))
    for k, v in ref_ext.decode_geom(fw["geomBuffer"], P).items():
        out["geom_" + k] = ref_ext.to_np(v)
    for k, v in ref_ext.decode_binning(fw["binningBuffer"], R).items():
        out["bin_" + k] = ref_ext.to_np(v)
    for k, v in ref_ext.decode_image(fw["imgBuffer"], W, H).items():
        out["img_" + k] = ref_ext.to_np(v)
    for k, v in gb.items():
        out["grad_" + k] = ref_ext.to_np(v)
    return out


def main():
    dev = torch.device("cuda:0")
    outdir = os.path.join(ROOT, "tests", "golden")
    if "--digests" in sys.argv[1:]:
        for name, make in BIG_CASES.items():
            inp = make()
            out = run_reference(inp, dev)
            np.savez_compressed(os.path.join(outdir, name + ".npz"), **digest_reference(inp, out))
            print(name, "R =", int(out["num_rendered"][0]), "visible =", int((out["radii"] > 0).sum()))
        return
    for name, kw in CASES.items():
        inp = build_case(**kw)
        out = run_reference(inp, dev)
        np.savez_compressed(os.path.join(outdir, name + ".npz"), **{"in_" + k: v for k, v in inp.items()},
                            **{"ref_" + k: v for k, v in out.items()})
        print(name, "R =", int(out["num_rendered"][0]), "visible =", int((out["radii"] > 0).sum()))


if __name__ == "__main__":
    main()
