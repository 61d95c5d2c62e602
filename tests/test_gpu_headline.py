"""GPU parity of the BENCHMARKED kernels at the BENCHMARKED configuration (300 K surfels, 512x512, bench.py's scene
and cameras) against the unmodified reference extension compiled for sm_100a, through the digests of its outputs in
tests/golden/ref_headline_*.npz (tests/golden/make_golden.py --digests): tile assignment / sort / ranges / contributor
counts bit-exact, rendered planes and all eight gradient tensors within 1e-4 (north_star), the latter at a fixed
sample of pixels and surfels and in their largest magnitude.
"""
import numpy as np
import pytest
import torch

from .conftest import load_golden
from .test_gpu_parity import TOL, _assert_close_to_digest, _assert_grads_close_to_digest, _assert_index_work_matches_digest, _np, _run_ours

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev(built):
    from vidu4d_b200 import _capi
    _capi.load()
    return torch.device("cuda:0")


@pytest.mark.parametrize("view", [None, 0, 17], ids=["identity", "orbit0", "orbit17"])
def test_headline_against_live_reference(view, dev):
    from tests.golden.make_golden import BIG_CASES, array_sha, inputs_sha
    name = "ref_headline_" + ("identity" if view is None else f"orbit{view}")
    g = load_golden(name)
    inp = BIG_CASES[name]()
    assert np.array_equal(inputs_sha(inp), g["inputs_sha"]), "the seeded inputs differ from the ones the digest was made of"
    r = _run_ours(inp, dev)
    assert int(g["num_rendered"][0]) > 300_000
    # ---- integer / index work: bit-exact
    _assert_index_work_matches_digest(r, g)
    # ---- rendered planes: 1e-4 relative (north_star).  Observed: depth/alpha/normal/median planes bit-identical; colour
    # within 1 ulp on ~0.1 % of the pixels (the SH -> RGB evaluation of a surfel is value-level, not FMA-mapped, since
    # no binning decision depends on it), distortion within 1e-7 (fp32 depth mapping, DESIGN.md 3.1).  Assert a
    # bound 100x tighter than the contract so that a real regression cannot hide.
    color, am = _np(r["color"]), _np(r["allmap"])
    _assert_close_to_digest(color.reshape(3, -1), g["pix"], g["color_at_pix"], g["absmax_color"],
                            1e-6 * max(1.0, float(g["absmax_color"])), "color")
    _assert_close_to_digest(am[6].reshape(-1), g["pix"], g["allmap_at_pix"][6], g["absmax_allmap"][6],
                            TOL * max(float(g["absmax_allmap"][6]), 1e-30), "allmap[6]")
    for ch in (0, 1, 2, 3, 4, 5, 7):
        assert np.array_equal(array_sha(am[ch]), g["sha_allmap"][ch]), f"allmap[{ch}] is expected bit-identical to the reference build"
    # ---- all eight gradient tensors: 1e-4 of the tensor's max magnitude
    _assert_grads_close_to_digest(r, g)
