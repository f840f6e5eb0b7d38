"""The reference's operator registry, parameter coercions and chain, as recorded from its own classes (src/preprocess/registry.py:14-28,
ops/clahe_dehaze.py:14-17, ops/median_derain.py:11-13; SURVEY.md section 8b, rows a6 / a11 and "Param coercions"; tests/golden/
chain_small.npz), against this package and the restatement in oracle/cv2_chain.py."""
import numpy as np
import pytest

from conftest import load_golden_cases

# the reference's REGISTRY keys and the message of its get_op_class() for an unknown name
REFERENCE_REGISTRY = {"CLAHEDehaze", "MedianDerain", "CUDACLAHEDehaze", "CUDAMedianDerain"}
REFERENCE_UNKNOWN_OP = "Preprocess op 'Nope' not found"

# raw CLAHEDehaze params -> (colour path, clip limit, tile grid) and raw ksize -> median size, as the reference's classes coerce them
# (exactly "LAB" after upper() selects LAB, anything else YCrCb; float(clip); max(2, int(grid)); int(k), even -> k + 1, clamp [3, 9])
REFERENCE_CLAHE = [({"space": "LAB", "clip_limit": 2.0, "tile_grid": 8}, ("LAB", 2.0, 8)),
                   ({"space": "ycrcb", "clip_limit": "3", "tile_grid": 1}, ("YCrCb", 3.0, 2)),
                   ({"space": "hsv", "clip_limit": 0, "tile_grid": 8.9}, ("YCrCb", 0.0, 8)),
                   ({}, ("YCrCb", 2.0, 8)),
                   ({"space": "Lab"}, ("LAB", 2.0, 8)),
                   ({"tile_grid": "8"}, ("YCrCb", 2.0, 8)),
                   ({"clip_limit": "2"}, ("YCrCb", 2.0, 8)),
                   ({"clip_limit": -1}, ("YCrCb", -1.0, 8)),
                   ({"bogus": 1}, ("YCrCb", 2.0, 8))]
REFERENCE_KSIZE = [(1, 3), (2, 3), (3, 3), (3.9, 3), ("5", 5), (6, 7), (11, 9), (100, 9)]


def test_cv2_chain_equals_reference_classes():
    """oracle/cv2_chain with raw, uncoerced parameters: its coercions are the reference's, and raw spellings of every reference-made
    golden case (lower-case space, clip as a string, fractional grid, even ksize) reproduce the reference's stored output."""
    from oracle import cv2_chain as R
    for params, (path, clip, grid) in REFERENCE_CLAHE:
        space, c, g = R.coerce_clahe_params(params)
        assert ("LAB" if space == "LAB" else "YCrCb", c, g) == (path, clip, grid), params
    for k, want in REFERENCE_KSIZE:
        assert R.coerce_ksize({"ksize": k}) == want, k
    cases, _, _ = load_golden_cases()
    for c in cases:
        raw = {"space": c["space"].lower(), "clip_limit": str(c["clip"]), "tile_grid": c["grid"] + 0.5}
        space, clip, grid = R.coerce_clahe_params(raw)
        k = R.coerce_ksize({"ksize": c["k"] - 1}) if c["k"] > 3 else (R.coerce_ksize({"ksize": 2}) if c["k"] else 0)
        assert np.array_equal(R.chain(c["inp"], space, clip, grid, k), c["out"]), c["idx"]


def test_registry_names_match_reference():
    import rvb200
    assert REFERENCE_REGISTRY <= set(rvb200.REGISTRY)
    with pytest.raises(KeyError) as e:
        rvb200.get_op_class("Nope")
    assert REFERENCE_UNKNOWN_OP in str(e.value)


def test_param_coercions_match_reference_source():
    """Our coerce() helpers against the coercions spelled out in clahe_dehaze.py:14-17 / median_derain.py:11-13."""
    from rvb200.preprocess.ops import clahe_dehaze as c, median_derain as m
    from oracle import cv2_chain as R
    for params in [{}, {"space": "Lab"}, {"space": "hsv"}, {"tile_grid": 1}, {"tile_grid": "8"}, {"tile_grid": 8.9},
                   {"clip_limit": "2"}, {"clip_limit": 0}, {"clip_limit": -1}, {"bogus": 1}]:
        space, clip, grid = R.coerce_clahe_params(params)
        assert c.coerce(params) == ("LAB" if space == "LAB" else "YCrCb", clip, grid)
    for k in [1, 2, 3, 3.9, "5", 6, 7, 8, 9, 11, 100]:
        assert m.coerce({"ksize": k}) == R.coerce_ksize({"ksize": k})
