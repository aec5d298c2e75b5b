"""The oracle against (i) the golden vectors produced by the unmodified reference (oracle/make_golden.py),
(ii) the reference's outputs on a second input at the tighter 1e-4, (iii) independent plain-loop restatements."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import GOLDEN, assert_close
from oracle.calibrate import synthetic_inputs
from oracle.siammask_oracle import Oracle, nearest_upsample_index, xcorr_depthwise_loops

# The golden vectors were produced on the build container's CPU.  The calibrated checkpoint is regenerated
# from its seed wherever the tests run; a different CPU (other conv kernels in the calibration pass) moves
# BN statistics by ~1e-7 and this seeded network amplifies perturbations ~100x, hence 1e-3 here.
GOLDEN_TOL = 1e-3
MASK_CH = slice(0, 3969, 97)


def _g(name):
    return {k: torch.from_numpy(v) for k, v in np.load(os.path.join(GOLDEN, name)).items()}


def test_xcorr_golden_and_loops():
    g = _g("xcorr_small.npz")
    out = Oracle.xcorr_depthwise(g["x"], g["k"])
    assert_close(out, g["out"], 1e-6, "xcorr oracle vs reference")
    loops = torch.from_numpy(xcorr_depthwise_loops(g["x"].numpy(), g["k"].numpy())).float()
    assert_close(loops, g["out"], 1e-6, "xcorr loops vs reference")


def test_xcorr_requires_paired_batch():
    # the reference cannot run 1 template x B searches (SURVEY 0.5): same failure in the restatement
    with pytest.raises(RuntimeError):
        Oracle.xcorr_depthwise(torch.zeros(2, 4, 9, 9), torch.zeros(1, 4, 5, 5))


@pytest.mark.parametrize("out_size,in_size", [(31, 15), (61, 31), (127, 61), (15, 15)])
def test_nearest_index_matches_torch(out_size, in_size):
    src = torch.arange(in_size, dtype=torch.float32).view(1, 1, 1, in_size)
    up = F.interpolate(src, size=(1, out_size)).flatten().long().numpy()
    assert np.array_equal(up, nearest_upsample_index(out_size, in_size))


def test_oracle_matches_golden_sharp(calib_sd):
    g = _g("sharp_b1_s255.npz")
    z, x = synthetic_inputs(1, 1)
    o = Oracle(calib_sd)
    o.template(z)
    cls, loc, mask = o.track_mask(x)
    assert_close(o.zf, g["zf"], GOLDEN_TOL, "zf")
    assert_close(cls, g["cls"], GOLDEN_TOL, "cls")
    assert_close(loc, g["loc"], GOLDEN_TOL, "loc")
    assert_close(mask[:, MASK_CH], g["mask_sub"], GOLDEN_TOL, "mask head (41 ch)")
    for i in range(4):
        assert_close(o.feature[i].flatten()[::257], g[f"p{i}"], GOLDEN_TOL, f"p{i}")
    assert_close(o.track_refine((12, 12)), g["refine_12_12"], GOLDEN_TOL, "refine (12,12)")
    assert_close(o.track_refine((3, 20)), g["refine_3_20"], GOLDEN_TOL, "refine (3,20)")


def test_oracle_matches_golden_batched_and_383(calib_sd):
    g = _g("rpn_b2_s255.npz")
    z, x = synthetic_inputs(2, 2)
    o = Oracle(calib_sd)
    o.template(z)
    cls, loc = o.track(x)
    assert_close(cls, g["cls"], GOLDEN_TOL, "cls B=2")
    assert_close(loc, g["loc"], GOLDEN_TOL, "loc B=2")
    g = _g("rpn_b1_s383.npz")
    z, x = synthetic_inputs(3, 1, search=383)
    o.template(z)
    cls, loc = o.track(x)
    assert cls.shape == (1, 10, 41, 41)      # 41x41, not 31x31 (SURVEY 0.4)
    assert_close(cls, g["cls"], GOLDEN_TOL, "cls @383")
    assert_close(loc, g["loc"], GOLDEN_TOL, "loc @383")


def test_oracle_matches_golden_sharp_383(calib_sd):
    """Sharp path at search 383 (BASELINE.json configs[4]): mask branch + refine incl. the corner positions."""
    g = _g("sharp_b1_s383.npz")
    z, x = synthetic_inputs(3, 1, search=383)
    o = Oracle(calib_sd)
    o.template(z)
    cls, loc, mask = o.track_mask(x)
    assert mask.shape == (1, 3969, 41, 41)
    assert_close(cls, g["cls"], GOLDEN_TOL, "cls @383")
    assert_close(mask[:, slice(0, 3969, 193)], g["mask_sub"], GOLDEN_TOL, "mask head @383")
    for i in range(4):
        assert_close(o.feature[i].flatten()[::509], g[f"p{i}"], GOLDEN_TOL, f"p{i} @383")
    assert_close(o.corr_feature.flatten()[::13], g["corr"], GOLDEN_TOL, "corr @383")
    for pos in ((0, 0), (40, 40), (7, 33)):
        assert_close(o.track_refine(pos), g[f"refine_{pos[0]}_{pos[1]}"], GOLDEN_TOL, f"refine {pos} @383")


def test_per_stream_refine_equals_per_sample_loop(calib_sd):
    z, x = synthetic_inputs(4, 2)
    o = Oracle(calib_sd)
    o.template(z)
    o.track_mask(x, with_mask_head=False)
    both = o.track_refine(np.array([[5, 7], [20, 2]]))
    o1 = Oracle(calib_sd)
    for b, pos in enumerate([(5, 7), (20, 2)]):
        o1.template(z[b:b + 1])
        o1.track_mask(x[b:b + 1], with_mask_head=False)
        assert_close(both[b:b + 1], o1.track_refine(pos), 1e-4, f"refine stream {b}")


def test_oracle_matches_reference_outputs(calib_sd):
    """The oracle against the unmodified reference model's own track_mask / track_refine outputs on the seed-11
    inputs, recorded by `python -m oracle.make_golden --only-seed11` (21 of the 3969 mask-head channels)."""
    g = _g("sharp_b1_s255_seed11.npz")
    z, x = synthetic_inputs(11, 1)
    o = Oracle(calib_sd)
    with torch.no_grad():
        o.template(z)
        cls, loc, mask = o.track_mask(x)
        assert_close(cls, g["cls"], 1e-4, "cls vs reference")
        assert_close(loc, g["loc"], 1e-4, "loc vs reference")
        assert_close(mask[:, slice(0, 3969, 193)], g["mask_sub"], 1e-4, "mask vs reference")
        assert_close(o.track_refine((0, 24)), g["refine_0_24"], 1e-4, "refine vs reference")
