"""Generates tests/golden/*.npz by running the UNMODIFIED reference model (imported read-only from
/root/reference) on the seeded, calibrated checkpoint.  TEST INFRASTRUCTURE ONLY; run in the build
container (the reference does not travel to the GPU box):

    python -m oracle.make_golden

The reference has no golden vectors of its own (SURVEY §4); these files pin `oracle/siammask_oracle.py`
to the reference implementation itself."""
from __future__ import annotations

import os
import sys
import warnings

import numpy as np
import torch

REF = os.environ.get("SIAMMASK_REFERENCE", "/root/reference")
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
MASK_CH = slice(0, 3969, 97)      # 41 of the 3969 mask-head channels (the full tensor is 9.9 MB)
ANCHORS = {"stride": 8, "ratios": [0.33, 0.5, 1, 2, 3], "scales": [8], "round_dight": 0}


def reference_model(sd):
    sys.path[:0] = [REF, os.path.join(REF, "experiments", "siammask_sharp")]
    from custom import Custom  # noqa: the reference's own class
    m = Custom(anchors=ANCHORS).eval()
    m.load_state_dict(sd, strict=False)
    return m


def sub(t, step):
    return t.flatten()[::step].numpy().copy()


def reference_loop_functions():
    """Import siamese_init / siamese_track from the UNMODIFIED tools/test.py with the shims SURVEY §8c lists
    (pyvotkit stub, numpy-2 aliases, cv2 version probe) — nothing in /root/reference is touched."""
    import types
    import cv2
    stub = types.ModuleType("utils.pyvotkit.region")
    stub.vot_overlap = lambda *a, **k: 0.0
    stub.vot_float2str = lambda *a, **k: ""
    sys.modules.setdefault("utils.pyvotkit.region", stub)
    pk = types.ModuleType("utils.pyvotkit")
    pk.__path__ = []
    sys.modules.setdefault("utils.pyvotkit", pk)
    for name, val in (("float", float), ("int", int), ("int0", np.intp)):
        if not hasattr(np, name):
            setattr(np, name, val)
    cv2.__version__ = "4.5.0"          # tools/test.py:285 probes __version__[-5]
    sys.path[:0] = [REF, os.path.join(REF, "experiments", "siammask_sharp")]
    from tools.test import siamese_init, siamese_track  # noqa
    return siamese_init, siamese_track


def tracker_loop_golden(sd):
    """The reference's own tracker loop (tools/test.py:132-315) driven by the oracle network on synthetic frames."""
    from oracle.siammask_oracle import Oracle
    from oracle.synthetic_video import make_frames
    siamese_init, siamese_track = reference_loop_functions()
    frames, boxes = make_frames()
    x, y, w, h = boxes[0]
    hp = {"instance_size": 255, "base_size": 8, "out_size": 127, "seg_thr": 0.35, "penalty_k": 0.04,
          "window_influence": 0.4, "lr": 1.0}                      # config_davis.json
    net = Oracle(sd)
    state = siamese_init(frames[0], np.array([x + w / 2, y + h / 2]), np.array([w, h]), net, hp, device="cpu")
    rec = {"pos": [], "sz": [], "score": [], "mask_area": [], "polygon": []}
    for f in frames[1:]:
        state = siamese_track(state, f, mask_enable=True, refine_enable=True, device="cpu")
        rec["pos"].append(state["target_pos"].copy())
        rec["sz"].append(state["target_sz"].copy())
        rec["score"].append(state["score"])
        rec["mask_area"].append(float((state["mask"] > hp["seg_thr"]).sum()))
        rec["polygon"].append(np.asarray(state["ploygon"], dtype=np.float64))
    np.savez_compressed(os.path.join(OUT, "tracker_loop.npz"), **{k: np.asarray(v) for k, v in rec.items()})


def sharp_383_golden(m):
    """Sharp path at search 383 (BASELINE.json configs[4]): 41x41 response, refine at the corners and an interior
    position, 21 mask-head channels, sub-sampled pyramid — from the unmodified reference model."""
    from oracle.calibrate import synthetic_inputs
    z, x = synthetic_inputs(3, 1, search=383)
    m.template(z)
    cls, loc, mask = m.track_mask(x)
    feats = {f"p{i}": sub(f, 509) for i, f in enumerate(m.feature)}
    ref = {f"refine_{dy}_{dx}": m.track_refine((dy, dx)).numpy() for dy, dx in ((0, 0), (40, 40), (7, 33))}
    np.savez_compressed(os.path.join(OUT, "sharp_b1_s383.npz"), cls=cls.numpy(), loc=loc.numpy(),
                        mask_sub=mask[:, slice(0, 3969, 193)].numpy(), search=sub(m.search, 13),
                        corr=sub(m.corr_feature, 13), **feats, **ref)


def sharp_seed11_golden(m):
    """Sharp path at search 255 on the seed-11 inputs: cls, loc, 21 mask-head channels and the refine logits at the
    border position (0, 24) — what tests/test_oracle.py::test_oracle_matches_reference_outputs compares against."""
    from oracle.calibrate import synthetic_inputs
    z, x = synthetic_inputs(11, 1)
    m.template(z)
    cls, loc, mask = m.track_mask(x)
    np.savez_compressed(os.path.join(OUT, "sharp_b1_s255_seed11.npz"), cls=cls.numpy(), loc=loc.numpy(),
                        mask_sub=mask[:, slice(0, 3969, 193)].numpy(), refine_0_24=m.track_refine((0, 24)).numpy())


def main():
    from oracle.calibrate import calibrated_state_dict, synthetic_inputs
    only = {"--only-383": sharp_383_golden, "--only-seed11": sharp_seed11_golden}
    for flag, fn in only.items():         # add one file's vectors without rewriting the other files
        if flag in sys.argv:
            warnings.filterwarnings("ignore")
            torch.set_num_threads(8)
            with torch.no_grad():
                fn(reference_model(calibrated_state_dict(0)))
            return
    warnings.filterwarnings("ignore")
    torch.set_num_threads(8)
    sd = calibrated_state_dict(0)
    m = reference_model(sd)
    os.makedirs(OUT, exist_ok=True)
    with torch.no_grad():
        # --- config 1: B=1, search 255
        z, x = synthetic_inputs(1, 1)
        m.template(z)
        cls, loc, mask = m.track_mask(x)
        feats = {f"p{i}": sub(f, 257) for i, f in enumerate(m.feature)}
        r1 = m.track_refine((12, 12))
        r2 = m.track_refine((3, 20))
        np.savez_compressed(os.path.join(OUT, "sharp_b1_s255.npz"), cls=cls.numpy(), loc=loc.numpy(),
                            mask_sub=mask[:, MASK_CH].numpy(), refine_12_12=r1.numpy(), refine_3_20=r2.numpy(),
                            zf=m.zf.numpy(), search=sub(m.search, 7), corr=sub(m.corr_feature, 7), **feats)
        # --- paired batch B=2 (the reference's batched semantics, SURVEY 0.5), track only
        z2, x2 = synthetic_inputs(2, 2)
        m.template(z2)
        cls2, loc2 = m.track(x2)
        np.savez_compressed(os.path.join(OUT, "rpn_b2_s255.npz"), cls=cls2.numpy(), loc=loc2.numpy())
        # --- large search 383 -> 41x41 response (SURVEY 0.4)
        z3, x3 = synthetic_inputs(3, 1, search=383)
        m.template(z3)
        cls3, loc3 = m.track(x3)
        np.savez_compressed(os.path.join(OUT, "rpn_b1_s383.npz"), cls=cls3.numpy(), loc=loc3.numpy())
        sharp_383_golden(m)
        sharp_seed11_golden(m)
        # --- standalone depthwise xcorr (models/rpn.py:32-38)
        sys.path[:0] = [REF]
        from models.rpn import conv2d_dw_group
        g = torch.Generator().manual_seed(7)
        xs = torch.randn(2, 8, 29, 29, generator=g)
        ks = torch.randn(2, 8, 5, 5, generator=g)
        np.savez_compressed(os.path.join(OUT, "xcorr_small.npz"), x=xs.numpy(), k=ks.numpy(),
                            out=conv2d_dw_group(xs, ks).numpy())
    tracker_loop_golden(sd)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
