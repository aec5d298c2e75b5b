"""End-to-end parity of the CUDA engine (through the Custom boundary / C ABI) against the CPU oracle on the
seeded calibrated checkpoint.  Tolerance: 1e-3 relative (BASELINE.json north_star), metric in conftest."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, assert_close
import siammask_b200 as smb
from oracle.calibrate import synthetic_inputs
from oracle.siammask_oracle import Oracle

pytestmark = pytest.mark.gpu
TOL = 1e-3


def _engine(sd, **kw):
    m = smb.Custom(anchors=smb.DEFAULT_ANCHORS, **kw)
    m.load_state_dict(sd)
    return m.eval().to("cuda")


def _check_intermediates(m, o, tol):
    for i, name in enumerate(("p0", "p1", "p2", "p3")):
        assert_close(m.export(name), o.feature[i], tol, name)
    assert_close(m.export("search"), o.search, tol, "search feature")
    assert_close(m.export("corr_mask"), o.corr_feature, tol, "mask corr feature")


@pytest.mark.parametrize("backend", ["tensor", "simt"])
def test_sharp_b1_matches_oracle(calib_sd, backend):
    z, x = synthetic_inputs(1, 1)
    o = Oracle(calib_sd)
    o.template(z)
    ocls, oloc, omask = o.track_mask(x)
    m = _engine(calib_sd, backend=backend)
    m.template(z.cuda())
    assert_close(m.export("zf"), o.zf, TOL, "zf")
    cls, loc, mask = m.track_mask(x.cuda())
    _check_intermediates(m, o, TOL)
    assert_close(cls, ocls, TOL, "cls")
    assert_close(loc, oloc, TOL, "loc")
    assert_close(mask, omask, TOL, "mask head")
    for pos in [(12, 12), (0, 0), (24, 24), (3, 20)]:
        assert_close(m.track_refine(pos), o.track_refine(pos), TOL, f"refine {pos}")
    # track() == track_mask() on cls/loc
    c2, l2 = m.track(x.cuda())
    assert_close(c2, ocls, TOL, "track cls")
    assert_close(l2, oloc, TOL, "track loc")


def test_sharp_matches_reference_golden(calib_sd):
    g = {k: torch.from_numpy(v) for k, v in np.load(os.path.join(GOLDEN, "sharp_b1_s255.npz")).items()}
    z, x = synthetic_inputs(1, 1)
    m = _engine(calib_sd)
    m.template(z.cuda())
    cls, loc, mask = m.track_mask(x.cuda())
    assert_close(cls, g["cls"], 2e-3, "cls vs reference golden")
    assert_close(loc, g["loc"], 2e-3, "loc vs reference golden")
    assert_close(mask[:, 0:3969:97], g["mask_sub"], 2e-3, "mask vs reference golden")
    assert_close(m.track_refine((12, 12)), g["refine_12_12"], 2e-3, "refine vs reference golden")


def test_batched_streams_and_slots(calib_sd):
    """B=3 paired streams in slots 1..3 of a 4-slot engine == three single-stream oracle runs; per-stream pos."""
    z, x = synthetic_inputs(21, 3)
    m = _engine(calib_sd, max_batch=3, num_slots=4)
    m.template(z.cuda(), slot0=1)
    cls, loc, _ = m.track_mask(x.cuda(), slot0=1, mask_head=False)
    pos = np.array([[5, 7], [20, 2], [12, 24]])
    ref = m.track_refine(pos)
    o = Oracle(calib_sd)
    for b in range(3):
        o.template(z[b:b + 1])
        ocls, oloc, _ = o.track_mask(x[b:b + 1], with_mask_head=False)
        assert_close(cls[b:b + 1], ocls, TOL, f"cls stream {b}")
        assert_close(loc[b:b + 1], oloc, TOL, f"loc stream {b}")
        assert_close(ref[b:b + 1], o.track_refine(pos[b]), TOL, f"refine stream {b}")
    # re-templating one slot must not disturb the others
    m.template(z[0:1].cuda(), slot0=2)
    cls2, _, _ = m.track_mask(x.cuda(), slot0=1, mask_head=False)
    assert_close(cls2[0:1], cls[0:1], 1e-6, "slot 1 untouched")
    assert float((cls2[1] - cls[1]).abs().max()) > 1e-3


def test_two_lane_batch_matches_single_stream_runs(calib_sd):
    """B=17 (>= 16) is split 9 + 8 over the engine's two concurrent lanes: every stream must equal its own
    single-stream run (B=1 engine = one lane, already pinned to the oracle), intermediates are gathered across the
    lanes, the graph-replay and host-buffer paths (lane 1 stays forked between track and refine) agree."""
    import ctypes as C
    from siammask_b200 import _lib
    B = 17
    z, x = synthetic_inputs(71, B)
    _, x2 = synthetic_inputs(72, B)
    pos = torch.tensor([[(3 * b) % 25, (7 * b + 2) % 25] for b in range(B)], dtype=torch.int32)
    m = _engine(calib_sd, max_batch=B, num_slots=B)
    m.template(z.cuda())
    cls, loc, mask = m.track_mask(x.cuda())
    p2 = m.export("p2")
    ref = m.track_refine(pos.cuda())
    assert p2.shape[0] == B
    one = _engine(calib_sd)
    o = Oracle(calib_sd)
    for b in (0, 8, 9, 16):                                  # last of lane 0, first / last of lane 1
        one.template(z[b:b + 1].cuda())
        c1, l1, m1 = one.track_mask(x[b:b + 1].cuda())
        assert_close(cls[b:b + 1], c1, 1e-6, f"cls stream {b}")
        assert_close(loc[b:b + 1], l1, 1e-6, f"loc stream {b}")
        assert_close(mask[b:b + 1], m1, 1e-6, f"mask stream {b}")
        assert_close(p2[b:b + 1], one.export("p2"), 1e-6, f"p2 stream {b}")
        assert_close(ref[b:b + 1], one.track_refine(tuple(int(v) for v in pos[b])), 1e-6, f"refine stream {b}")
    o.template(z[9:10])
    ocls, oloc, _ = o.track_mask(x[9:10], with_mask_head=False)
    assert_close(cls[9:10], ocls, TOL, "cls stream 9 vs oracle")
    assert_close(ref[9:10], o.track_refine(tuple(int(v) for v in pos[9])), TOL, "refine stream 9 vs oracle")
    # graph replay with both lanes captured
    g = _engine(calib_sd, max_batch=B, num_slots=B, graphs=True)
    g.template(z.cuda())
    for it, xin in enumerate([x, x2, x]):
        ce, le, _ = m.track_mask(xin.cuda(), mask_head=False)
        re_ = m.track_refine(pos.cuda())
        cg, lg, _ = g.track_mask(xin.cuda(), mask_head=False)
        rg = g.track_refine(pos.cuda())
        assert_close(cg, ce, 1e-6, f"two-lane graph cls call {it}")
        assert_close(rg, re_, 1e-6, f"two-lane graph refine call {it}")
    # host-buffer pipeline
    lib = _lib.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    want = []
    for xin in (x, x2):
        c, l, _ = m.track_mask(xin.cuda(), mask_head=False)
        want.append((c.cpu(), l.cpu(), m.track_refine(pos.cuda()).cpu()))
    xs = [x.contiguous().pin_memory(), x2.contiguous().pin_memory()]
    outs = [(torch.empty(B, 10, 25, 25).pin_memory(), torch.empty(B, 20, 25, 25).pin_memory(),
             torch.empty(B, 127 * 127).pin_memory()) for _ in range(2)]
    posh = pos.contiguous().pin_memory()
    tickets = []
    for i in range(2):
        tk = C.c_int32()
        _lib.check(lib.sm_track_host_async(m.handle, 0, B, xs[i].data_ptr(), outs[i][0].data_ptr(),
                                           outs[i][1].data_ptr(), posh.data_ptr(), outs[i][2].data_ptr(), st, C.byref(tk)))
        tickets.append(tk.value)
    for i in range(2):
        _lib.check(lib.sm_track_host_wait(m.handle, tickets[i]))
        for got, r, n in zip(outs[i], want[i], ("cls", "loc", "refine")):
            assert_close(got, r, 1e-6, f"two-lane host path {n} step {i}")


def test_search_383_response_41(calib_sd):
    g = {k: torch.from_numpy(v) for k, v in np.load(os.path.join(GOLDEN, "rpn_b1_s383.npz")).items()}
    z, x = synthetic_inputs(3, 1, search=383)
    m = _engine(calib_sd, search_size=383)
    m.template(z.cuda())
    cls, loc = m.track(x.cuda())
    assert cls.shape == (1, 10, 41, 41) and loc.shape == (1, 20, 41, 41)
    o = Oracle(calib_sd)
    o.template(z)
    ocls, oloc = o.track(x)
    assert_close(cls, ocls, TOL, "cls @383")
    assert_close(loc, oloc, TOL, "loc @383")
    assert_close(cls, g["cls"], 2e-3, "cls @383 vs reference golden")


def test_rpn_only_engine(calib_sd):
    """experiments/siamrpn_resnet: same backbone + cls/loc, no mask/refine weights needed."""
    sd = {k: v for k, v in calib_sd.items() if not k.startswith(("mask_model", "refine_model"))}
    z, x = synthetic_inputs(2, 2)
    m = _engine(sd, mask=False, max_batch=2)
    m.template(z.cuda())
    cls, loc = m.track(x.cuda())
    o = Oracle(calib_sd)
    o.template(z)
    ocls, oloc = o.track(x)
    assert_close(cls, ocls, TOL, "rpn-only cls")
    assert_close(loc, oloc, TOL, "rpn-only loc")
    with pytest.raises(RuntimeError):
        m.track_mask(x.cuda())


def test_fast_mode_tracks_fp16_model(calib_sd):
    """Single-pass fp16: checked against the oracle's fp16 emulation of the same rounding points is out of
    scope here; against fp32 it must stay within the error the emulation predicts (a few 1e-2 on this
    chaotic seeded net) — guards against gross errors only.  The parity mode is 'exact'."""
    z, x = synthetic_inputs(1, 1)
    o = Oracle(calib_sd)
    o.template(z)
    ocls, oloc, _ = o.track_mask(x, with_mask_head=False)
    m = _engine(calib_sd, precision="fast")
    m.template(z.cuda())
    cls, loc, _ = m.track_mask(x.cuda(), mask_head=False)
    assert_close(cls, ocls, 0.25, "fast cls")
    assert_close(loc, oloc, 0.25, "fast loc")


def test_errors_are_loud(calib_sd):
    m = _engine(calib_sd)
    with pytest.raises(ValueError):
        m.track(torch.zeros(2, 3, 255, 255).cuda())          # batch > max_batch
    with pytest.raises(ValueError):
        m.track(torch.zeros(1, 3, 200, 200).cuda())          # wrong search size
    z, x = synthetic_inputs(1, 1)
    m.template(z.cuda())
    m.track(x.cuda())
    with pytest.raises(RuntimeError):
        m.track_refine((1, 1))                                # refine without track_mask features
    m.track_mask(x.cuda())
    with pytest.raises(IndexError):
        m.track_refine((25, 0))


def test_graph_replay_matches_eager(calib_sd):
    """CUDA-graph replay (sm_engine_set_graphs): call 1 eager, call 2 captured, calls 3+ replayed — same results,
    fresh inputs are honoured (persistent staging buffers), refine positions too."""
    z, x = synthetic_inputs(41, 2)
    _, x2 = synthetic_inputs(42, 2)
    eager = _engine(calib_sd, max_batch=2)
    eager.template(z.cuda())
    g = _engine(calib_sd, max_batch=2, graphs=True)
    g.template(z.cuda())
    for it, xin in enumerate([x, x2, x, x2, x]):
        ce, le, _ = eager.track_mask(xin.cuda(), mask_head=False)
        cg, lg, _ = g.track_mask(xin.cuda(), mask_head=False)
        pos = np.array([[3 + it, 5], [20, 2 + it]])
        re_, rg = eager.track_refine(pos), g.track_refine(pos)
        assert_close(cg, ce, 1e-6, f"graph cls call {it}")
        assert_close(lg, le, 1e-6, f"graph loc call {it}")
        assert_close(rg, re_, 1e-6, f"graph refine call {it}")
    assert g.launch_count == eager.launch_count


def test_host_buffer_path_sync_and_async(calib_sd):
    """sm_track_host (synchronous) and the pipelined sm_track_host_async / _wait pair deliver the same results as
    the device-pointer API."""
    import ctypes as C
    from siammask_b200 import _lib
    lib = _lib.load()
    z, x = synthetic_inputs(51, 2)
    _, x2 = synthetic_inputs(52, 2)
    m = _engine(calib_sd, max_batch=2)
    m.template(z.cuda())
    pos = torch.tensor([[4, 9], [17, 3]], dtype=torch.int32)
    want = []
    for xin in (x, x2):
        cls, loc, _ = m.track_mask(xin.cuda(), mask_head=False)
        want.append((cls.cpu(), loc.cpu(), m.track_refine(pos.cuda()).cpu()))
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    xs = [x.contiguous().pin_memory(), x2.contiguous().pin_memory()]
    outs = [(torch.empty(2, 10, 25, 25).pin_memory(), torch.empty(2, 20, 25, 25).pin_memory(),
             torch.empty(2, 127 * 127).pin_memory()) for _ in range(2)]
    posh = pos.contiguous().pin_memory()
    # synchronous
    for i in range(2):
        _lib.check(lib.sm_track_host(m.handle, 0, 2, xs[i].data_ptr(), outs[i][0].data_ptr(), outs[i][1].data_ptr(),
                                     posh.data_ptr(), outs[i][2].data_ptr(), st))
        for got, ref, n in zip(outs[i], want[i], ("cls", "loc", "refine")):
            assert_close(got, ref, 1e-6, f"sync host path {n} step {i}")
    # pipelined: submit both steps, then collect
    for o in outs:
        for t in o:
            t.zero_()
    tickets = []
    for i in range(2):
        tk = C.c_int32()
        _lib.check(lib.sm_track_host_async(m.handle, 0, 2, xs[i].data_ptr(), outs[i][0].data_ptr(),
                                           outs[i][1].data_ptr(), posh.data_ptr(), outs[i][2].data_ptr(), st, C.byref(tk)))
        tickets.append(tk.value)
    assert tickets == [0, 1] or tickets == [1, 0]
    for i in range(2):
        _lib.check(lib.sm_track_host_wait(m.handle, tickets[i]))
        for got, ref, n in zip(outs[i], want[i], ("cls", "loc", "refine")):
            assert_close(got, ref, 1e-6, f"async host path {n} step {i}")


def test_packed_weight_file_roundtrip(calib_sd, tmp_path):
    """save_packed / load_packed: an engine that never saw the checkpoint reproduces the packing engine bit for bit."""
    z, x = synthetic_inputs(61, 1)
    a = _engine(calib_sd)
    path = str(tmp_path / "weights.smb")
    a.save_packed(path)
    b = smb.Custom(anchors=smb.DEFAULT_ANCHORS).eval().to("cuda")
    with pytest.raises(RuntimeError):
        b.template(z.cuda())                       # no weights yet: loud failure
    b.load_packed(path)
    outs = []
    for m in (a, b):
        m.template(z.cuda())
        cls, loc, _ = m.track_mask(x.cuda(), mask_head=False)
        outs.append((cls.clone(), loc.clone(), m.track_refine((7, 11)).clone()))
    for u, v in zip(*outs):
        assert torch.equal(u, v)
    c = smb.Custom(anchors=smb.DEFAULT_ANCHORS, mask=False).eval().to("cuda")
    with pytest.raises(ValueError):
        c.load_packed(path)                        # RPN-only engine has a different arena layout


@pytest.mark.parametrize("seed,kind", [(101, "noise"), (202, "noise"), (303, "smooth"), (404, "smooth")])
def test_parity_holds_across_inputs(calib_sd, seed, kind):
    """1e-3 parity is not an accident of one input: other noise seeds and image-like (low-pass) crops."""
    g = torch.Generator().manual_seed(seed)
    if kind == "noise":
        z = torch.rand(1, 3, 127, 127, generator=g) * 255
        x = torch.rand(1, 3, 255, 255, generator=g) * 255
    else:   # smooth structure: upsampled coarse noise + a little fine noise, clipped to the pixel range
        def img(n):
            coarse = torch.rand(1, 3, n // 16 + 2, n // 16 + 2, generator=g)
            fine = torch.rand(1, 3, n, n, generator=g)
            up = torch.nn.functional.interpolate(coarse, size=(n, n), mode="bilinear", align_corners=False)
            return ((0.85 * up + 0.15 * fine) * 255).clamp(0, 255).round()
        z, x = img(127), img(255)
    o = Oracle(calib_sd)
    o.template(z)
    ocls, oloc, _ = o.track_mask(x, with_mask_head=False)
    m = _engine(calib_sd)
    m.template(z.cuda())
    cls, loc, _ = m.track_mask(x.cuda(), mask_head=False)
    assert_close(cls, ocls, TOL, f"cls seed {seed} {kind}")
    assert_close(loc, oloc, TOL, f"loc seed {seed} {kind}")
    assert_close(m.track_refine((9, 14)), o.track_refine((9, 14)), TOL, f"refine seed {seed} {kind}")
