"""Pin oracle/propainter_oracle.py to outputs of the REAL reference (tests/golden/reference_outputs.npz).

The fixtures were produced by tests/golden/make_golden.py, which imports the unmodified reference;
inputs are regenerated from seeds here and outputs compared at the fixture's sampled pixels.  CPU only, fp32.
"""
import numpy as np
import torch

from comfyui_propainter_nodes_b200 import weights as Wt
from comfyui_propainter_nodes_b200.utils import image_utils as IU
from oracle import propainter_oracle as O
from tests.golden import cases


def _close(golden, k, a, atol):
    a, ref = golden.pick(k, a), golden[k]          # pick() checks the full shape
    err = np.abs(a.astype(np.float64) - ref.astype(np.float64)).max()
    assert err <= atol, f"{k}: max abs err {err} > {atol}"


def test_raft_matches_reference(golden):
    with torch.no_grad():
        ff, fb = O.raft_bidirectional(Wt.synthetic_raft_state_dict(), cases.raft_case(), cases.RAFT_ITERS)
    _close(golden, "raft_ff", ff, 2e-3)
    _close(golden, "raft_fb", fb, 2e-3)


def test_flow_completion_matches_reference(golden):
    flows, masks = cases.rfc_case()
    with torch.no_grad():
        f, b = O.rfc_bidirectional(Wt.synthetic_rfc_state_dict(), flows, masks)
    _close(golden, "rfc_f", f, 1e-3)
    _close(golden, "rfc_b", b, 1e-3)


def test_image_propagation_matches_reference(golden):
    frames, m, fl = cases.imgprop_case()
    with torch.no_grad():
        uf, um = O.image_propagation(frames, m, fl, 80)
    _close(golden, "imgprop_frames", uf, 1e-6)
    _close(golden, "imgprop_masks", um, 0)


def test_generator_window_matches_reference(golden):
    g = cases.window_case()
    with torch.no_grad():
        pred = O.inpaint_window(Wt.synthetic_generator_state_dict(), g["frames"], g["flows"], g["masks_in"],
                                g["masks_upd"], g["l_t"])
    _close(golden, "window_pred", pred, 1e-3)


def test_end_to_end_matches_reference(golden):
    e = cases.e2e_case()
    cfg = IU.ImageConfig(e["W"], e["H"], 5, 8, (e["W"], e["H"]), e["T"])
    frames_u8 = IU.convert_image_to_frames(e["image"])
    ft, fm, md, orig = IU.prepare_frames_and_masks(frames_u8, e["mask"], cfg, torch.device("cpu"))
    _close(golden, "e2e_flow_masks", fm, 0)
    _close(golden, "e2e_masks_dilated", md, 0)
    comp, st = O.run_pipeline(Wt.synthetic_raft_state_dict(), Wt.synthetic_rfc_state_dict(),
                              Wt.synthetic_generator_state_dict(), ft, fm, md, orig,
                              raft_iter=e["raft_iter"], subvideo_length=e["subvideo_length"],
                              neighbor_length=e["neighbor_length"], ref_stride=e["ref_stride"],
                              return_stages=True)
    _close(golden, "e2e_pred_flow_f", st["pred_flows"][0], 5e-3)
    # nearest-neighbour propagation may flip single pixels when a coordinate lands on .5 +- 1 ulp
    d = np.abs(golden.pick("e2e_updated_frames", st["updated_frames"]) - golden["e2e_updated_frames"])
    assert (d > 1e-4).mean() < 1e-3
    out = golden.pick("e2e_frames_u8", np.stack(comp)).astype(np.int32)
    ref = golden["e2e_frames_u8"].astype(np.int32)
    assert (np.abs(out - ref) > 1).mean() < 2e-3, (np.abs(out - ref) > 1).mean()


def test_window_schedule_defaults():
    """80 frames, defaults: 16 windows, sum(t) = 275, sum(l_t) = 170 (SURVEY.md section 3E)."""
    s = O.window_schedule(80, 10, 10, 80)
    assert len(s) == 16
    assert sum(len(a) + len(b) for a, b in s) == 275
    assert sum(len(a) for a, _ in s) == 170
    # long video: references limited to ref_num=8 within +-40 frames, up to 9 (quirk 17)
    s = O.window_schedule(240, 10, 10, 80)
    assert len(s) == 48 and max(len(b) for _, b in s) <= 9
