"""Pin the oracle (and the host-side image utilities) to the reference on BASELINE.json's config[0] and on the
branches the round-1 cases never take: the chunked complete_flow / image_propagation halos and the ref_num window
schedule (T > subvideo_length), the Outpaint node, 20 RAFT iterations at 640x360.  Fixtures:
tests/golden/reference_outputs_r2.npz, generated from the unmodified reference by tests/golden/make_golden_r2.py;
large outputs are compared at the fixture's sampled pixels.  CPU only, fp32."""
import numpy as np
import torch

from comfyui_propainter_nodes_b200 import weights as Wt
from comfyui_propainter_nodes_b200.utils import image_utils as IU
from oracle import propainter_oracle as O
from tests.golden import cases

SDS = None


def _sds():
    global SDS
    if SDS is None:
        SDS = (Wt.synthetic_raft_state_dict(), Wt.synthetic_rfc_state_dict(), Wt.synthetic_generator_state_dict())
    return SDS


def _max_diff(golden2, k, a):
    """max |a - reference| over the fixture's pixels of `k` (float16 fixtures compared in float32)."""
    return float(np.abs(golden2.pick(k, a).astype(np.float32) - golden2[k].astype(np.float32)).max())


def _u8_close(golden2, k, out, frac=2e-3):
    out, ref = golden2.pick(k, np.asarray(out)).astype(np.int32), golden2[k].astype(np.int32)
    bad = (np.abs(out - ref) > 1).mean()
    assert bad < frac, bad


def test_config1_inpaint_node_path(golden2):
    """BASELINE config[0]: 16 frames 320x180 -> 320x176 (PIL bicubic), raft_iter=5, fp32."""
    c = cases.c1_case()
    kw = c["kwargs"]
    T, H, W = c["image"].shape[:3]
    icfg = IU.ImageConfig(kw["width"], kw["height"], kw["mask_dilates"], kw["flow_mask_dilates"], (W, H), T)
    assert tuple(icfg.process_size) == (320, 176)
    ft, fm, md, orig = IU.prepare_frames_and_masks(IU.convert_image_to_frames(c["image"]), c["mask"], icfg,
                                                   torch.device("cpu"))
    assert np.array_equal((fm[0, :, 0].numpy() * 255).astype(np.uint8), golden2["c1_flow_masks_u8"])
    assert np.array_equal((md[0, :, 0].numpy() * 255).astype(np.uint8), golden2["c1_masks_dilated_u8"])
    comp, st = O.run_pipeline(*_sds(), ft, fm, md, orig, raft_iter=kw["raft_iter"],
                              subvideo_length=kw["subvideo_length"], neighbor_length=kw["neighbor_length"],
                              ref_stride=kw["ref_stride"], return_stages=True)
    d = _max_diff(golden2, "c1_gt_flow_f_s2", st["gt_flows"][0][..., ::2, ::2])
    assert d < 1e-2, d                      # float16 storage of the fixture: ulp 0.004 below 8 px
    d = _max_diff(golden2, "c1_pred_flow_f", st["pred_flows"][0])
    assert d < 1e-2, d
    assert np.array_equal((st["updated_masks"].numpy() * 255).astype(np.uint8), golden2["c1_updated_masks_u8"])
    _u8_close(golden2, "c1_image_u8", np.stack(comp))


def test_raft_20_iterations_640x360(golden2):
    fr = cases.raft20_case()
    for tag, gain in cases.RAFT20_GAINS.items():
        sd = O.strip_module_prefix(Wt.synthetic_raft_state_dict(flow_head_gain=gain))
        with torch.no_grad():
            _, trace = O.raft_pairs(sd, fr[0, :-1], fr[0, 1:], max(cases.RAFT20_ITERS), return_trace=True)
        for it in cases.RAFT20_ITERS:
            d = _max_diff(golden2, f"raft20_{tag}_it{it}_s4", trace[it - 1][:, :, ::4, ::4])
            assert d < 2e-2, (tag, it, d)


def test_chunked_clip_halos_and_ref_num(golden2):
    e = cases.chunked_case()
    assert e["T"] > e["subvideo_length"]
    icfg = IU.ImageConfig(e["W"], e["H"], 5, 8, (e["W"], e["H"]), e["T"])
    ft, fm, md, orig = IU.prepare_frames_and_masks(IU.convert_image_to_frames(e["image"]), e["mask"], icfg,
                                                   torch.device("cpu"))
    comp, st = O.run_pipeline(*_sds(), ft, fm, md, orig, raft_iter=e["raft_iter"], subvideo_length=e["subvideo_length"],
                              neighbor_length=e["neighbor_length"], ref_stride=e["ref_stride"], return_stages=True)
    for k, i in (("chunk_pred_flow_f", 0), ("chunk_pred_flow_b", 1)):
        d = _max_diff(golden2, k, st["pred_flows"][i])
        assert d < 1e-2, (k, d)
    um = (st["updated_masks"].numpy() * 255).astype(np.uint8)
    assert (um != golden2["chunk_updated_masks_u8"]).mean() < 1e-4
    _u8_close(golden2, "chunk_frames_u8", np.stack(comp))
    # the schedule itself: windows of a long clip use <= ref_num + 1 references around the window
    sched = O.window_schedule(e["T"], e["neighbor_length"], e["ref_stride"], e["subvideo_length"])
    assert max(len(r) for _, r in sched) <= e["subvideo_length"] // e["ref_stride"] + 1
    assert any(len(r) > 0 for _, r in sched)


def test_outpaint_node_path(golden2):
    o = cases.outpaint_case()
    kw = o["kwargs"]
    T, H, W = o["image"].shape[:3]
    icfg = IU.ImageOutpaintConfig(kw["width"], kw["height"], kw["mask_dilates"], kw["flow_mask_dilates"], (W, H), T,
                                  kw["width_scale"], kw["height_scale"])
    assert list(icfg.outpaint_size) == list(golden2["outpaint_size"])
    canvas, fmk, mdl = IU.extrapolation(IU.convert_image_to_frames(o["image"]), icfg)
    ft, fm, md, orig = IU.prepare_frames_and_masks_for_outpaint(canvas, fmk, mdl, torch.device("cpu"))
    assert np.array_equal((fm[0, :, 0].numpy() * 255).astype(np.uint8), golden2["outpaint_mask_u8"])
    comp, st = O.run_pipeline(*_sds(), ft, fm, md, orig, raft_iter=kw["raft_iter"],
                              subvideo_length=kw["subvideo_length"], neighbor_length=kw["neighbor_length"],
                              ref_stride=kw["ref_stride"], return_stages=True)
    d = _max_diff(golden2, "outpaint_pred_flow_f", st["pred_flows"][0])
    assert d < 1e-2, d
    _u8_close(golden2, "outpaint_image_u8", np.stack(comp))
