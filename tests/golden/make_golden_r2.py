"""Round-2 golden fixtures: the reference run on BASELINE.json's configs and on the branches the round-1 cases
never take (tests/golden/reference_outputs_r2.npz).  Needs a checkout of the reference, CPU:

    python tests/golden/make_golden_r2.py PATH/TO/ComfyUI_ProPainter_Nodes

Like make_golden.py it imports the UNMODIFIED reference (stub ``comfy.model_management``); the two node classes are
called through their own ``propainter_inpainting`` / ``propainter_outpainting`` methods with
``initialize_models`` (which downloads checkpoints) replaced by a function returning the reference's own modules
loaded with the seeded synthetic checkpoints.  Inputs are regenerated from seeds by the tests; only reference
OUTPUTS are stored (float32 samples for the RAFT error-growth case, float16 for the other flows -- their
tolerances are >= 0.02 px and a float16 ulp below 8 px is <= 0.004 px --, uint8 for frames and masks).  Masks and
small arrays are stored whole, frames and flows as fixed samples of their pixels (tests/golden/sampled.py, SPEC below).
"""
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as MG  # noqa: E402

import numpy as np  # noqa: E402
import torch  # noqa: E402

from comfyui_propainter_nodes_b200 import weights as Wt  # noqa: E402
from tests.golden import cases, sampled  # noqa: E402

# sampled arrays: name -> (channel axis, positions); every other output is stored whole
SPEC = {"c1_image_u8": (3, 4096), "c1_gt_flow_f_s2": (2, 2048), "c1_pred_flow_f": (2, 2048),
        "chunk_gt_flow_f_s2": (2, 1024), "chunk_pred_flow_f": (2, 2048), "chunk_pred_flow_b": (2, 2048),
        "chunk_frames_u8": (3, 4096), "outpaint_image_u8": (3, 4096), "outpaint_pred_flow_f": (2, 1024)}
for _tag in cases.RAFT20_GAINS:
    SPEC.update({f"raft20_{_tag}_it{it}_s4": (1, 512) for it in cases.RAFT20_ITERS})
    SPEC[f"raft20_{_tag}_final_s2"] = (1, 1024)


def main(reference_dir):
    MG.load_reference(reference_dir)
    from reference import propainter_nodes as RN
    from reference import propainter_inference as RI
    from reference.utils import image_utils as RU
    from reference.utils.model_utils import Models
    from reference.model.modules.flow_comp_raft import RAFT_bi
    torch.manual_seed(0)
    torch.set_num_threads(min(16, os.cpu_count() or 1))
    raft, rfc, gen = MG.build_models()
    models = Models(raft, rfc, gen)
    RN.initialize_models = lambda device, fp16: models
    # stage taps: the node's own calls, recorded on the way through
    taps = {}
    orig_pi, orig_cf = RI.process_inpainting, RI.compute_flow

    def tap_process(m, frames, fm, md, cfg):
        out = orig_pi(m, frames, fm, md, cfg)
        taps["updated_frames"], taps["updated_masks"], taps["pred_flows"] = out
        taps["flow_masks"], taps["masks_dilated"] = fm, md
        return out

    def tap_flow(m, frames, cfg):
        out = orig_cf(m, frames, cfg)
        taps["gt_flows"] = out
        return out

    RN.process_inpainting = tap_process
    RI.compute_flow = tap_flow
    out = {}
    u8 = lambda t: (t.detach().cpu().float().numpy() * 255.0 + 0.5).astype(np.uint8)
    with torch.no_grad():
        # ---- (a) BASELINE config[0] through the Inpaint node
        t0 = time.time()
        c = cases.c1_case()
        img, fmask, dmask = RN.ProPainterInpaint().propainter_inpainting(c["image"], c["mask"], **c["kwargs"])
        out["c1_image_u8"] = u8(img)                      # handle_output: uint8 / 255 -> exact after *255 + .5
        out["c1_flow_masks_u8"], out["c1_masks_dilated_u8"] = u8(fmask), u8(dmask)
        out["c1_gt_flow_f_s2"] = taps["gt_flows"][0][..., ::2, ::2].half()     # RAFT flow, every 2nd pixel
        out["c1_pred_flow_f"] = taps["pred_flows"][0].half()
        out["c1_updated_masks_u8"] = u8(taps["updated_masks"])
        print(f"c1 node: {time.time() - t0:.1f} s", flush=True)

        # ---- (b) RAFT at 640x360, 20 iterations, damped (bench weights) and un-damped flow head
        fr = cases.raft20_case()
        for tag, gain in cases.RAFT20_GAINS.items():
            t0 = time.time()
            import tempfile
            p = os.path.join(tempfile.mkdtemp(), "raft.pth")
            torch.save(Wt.synthetic_raft_state_dict(flow_head_gain=gain), p)
            net = RAFT_bi(p, "cpu").fix_raft
            preds = net(fr[0, :-1], fr[0, 1:], iters=max(cases.RAFT20_ITERS), test_mode=False)
            for it in cases.RAFT20_ITERS:
                out[f"raft20_{tag}_it{it}_s4"] = preds[it - 1][:, :, ::4, ::4]   # every 4th pixel of flow_up
            out[f"raft20_{tag}_final_s2"] = preds[-1][:, :, ::2, ::2]
            # sensitivity of the fp32 reference itself: the same network on input frames rounded to fp16 (a relative
            # perturbation <= 4.9e-4, applied ONCE).  With random weights the 20-step recursion amplifies any
            # perturbation; this is the yardstick the fp16 engine (which rounds at every layer) is measured against.
            frh = fr.half().float()
            pert = net(frh[0, :-1], frh[0, 1:], iters=max(cases.RAFT20_ITERS), test_mode=False)
            sens = [[float((preds[it - 1] - pert[it - 1]).abs().mean()), float((preds[it - 1] - pert[it - 1]).abs().max())]
                    for it in cases.RAFT20_ITERS]
            out[f"raft20_{tag}_sens"] = torch.tensor(sens)       # [iteration][mean, max] in px
            print(f"raft20 {tag}: {time.time() - t0:.1f} s, |flow| mean {float(preds[-1].abs().mean()):.3f} "
                  f"max {float(preds[-1].abs().max()):.3f}", flush=True)

        # ---- (c) chunked clip: T=30 > subvideo_length=12
        t0 = time.time()
        e = cases.chunked_case()
        icfg = RU.ImageConfig(e["W"], e["H"], 5, 8, (e["W"], e["H"]), e["T"])
        ft, fm, md, orig = RU.prepare_frames_and_masks(RU.convert_image_to_frames(e["image"]), e["mask"], icfg,
                                                       torch.device("cpu"))
        pcfg = RI.ProPainterConfig(e["ref_stride"], e["neighbor_length"], e["subvideo_length"], e["raft_iter"],
                                   "disable", e["T"], torch.device("cpu"), icfg.process_size)
        uf, um, pf = orig_pi(models, ft, fm, md, pcfg)
        comp = RI.feature_propagation(gen, uf, um, md, pf, orig, pcfg)
        out["chunk_gt_flow_f_s2"] = taps["gt_flows"][0][..., ::2, ::2].half()
        out["chunk_pred_flow_f"], out["chunk_pred_flow_b"] = pf[0].half(), pf[1].half()
        out["chunk_updated_masks_u8"] = u8(um)
        out["chunk_frames_u8"] = torch.from_numpy(np.stack(comp))
        print(f"chunked: {time.time() - t0:.1f} s", flush=True)

        # ---- (d) Outpaint node (also the token grid padded in both axes)
        t0 = time.time()
        o = cases.outpaint_case()
        img, omask, ow, oh = RN.ProPainterOutpaint().propainter_outpainting(o["image"], **o["kwargs"])
        out["outpaint_image_u8"] = u8(img)
        out["outpaint_mask_u8"] = u8(omask)
        out["outpaint_size"] = torch.tensor([ow, oh])
        out["outpaint_pred_flow_f"] = taps["pred_flows"][0].half()
        print(f"outpaint node: {time.time() - t0:.1f} s -> {ow}x{oh}", flush=True)

    store = {}
    for k, v in out.items():
        a = v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)
        store[k] = a
    np.savez_compressed(os.path.join(HERE, "reference_outputs_r2.npz"), **sampled.shrink(store, SPEC))
    for k, v in store.items():
        print(k, v.shape, v.dtype, float(np.abs(v.astype(np.float64)).mean()))


if __name__ == "__main__":
    main(sys.argv[1])
