"""Generate the golden fixtures that pin oracle/propainter_oracle.py to the REAL reference.

Needs a checkout of the reference (ComfyUI_ProPainter_Nodes); runs on the CPU:

    python tests/golden/make_golden.py PATH/TO/ComfyUI_ProPainter_Nodes

It imports the unmodified reference package with a stub ``comfy.model_management``, loads the seeded
synthetic checkpoints from comfyui_propainter_nodes_b200.weights into the reference's own modules
(strict=True) and stores per-stage outputs as float32 / uint8 in an .npz file: masks whole, the large
arrays as fixed samples of their pixels (tests/golden/sampled.py, SPEC below).
Inputs are regenerated from seeds by the tests; only reference OUTPUTS are stored.
"""
import importlib.util
import os
import sys
import types
import tempfile

os.environ["PYTHONDONTWRITEBYTECODE"] = "1"
sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from comfyui_propainter_nodes_b200 import weights as Wt  # noqa: E402
from tests.golden import cases, sampled  # noqa: E402

# sampled arrays: name -> (channel axis, positions); every other output is stored whole
SPEC = {"raft_ff": (2, 1024), "raft_fb": (2, 1024), "rfc_f": (2, 1024), "rfc_b": (2, 1024),
        "imgprop_frames": (2, 2048), "window_pred": (2, 1024), "e2e_updated_frames": (2, 2048),
        "e2e_pred_flow_f": (2, 1024), "e2e_frames_u8": (3, 4096)}


def load_reference(path):
    """Import the reference checkout at `path` as the package ``reference``, with a stub ``comfy.model_management``
    (the one ComfyUI module it imports)."""
    comfy = types.ModuleType("comfy")
    mm = types.ModuleType("comfy.model_management")
    mm.get_torch_device = lambda: torch.device("cpu")
    comfy.model_management = mm
    sys.modules["comfy"] = comfy
    sys.modules["comfy.model_management"] = mm
    path = os.path.abspath(path)
    spec = importlib.util.spec_from_file_location("reference", os.path.join(path, "__init__.py"),
                                                  submodule_search_locations=[path])
    mod = importlib.util.module_from_spec(spec)
    sys.modules["reference"] = mod
    spec.loader.exec_module(mod)


def build_models():
    from reference.model.modules.flow_comp_raft import RAFT_bi
    from reference.model.recurrent_flow_completion import RecurrentFlowCompleteNet
    from reference.model.propainter import InpaintGenerator
    tmp = tempfile.mkdtemp()
    rp = os.path.join(tmp, "raft.pth")
    torch.save(Wt.synthetic_raft_state_dict(), rp)
    raft = RAFT_bi(rp, "cpu")
    rfc = RecurrentFlowCompleteNet()
    rfc.load_state_dict(Wt.synthetic_rfc_state_dict(), strict=True)
    rfc.eval()
    gen = InpaintGenerator()
    gen.load_state_dict(Wt.synthetic_generator_state_dict(), strict=True)
    gen.eval()
    return raft, rfc, gen


def main(reference_dir):
    load_reference(reference_dir)
    from reference import propainter_inference as RI
    from reference.utils import image_utils as RU
    from reference.utils.model_utils import Models
    torch.manual_seed(0)
    torch.set_num_threads(8)
    raft, rfc, gen = build_models()
    out = {}
    with torch.no_grad():
        # ---- RAFT
        fr = cases.raft_case()
        ff, fb = raft(fr, iters=cases.RAFT_ITERS)
        out["raft_ff"], out["raft_fb"] = ff, fb
        # ---- flow completion
        flows, masks = cases.rfc_case()
        pred, _ = rfc.forward_bidirect_flow(flows, masks)
        comb = rfc.combine_flow(flows, pred, masks)
        out["rfc_f"], out["rfc_b"] = comb
        # ---- image propagation
        frames, m, fl = cases.imgprop_case()
        cfg = RI.ProPainterConfig(10, 10, 80, 5, "disable", frames.shape[1], torch.device("cpu"),
                                  (frames.shape[-1], frames.shape[-2]))
        uf, um = RI.image_propagation(gen, frames, m, fl, cfg)
        out["imgprop_frames"], out["imgprop_masks"] = uf, um
        # ---- generator window
        g = cases.window_case()
        pred_img = gen(g["frames"], g["flows"], g["masks_in"], g["masks_upd"], g["l_t"])
        out["window_pred"] = pred_img
        # ---- end-to-end through the reference node-level functions
        e = cases.e2e_case()
        icfg = RU.ImageConfig(e["W"], e["H"], 5, 8, (e["W"], e["H"]), e["T"])
        frames_pil = RU.convert_image_to_frames(e["image"])
        ft, fm, md, orig = RU.prepare_frames_and_masks(frames_pil, e["mask"], icfg, torch.device("cpu"))
        out["e2e_flow_masks"], out["e2e_masks_dilated"] = fm, md
        pcfg = RI.ProPainterConfig(e["ref_stride"], e["neighbor_length"], e["subvideo_length"], e["raft_iter"],
                                   "disable", e["T"], torch.device("cpu"), icfg.process_size)
        models = Models(raft, rfc, gen)
        uf, um, pf = RI.process_inpainting(models, ft, fm, md, pcfg)
        comp = RI.feature_propagation(gen, uf, um, md, pf, orig, pcfg)
        out["e2e_updated_frames"] = uf
        out["e2e_pred_flow_f"] = pf[0]
        out["e2e_frames_u8"] = torch.from_numpy(np.stack(comp))
    store = {}
    for k, v in out.items():
        a = v.detach().cpu().numpy()
        store[k] = a if a.dtype == np.uint8 else a.astype(np.float32)
    np.savez_compressed(os.path.join(HERE, "reference_outputs.npz"), **sampled.shrink(store, SPEC))
    for k, v in store.items():
        print(k, v.shape, v.dtype, float(np.abs(v.astype(np.float64)).mean()))


if __name__ == "__main__":
    main(sys.argv[1])
