"""GPU parity checks shared by the pytest -m gpu tests and the diagnostic report (python -m tests.gpu_checks).

Every check returns a dict of error statistics of the CUDA path (through the C ABI) against the CPU oracle
or a plain PyTorch fp32 evaluation of the same operator on the same fp16-rounded inputs."""
import math
import sys
import time
import traceback

import numpy as np
import torch
import torch.nn.functional as F

from comfyui_propainter_nodes_b200 import engine as E
from comfyui_propainter_nodes_b200 import weights as Wt
from comfyui_propainter_nodes_b200 import propainter_inference as PI
from comfyui_propainter_nodes_b200.utils import image_utils as IU
from comfyui_propainter_nodes_b200.utils.model_utils import Models, StageHandle
from oracle import propainter_oracle as O
from tests.golden import cases
from tests.golden.sampled import Golden

DEV = "cuda:0"
_ENG = {}


def bare_engine():
    if "bare" not in _ENG:
        _ENG["bare"] = E.Engine(DEV, workspace_gb=2.0)
    return _ENG["bare"]


def full_models():
    if "full" not in _ENG:
        eng = E.Engine(DEV, workspace_gb=16.0).load_weights(Wt.synthetic_raft_state_dict(), Wt.synthetic_rfc_state_dict(),
                                                           Wt.synthetic_generator_state_dict())
        _ENG["full"] = Models(StageHandle(eng, "raft"), StageHandle(eng, "flow"), StageHandle(eng, "inpaint"))
    return _ENG["full"]


def stats(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    d = (a - b).abs()
    return dict(max_abs=float(d.max()), mean_abs=float(d.mean()), ref_mean_abs=float(b.abs().mean()),
                rel=float(d.max() / (b.abs().max() + 1e-12)), nan=bool(torch.isnan(a).any()))


def stats_at(golden, k, a):
    """stats() of the full output `a` against the reference fixture `k`, at the fixture's pixels."""
    return stats(torch.from_numpy(golden.pick(k, a)), torch.from_numpy(golden[k]))


# ------------------------------------------------------------------------------------------------ conv
CONV_CASES = {
    # name: (N, H, W, Cin_ref, Cout, kh, kw, stride, pad, dil, groups, replicate, act, slope, residual, cin_pad_to)
    "linear_512_1536": (1, 1, 1000, 512, 1536, 1, 1, 1, 0, 1, 1, 0, E.ACT_NONE, 0.0, False, None),
    "conv3x3_128_128_lrelu_res": (2, 45, 80, 128, 128, 3, 3, 1, 1, 1, 1, 0, E.ACT_LRELU, 0.2, True, None),
    "conv7x7_s2_3_64": (2, 64, 96, 3, 64, 7, 7, 2, 3, 1, 1, 0, E.ACT_RELU, 0.0, False, 8),
    "conv3x3_dil3": (1, 45, 80, 128, 128, 3, 3, 1, 3, 3, 1, 0, E.ACT_LRELU, 0.2, False, None),
    "conv5x5_s2_replicate": (2, 64, 96, 3, 32, 5, 5, 2, 2, 1, 1, 1, E.ACT_LRELU, 0.2, False, 8),
    "grouped_g4": (1, 30, 40, 768, 384, 3, 3, 1, 1, 1, 4, 0, E.ACT_LRELU, 0.2, False, None),
    "cout2": (1, 64, 96, 32, 2, 3, 3, 1, 1, 1, 1, 0, E.ACT_NONE, 0.0, False, None),
    "cout126": (1, 45, 80, 256, 126, 3, 3, 1, 1, 1, 1, 0, E.ACT_RELU, 0.0, False, None),
    "cout432": (1, 45, 80, 128, 432, 3, 3, 1, 1, 1, 1, 0, E.ACT_NONE, 0.0, False, None),
    "cin261": (1, 44, 80, 261, 128, 3, 3, 1, 1, 1, 1, 0, E.ACT_LRELU, 0.1, False, 264),
    "conv7x7_s3_40_512": (2, 44, 80, 40, 512, 7, 7, 3, 3, 1, 1, 0, E.ACT_NONE, 0.0, True, None),
    "conv1x5": (1, 45, 80, 384, 256, 1, 5, 1, (0, 2), 1, 1, 0, E.ACT_SIGMOID, 0.0, False, None),
    "conv5x1_tanh": (1, 45, 80, 384, 128, 5, 1, 1, (2, 0), 1, 1, 0, E.ACT_TANH, 0.0, False, None),
    "k2304": (1, 45, 80, 2304, 128, 1, 1, 1, 0, 1, 1, 0, E.ACT_NONE, 0.0, False, None),
    # TMA halo-tile kernel (conv_halo.cu): 16x16 tiles (MT=2), odd sizes with MT=1 + narrowed N tiles, two N tiles
    "halo_mt2_64_64": (3, 90, 160, 64, 64, 3, 3, 1, 1, 1, 1, 0, E.ACT_LRELU, 0.2, True, None),
    "halo_odd_size": (2, 37, 53, 192, 96, 3, 3, 1, 1, 1, 1, 0, E.ACT_RELU, 0.0, False, None),
    "halo_mt2_256_192": (8, 45, 80, 256, 192, 3, 3, 1, 1, 1, 1, 0, E.ACT_NONE, 0.0, True, None),
    "halo_flat_328_256": (1, 45, 80, 324, 256, 1, 1, 1, 0, 1, 1, 0, E.ACT_RELU, 0.0, False, 328),
    "halo_flat_ragged_rows": (1, 1, 2999, 512, 1960, 1, 1, 1, 0, 1, 1, 0, E.ACT_GELU, 0.0, True, None),
    "halo_5x5_dil2": (4, 48, 64, 64, 128, 5, 5, 1, 4, 2, 1, 0, E.ACT_NONE, 0.0, False, None),
}


def check_conv(name):
    (N, H, W, cin, cout, kh, kw, s, pad, dil, groups, rep, act, slope, use_res, cin_pad) = CONV_CASES[name]
    eng = bare_engine()
    g = torch.Generator().manual_seed(hash(name) % 1000)
    w = torch.randn(cout, cin // groups, kh, kw, generator=g) / math.sqrt(cin // groups * kh * kw)
    b = torch.randn(cout, generator=g) * 0.1
    x = torch.randn(N, cin, H, W, generator=g)
    cin_k = cin if cin_pad is None else cin_pad
    cmap = None if cin_pad is None else list(range(cin)) + [-1] * (cin_pad - cin)
    eng.register_conv("t." + name, w, b, groups, cmap)
    xh = torch.zeros(N, H, W, cin_k, dtype=torch.float16)
    xh[..., :cin] = x.permute(0, 2, 3, 1).half()
    xh = xh.to(DEV)
    ph, pw = (pad if isinstance(pad, tuple) else (pad, pad))
    # torch reference on the fp16-rounded operands, fp32 math
    xr, wr = x.half().float().to(DEV), w.half().float().to(DEV)
    if rep:
        xr = F.pad(xr, (pw, pw, ph, ph), mode="replicate")
        ref = F.conv2d(xr, wr, b.to(DEV), s, 0, dil, groups)
    else:
        ref = F.conv2d(xr, wr, b.to(DEV), s, (ph, pw), dil, groups)
    res = None
    if act == E.ACT_RELU: ref = F.relu(ref)
    elif act == E.ACT_LRELU: ref = F.leaky_relu(ref, slope)
    elif act == E.ACT_SIGMOID: ref = torch.sigmoid(ref)
    elif act == E.ACT_TANH: ref = torch.tanh(ref)
    elif act == E.ACT_GELU: ref = F.gelu(ref)
    if use_res:
        res = torch.randn(ref.shape, generator=g).permute(0, 2, 3, 1).contiguous().half().to(DEV)
        ref = ref + res.float().permute(0, 3, 1, 2)
    if ph != pw:
        # op_conv takes a single pad; asymmetric kernels go through the lower-level builder in the stages.
        # Emulate with explicit zero padding of the input.
        xh = F.pad(xh, (0, 0, pw, pw, ph, ph))
        out = eng.op_conv("t." + name, xh.contiguous(), s, 0, dil, bool(rep), act, slope, res)
    else:
        out = eng.op_conv("t." + name, xh, s, ph, dil, bool(rep), act, slope, res)
    torch.cuda.synchronize()
    return stats(out.permute(0, 3, 1, 2), ref)


# ------------------------------------------------------------------------------------------------ HBM kernels
def check_corr_lookup():
    eng = bare_engine()
    g = torch.Generator().manual_seed(3)
    B, h8, w8 = 2, 22, 40
    P = h8 * w8
    f1, f2 = torch.randn(B, 64, h8, w8, generator=g), torch.randn(B, 64, h8, w8, generator=g)
    pyr = [p.half().float() for p in O.corr_pyramid(f1, f2)]  # level-wise fp16 rounding like the CUDA path stores
    coords = torch.stack(torch.meshgrid(torch.arange(w8), torch.arange(h8), indexing="xy"), 0).float()[None].repeat(B, 1, 1, 1)
    coords = coords + 6 * torch.randn(B, 2, h8, w8, generator=g)
    ref = O.corr_lookup(pyr, coords)  # [B,324,h,w]
    lv = [p.reshape(B * P, -1).half().to(DEV).contiguous() for p in pyr]
    cd = coords.permute(0, 2, 3, 1).reshape(B * P, 2).contiguous().to(DEV)
    out = eng.op_corr_lookup(lv, cd, h8, w8)
    torch.cuda.synchronize()
    st = stats(out[:, :324].reshape(B, h8, w8, 324).permute(0, 3, 1, 2), ref)
    st["pad_zero"] = float(out[:, 324:].abs().max())
    return st


def check_imgprop_step():
    eng = bare_engine()
    H, W = 48, 64
    frames, m, (ff, fb) = cases.imgprop_case()
    cur = (frames[0, 1] * (1 - m[0, 1])).half().float()
    prop = (frames[0, 2] * (1 - m[0, 2])).half().float()
    mc, mp = m[0, 1], m[0, 2]
    fp_, fc_ = ff[0, 1].half().float(), fb[0, 1].half().float()
    valid = O.fb_consistency(fp_[None], fc_[None])
    warped = O.warp_by_flow(prop[None], fp_[None].permute(0, 2, 3, 1), "nearest")
    mv = O._bin(O.warp_by_flow(mp[None], fp_[None].permute(0, 2, 3, 1)))
    u = O._bin(mc[None] * valid * (1 - mv))
    ref_f = u * warped + (1 - u) * cur[None]
    ref_m = O._bin(mc[None] * (1 - valid * (1 - mv)))
    pack = lambda f, k: torch.cat([f, k], 0).permute(1, 2, 0).contiguous().half().to(DEV)
    n2 = lambda f: f.permute(1, 2, 0).contiguous().half().to(DEV)
    out = eng.op_imgprop_step(pack(cur, mc), pack(prop, mp), n2(fp_), n2(fc_)).float().cpu()
    d = (out[..., :3].permute(2, 0, 1) - ref_f[0]).abs()
    return dict(frame_mismatch_frac=float((d.max(0).values > 1e-3).float().mean()), max_abs=float(d.max()),
                mask_mismatch_frac=float((out[..., 3] != ref_m[0, 0]).float().mean()))


def check_attention():
    eng = bare_engine()
    g = torch.Generator().manual_seed(5)
    t, gh, gw, C = 5, 8, 12, 512     # padded grid 10 x 18 -> 4 windows, pooled 2 x 4
    nh, nw = 10, 18
    x = torch.randn(1, t, gh, gw, C, generator=g).half().float()
    sd = {}
    p = "a."
    eye = torch.eye(C)
    for n in ("query", "key", "value", "proj"):
        sd[p + n + ".weight"], sd[p + n + ".bias"] = eye, torch.zeros(C)
    sd[p + "pool_layer.weight"] = torch.full((C, 1, 4, 4), 1 / 16.0) + 0.02 * torch.randn(C, 1, 4, 4, generator=g)
    sd[p + "pool_layer.bias"] = 0.1 * torch.randn(C, generator=g)
    sd[p + "valid_ind_rolled"] = torch.from_numpy(Wt.rolled_valid_indices())
    mask = torch.zeros(1, 3, gh, gw, 1)
    mask[0, :, 1:3, 2:5] = 1  # only window (0,0) is masked
    res = {}
    for parity in (0, 1):
        t_ind = torch.arange(parity, t, 2)
        ref = O.sparse_window_attention(sd, p, x, mask, t_ind)
        xp = F.pad(x, (0, 0, 0, nw - gw, 0, nh - gh))
        px = F.conv2d(xp.view(t, nh, nw, C).permute(0, 3, 1, 2), sd[p + "pool_layer.weight"], sd[p + "pool_layer.bias"],
                      stride=4, groups=C)
        n_pool = px.shape[-2] * px.shape[-1]
        pkv = px.permute(0, 2, 3, 1).reshape(t, n_pool, C)
        qkv = torch.cat([xp, xp, xp], -1).view(t, nh * nw, 3 * C).half().to(DEV).contiguous()
        pkv2 = torch.cat([pkv, pkv], -1).half().to(DEV).contiguous()
        flags = torch.tensor([1, 0, 0, 0], dtype=torch.int32, device=DEV)
        out = eng.op_attention(qkv, pkv2, flags, t, gh, gw, n_pool, parity)
        torch.cuda.synchronize()
        res[f"parity{parity}"] = stats(out[None], ref)
    return res


# ------------------------------------------------------------------------------------------------ stages
def check_raft(golden):
    m = full_models()
    fr = cases.raft_case()
    ff, fb = m.raft_model.engine.raft_bidir(fr[0].to(DEV), cases.RAFT_ITERS)
    torch.cuda.synchronize()
    return dict(fwd=stats_at(golden, "raft_ff", ff[None]), bwd=stats_at(golden, "raft_fb", fb[None]))


def check_rfc(golden):
    m = full_models()
    (ff, fb), masks = cases.rfc_case()
    of, ob = m.flow_model.engine.flow_complete(ff[0].to(DEV), fb[0].to(DEV), masks[0].to(DEV))
    torch.cuda.synchronize()
    return dict(fwd=stats_at(golden, "rfc_f", of[None]), bwd=stats_at(golden, "rfc_b", ob[None]))


def check_imgprop(golden):
    m = full_models()
    frames, mk, (ff, fb) = cases.imgprop_case()
    uf, um = m.inpaint_model.engine.image_propagate(frames[0].to(DEV), mk[0].to(DEV), ff[0].to(DEV), fb[0].to(DEV))
    torch.cuda.synchronize()
    d = np.abs(golden.pick("imgprop_frames", uf[None].float()) - golden["imgprop_frames"]).max(1)   # per pixel
    return dict(frame_mismatch_frac=float((d > 2e-3).mean()), frame_max_abs=float(d.max()),
                mask_mismatch_frac=float((um.cpu() != torch.from_numpy(golden["imgprop_masks"])[0]).float().mean()))


def check_window(golden):
    m = full_models()
    eng = m.inpaint_model.engine
    c = cases.window_case()
    t, l_t = c["frames"].shape[1], c["l_t"]
    # the session API wants flows for all T-1 pairs; only the local ones are used
    H, W = c["frames"].shape[-2:]
    ff = torch.zeros(t - 1, 2, H, W)
    fb = torch.zeros(t - 1, 2, H, W)
    ff[:l_t - 1], fb[:l_t - 1] = c["flows"][0][0], c["flows"][1][0]
    eng.gen_begin(c["frames"][0].to(DEV), c["masks_in"][0].to(DEV), c["masks_upd"][0].to(DEV), ff.to(DEV), fb.to(DEV))
    pred = eng.gen_window(list(range(t)), l_t)
    eng.gen_end()
    torch.cuda.synchronize()
    out = pred[..., :3].permute(0, 3, 1, 2).float()
    return stats_at(golden, "window_pred", out[None])


def check_e2e(golden):
    m = full_models()
    e = cases.e2e_case()
    icfg = IU.ImageConfig(e["W"], e["H"], 5, 8, (e["W"], e["H"]), e["T"])
    ft, fm, md, orig = IU.prepare_frames_and_masks(IU.convert_image_to_frames(e["image"]), e["mask"], icfg, torch.device(DEV))
    cfg = PI.ProPainterConfig(e["ref_stride"], e["neighbor_length"], e["subvideo_length"], e["raft_iter"], "enable",
                              e["T"], torch.device(DEV), icfg.process_size)
    uf, um, flows = PI.process_inpainting(m, ft, fm, md, cfg)
    comp = PI.feature_propagation(m.inpaint_model, uf, um, md, flows, orig, cfg)
    torch.cuda.synchronize()
    a, b = golden.pick("e2e_frames_u8", np.stack(comp)).astype(np.float64), golden["e2e_frames_u8"].astype(np.float64)
    mse = ((a - b) ** 2).mean()
    hole = golden.pick("e2e_frames_u8", golden["e2e_masks_dilated"][0, :, 0] > 0.5)
    mse_hole = (((a - b) ** 2).sum(-1)[hole]).mean() / 3
    return dict(psnr=float(10 * np.log10(255 ** 2 / max(mse, 1e-12))),
                psnr_hole=float(10 * np.log10(255 ** 2 / max(mse_hole, 1e-12))),
                max_abs_u8=float(np.abs(a - b).max()), frac_gt1=float((np.abs(a - b) > 1).mean()),
                flow=stats_at(golden, "e2e_pred_flow_f", flows[0].float()),
                upd_frames=stats_at(golden, "e2e_updated_frames", uf.float()))


# ------------------------------------------------------------------------------------------------ round 2
def _psnr_stats(a, b, hole=None):
    """a, b: [..., 3] uint8 pixels (full frames or the fixture's sampled pixels); hole: [...] bool."""
    a, b = np.asarray(a).astype(np.float64), np.asarray(b).astype(np.float64)
    mse = ((a - b) ** 2).mean()
    out = dict(psnr=float(10 * np.log10(255 ** 2 / max(mse, 1e-12))), max_abs_u8=float(np.abs(a - b).max()),
               frac_gt1=float((np.abs(a - b) > 1).mean()), frac_ne=float((a != b).mean()))
    if hole is not None and hole.any():
        mh = (((a - b) ** 2).sum(-1)[hole]).mean() / 3
        out["psnr_hole"] = float(10 * np.log10(255 ** 2 / max(mh, 1e-12)))
    return out


def _node_models():
    """The node classes find the synthetic-weight engine through model_utils.set_resident_models."""
    from comfyui_propainter_nodes_b200.utils import model_utils as MU
    m = full_models()
    MU.set_resident_models(DEV, m)
    return m


def _img_u8(img):
    return (img.detach().cpu().float().numpy() * 255.0 + 0.5).astype(np.uint8)


def check_c1_node(golden2):
    """BASELINE config[0] through ProPainterInpaint (320x180 -> 320x176 resize inside the node), fp16="disable"."""
    from comfyui_propainter_nodes_b200.propainter_nodes import ProPainterInpaint
    m = _node_models()
    c = cases.c1_case()
    img, fmask, dmask = ProPainterInpaint().propainter_inpainting(c["image"], c["mask"], **c["kwargs"])
    torch.cuda.synchronize()
    assert img.device.type == "cpu" and img.dtype == torch.float32
    hole = golden2.pick("c1_image_u8", golden2["c1_masks_dilated_u8"] > 0)
    st = _psnr_stats(golden2.pick("c1_image_u8", _img_u8(img)), golden2["c1_image_u8"], hole)
    st["flow_masks_equal"] = bool(np.array_equal(_img_u8(fmask), golden2["c1_flow_masks_u8"]))
    st["masks_dilated_equal"] = bool(np.array_equal(_img_u8(dmask), golden2["c1_masks_dilated_u8"]))
    # stage tensors of the same run
    kw = c["kwargs"]
    T, H, W = c["image"].shape[:3]
    icfg = IU.ImageConfig(kw["width"], kw["height"], kw["mask_dilates"], kw["flow_mask_dilates"], (W, H), T)
    ft, fm, md, orig = IU.prepare_frames_and_masks(IU.convert_image_to_frames(c["image"]), c["mask"], icfg, torch.device(DEV))
    cfg = PI.ProPainterConfig(kw["ref_stride"], kw["neighbor_length"], kw["subvideo_length"], kw["raft_iter"], kw["fp16"],
                              T, torch.device(DEV), icfg.process_size)
    gt = PI.compute_flow(m.raft_model, ft, cfg)
    uf, um, pf = PI.process_inpainting(m, ft, fm, md, cfg)
    st["raft_flow"] = stats_at(golden2, "c1_gt_flow_f_s2", gt[0][..., ::2, ::2])
    st["pred_flow"] = stats_at(golden2, "c1_pred_flow_f", pf[0])
    st["updated_masks_mismatch"] = float((_img_u8(um) != golden2["c1_updated_masks_u8"]).mean())
    return st


def check_raft20(golden2):
    """20 GRU iterations at 640x360 against the fp32 reference, error vs iteration, damped and un-damped flow head."""
    fr = cases.raft20_case()[0].to(DEV)
    out = {}
    for tag, gain in cases.RAFT20_GAINS.items():
        eng = E.Engine(DEV, workspace_gb=6.0).load_weights(Wt.synthetic_raft_state_dict(flow_head_gain=gain),
                                                           Wt.synthetic_rfc_state_dict(), Wt.synthetic_generator_state_dict())
        for it in cases.RAFT20_ITERS:
            ff, _ = eng.raft_bidir(fr, it)
            torch.cuda.synchronize()
            k = f"raft20_{tag}_it{it}_s4"
            got, ref = torch.from_numpy(golden2.pick(k, ff[:, :, ::4, ::4])), torch.from_numpy(golden2[k])
            s = stats(got, ref)
            d = (got.float() - ref).abs().flatten()
            s["p99_abs"] = float(torch.quantile(d, 0.99))
            out[f"{tag}_it{it}"] = s
            if it == max(cases.RAFT20_ITERS):
                out[f"{tag}_final"] = stats_at(golden2, f"raft20_{tag}_final_s2", ff[:, :, ::2, ::2])
        eng.close()
    return out


def check_chunked(golden2):
    """T=26 > subvideo_length=12: chunked complete_flow / image_propagation halos + ref_num schedule."""
    m = full_models()
    e = cases.chunked_case()
    icfg = IU.ImageConfig(e["W"], e["H"], 5, 8, (e["W"], e["H"]), e["T"])
    ft, fm, md, orig = IU.prepare_frames_and_masks(IU.convert_image_to_frames(e["image"]), e["mask"], icfg, torch.device(DEV))
    cfg = PI.ProPainterConfig(e["ref_stride"], e["neighbor_length"], e["subvideo_length"], e["raft_iter"], "disable",
                              e["T"], torch.device(DEV), icfg.process_size)
    gt = PI.compute_flow(m.raft_model, ft, cfg)
    uf, um, pf = PI.process_inpainting(m, ft, fm, md, cfg)
    comp = PI.feature_propagation(m.inpaint_model, uf, um, md, pf, orig, cfg)
    torch.cuda.synchronize()
    hole = golden2.pick("chunk_frames_u8", md[0, :, 0].cpu().numpy() > 0.5)
    st = _psnr_stats(golden2.pick("chunk_frames_u8", np.stack(comp)), golden2["chunk_frames_u8"], hole)
    st["raft_flow"] = stats_at(golden2, "chunk_gt_flow_f_s2", gt[0][..., ::2, ::2])
    st["pred_flow_f"] = stats_at(golden2, "chunk_pred_flow_f", pf[0])
    st["pred_flow_b"] = stats_at(golden2, "chunk_pred_flow_b", pf[1])
    st["updated_masks_mismatch"] = float((_img_u8(um) != golden2["chunk_updated_masks_u8"]).mean())
    return st


def check_outpaint_node(golden2):
    from comfyui_propainter_nodes_b200.propainter_nodes import ProPainterOutpaint
    _node_models()
    o = cases.outpaint_case()
    img, omask, ow, oh = ProPainterOutpaint().propainter_outpainting(o["image"], **o["kwargs"])
    torch.cuda.synchronize()
    hole = golden2.pick("outpaint_image_u8", golden2["outpaint_mask_u8"] > 0)
    st = _psnr_stats(golden2.pick("outpaint_image_u8", _img_u8(img)), golden2["outpaint_image_u8"], hole)
    st["mask_equal"] = bool(np.array_equal(_img_u8(omask), golden2["outpaint_mask_u8"]))
    st["size_equal"] = [int(ow), int(oh)] == [int(v) for v in golden2["outpaint_size"]]
    return st


def check_composite_exact():
    """pp_composite vs the numpy restatement of the reference loop on IDENTICAL predictions: byte for byte, in the
    float32 mode and in the half mode, over a schedule with up to three visits per frame."""
    eng = bare_engine()
    g = torch.Generator().manual_seed(77)
    T, H, W = 9, 40, 56
    sched = O.window_schedule(T, 4, 3, 80)
    orig = torch.randint(0, 256, (T, H, W, 3), generator=g, dtype=torch.uint8)
    md = (torch.rand(T, 1, H, W, generator=g) > 0.4).float()
    res = {}
    for half in (False, True):
        comp_ref = [None] * T
        comp = torch.zeros_like(orig).to(DEV)
        visited = [False] * T
        for nb, _ in sched:
            # tanh outputs incl. the exact ends and values whose *255 image sits next to an integer
            pred = (torch.rand(len(nb), H, W, 4, generator=g) * 2 - 1).half()
            pred[0, 0, :8, :3] = torch.tensor([-1.0, 1.0, 0.0, 0.5, -0.5, 0.9961, 0.00392, -0.00392]).half()[:, None]
            p = pred[..., :3]
            if half:   # the reference's fp16 mode: (pred + 1) / 2 in half on the device, numpy * 255 stays half
                p255 = ((p + 1) / 2).numpy() * 255
                assert p255.dtype == np.float16
            else:      # fp32 mode, same prediction values
                p255 = ((p.float() + 1) / 2).numpy() * 255
            bm = md[nb].permute(0, 2, 3, 1).numpy().astype(np.uint8)
            O.composite_window(comp_ref, p255, bm, [o.numpy() for o in orig], nb)
            ids = torch.tensor(nb, dtype=torch.int32, device=DEV)
            first = torch.tensor([0 if visited[i] else 1 for i in nb], dtype=torch.int32, device=DEV)
            for i in nb:
                visited[i] = True
            eng.composite(pred.to(DEV), md.to(DEV), orig.to(DEV), comp, ids, first, half)
        torch.cuda.synchronize()
        res["half" if half else "float"] = int((comp.cpu().numpy() != np.stack(comp_ref)).sum())
    return res


def check_dcn_samplers(timing=False):
    """TMA-staged tiled sampler == plain L2 sampler, bit for bit (same arithmetic in the same order), on the two shapes
    of the pipeline: C=256 / |offset| <= 5 (flow completion) and C=128 / 3*tanh + flow (generator), with offsets that also
    leave the staged box (large flows) and the image."""
    eng = bare_engine()
    g = torch.Generator().manual_seed(9)
    res = {}
    for tag, (N, H, W, C, mag, fscale) in {"rfc": (2, 45, 80, 256, 5.0, None), "gen": (3, 90, 160, 128, 3.0, 2.5),
                                           "gen_big_flow": (2, 40, 56, 128, 3.0, 12.0)}.items():
        x = torch.randn(N, H, W, C, generator=g).half().to(DEV)
        offs = (torch.randn(N, H, W, 432, generator=g) * 1.5).half().to(DEV)
        flow = None if fscale is None else (torch.randn(N, H, W, 2, generator=g) * fscale).half().to(DEV)
        a = eng.op_dcn_sample(x, offs, flow, mag, False)
        b = eng.op_dcn_sample(x, offs, flow, mag, True)
        torch.cuda.synchronize()
        res[tag] = dict(mismatch=int((a != b).sum()), nonzero=float((a != 0).float().mean()), nan=bool(torch.isnan(b.float()).any()))
        if timing:
            for name, tl in (("plain", False), ("tiled", True)):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                eng.op_dcn_sample(x, offs, flow, mag, tl)
                s.record()
                for _ in range(20):
                    eng.op_dcn_sample(x, offs, flow, mag, tl)
                e.record()
                torch.cuda.synchronize()
                res[tag][name + "_us"] = s.elapsed_time(e) / 20 * 1000
    return res


def check_step_variants():
    """The recurrent propagation steps have three execution variants -- multi-layer program kernel (default), one launch
    per layer with the TMA-staged deformable sampler, one launch per layer with the plain L2 sampler -- that perform the
    same arithmetic in the same order: outputs must be bit-identical (flow completion, generator window)."""
    import os
    m = full_models()
    eng = m.flow_model.engine
    (ff, fb), masks = cases.rfc_case()
    c = cases.window_case()
    t, l_t = c["frames"].shape[1], c["l_t"]
    H, W = c["frames"].shape[-2:]
    wf = torch.zeros(t - 1, 2, H, W)
    wb = torch.zeros(t - 1, 2, H, W)
    wf[:l_t - 1], wb[:l_t - 1] = c["flows"][0][0], c["flows"][1][0]
    outs = {}
    keep = {k: os.environ.get(k) for k in ("PP_PROG", "PP_DCN_TILED")}
    try:
        for tag, env in (("program", {"PP_PROG": "1", "PP_DCN_TILED": "1"}), ("tiled", {"PP_PROG": "0", "PP_DCN_TILED": "1"}),
                         ("plain", {"PP_PROG": "0", "PP_DCN_TILED": "0"})):
            os.environ.update(env)
            of, ob = eng.flow_complete(ff[0].to(DEV), fb[0].to(DEV), masks[0].to(DEV))
            eng.gen_begin(c["frames"][0].to(DEV), c["masks_in"][0].to(DEV), c["masks_upd"][0].to(DEV), wf.to(DEV), wb.to(DEV))
            pred = eng.gen_window(list(range(t)), l_t)
            eng.gen_end()
            torch.cuda.synchronize()
            outs[tag] = (of.clone(), ob.clone(), pred.clone())
    finally:
        for k, v in keep.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    res = {}
    for tag in ("program", "tiled"):
        # lane 3 of the prediction tensor is never written (3 output channels in a 4-wide pixel): compare rgb only
        res[tag + "_vs_plain"] = [int((a[..., :3] != b[..., :3]).sum()) if a.dim() == 4 and a.shape[-1] == 4 else int((a != b).sum())
                                  for a, b in zip(outs[tag], outs["plain"])]
    return res


def check_small_workspace_fallback():
    """A workspace far below what one batched pass needs: gen_run splits the schedule into sub-batches (down to one
    window) and the result is bit-identical; a failing call leaves the arena untouched (no leak)."""
    m = full_models()
    e = cases.e2e_case()
    icfg = IU.ImageConfig(e["W"], e["H"], 5, 8, (e["W"], e["H"]), e["T"])
    ft, fm, md, orig = IU.prepare_frames_and_masks(IU.convert_image_to_frames(e["image"]), e["mask"], icfg, torch.device(DEV))
    cfg = PI.ProPainterConfig(e["ref_stride"], e["neighbor_length"], e["subvideo_length"], e["raft_iter"], "enable",
                              e["T"], torch.device(DEV), icfg.process_size)
    uf, um, pf = PI.process_inpainting(m, ft, fm, md, cfg)
    ref = np.stack(PI.feature_propagation(m.inpaint_model, uf, um, md, pf, orig, cfg))
    small = E.Engine(DEV, workspace_gb=0.3).load_weights(Wt.synthetic_raft_state_dict(), Wt.synthetic_rfc_state_dict(),
                                                         Wt.synthetic_generator_state_dict())
    ms = Models(StageHandle(small, "raft"), StageHandle(small, "flow"), StageHandle(small, "inpaint"))
    sched = PI.window_schedule(cfg)
    out = np.stack(PI.feature_propagation(ms.inpaint_model, uf, um, md, pf, orig, cfg))
    n_batches = small.gen_run_calls            # engine passes the small arena forced for one clip
    # an impossible request fails loudly and leaves the arena as it was
    leaked = None
    try:
        small.raft_bidir(torch.zeros(3, 3, 1024, 2048, device=DEV), 1)
    except RuntimeError as ex:
        leaked = str(ex)
    out2 = np.stack(PI.feature_propagation(ms.inpaint_model, uf, um, md, pf, orig, cfg))
    small.close()
    return dict(mismatch=int((out != ref).sum()), mismatch_after_failure=int((out2 != ref).sum()), sub_batches=n_batches,
                failure=leaked)


def main():
    import json
    import os
    golden = Golden(os.path.join(os.path.dirname(__file__), "golden", "reference_outputs.npz"))
    golden2 = Golden(os.path.join(os.path.dirname(__file__), "golden", "reference_outputs_r2.npz"))
    only = sys.argv[1:]
    checks = [(f"conv:{n}", (lambda n=n: check_conv(n))) for n in CONV_CASES]
    checks += [("corr_lookup", check_corr_lookup), ("imgprop_step", check_imgprop_step), ("attention", check_attention),
               ("raft", lambda: check_raft(golden)), ("rfc", lambda: check_rfc(golden)),
               ("imgprop", lambda: check_imgprop(golden)), ("window", lambda: check_window(golden)),
               ("e2e", lambda: check_e2e(golden)), ("c1_node", lambda: check_c1_node(golden2)),
               ("raft20", lambda: check_raft20(golden2)), ("chunked", lambda: check_chunked(golden2)),
               ("outpaint_node", lambda: check_outpaint_node(golden2)), ("composite_exact", check_composite_exact),
               ("small_workspace", check_small_workspace_fallback), ("step_variants", check_step_variants),
               ("dcn_samplers", lambda: check_dcn_samplers(True))]
    for name, fn in checks:
        if only and not any(o in name for o in only):
            continue
        t0 = time.time()
        try:
            r = fn()
            print(f"[{name}] {time.time() - t0:.2f}s {json.dumps(r)}", flush=True)
        except Exception as ex:  # keep going: one report per GPU call
            print(f"[{name}] FAILED {type(ex).__name__}: {ex}", flush=True)
            traceback.print_exc()
            try:
                torch.cuda.synchronize()
            except Exception as ex2:
                print("CUDA context is broken, stopping:", ex2, flush=True)
                break


if __name__ == "__main__":
    main()
