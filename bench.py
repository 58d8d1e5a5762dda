#!/usr/bin/env python
"""Bench of the ProPainter hot path: inpainted frames/s at 640x360 on an 80-frame subvideo (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--mode strong|weak] [--dump-outputs DIR]

One "step" = one pass of the whole hot path (RAFT -> flow completion -> image propagation -> sliding-window
generator -> composite) over one synthetic 80-frame 640x360 clip.  `value` is measured with the prepared tensors
already resident in HBM; `e2e` goes through the ComfyUI node call with pageable host tensors (pre-processing, H2D and
the D2H of the result inside the timed region).  Weights are seeded synthetic checkpoints of the real architectures
(no network in this environment).

N > 1 (torchrun, one rank per GPU): the default is north_star's split -- ONE 80-frame subvideo shared by all N GPUs
(`scaling: "strong"`): RAFT pairs, the per-frame parts of flow completion and the sliding windows are sharded, the
exchange steps are NCCL all-gathers over NVLink; BASELINE config[2] (240 frames, subvideo_length 80, same sharding) is
reported alongside as `config2_240f`.  `--mode weak` runs one independent subvideo per GPU instead.

`--impl reference` times the UNMODIFIED reference (installed by __graft_entry__.build() into baseline/_ref, which is
git-ignored but travels to the GPU box) on the host cores: one pass over the first 16 frames of the same clip, all
threads; it also reports the reference's own PyTorch-CUDA fp16 path on the same B200 at the full 80 frames
(`reference_cuda`, the number SURVEY.md 8d calls "the number to beat").  Without baseline/_ref it falls back to the
CPU oracle port.

`--dump-outputs DIR` (b200 arm) writes what the last timed step returned -- the composited uint8 frames [T,H,W,3] --
as DIR/frames.npy, float32 values of a fixed seeded sample of DUMP_PIXELS pixels (all three channels, pixels in
ascending flat order), so that two builds can be compared output for output on identical inputs.
"""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

T_FRAMES, HEIGHT, WIDTH = 80, 360, 640
T_CONFIG2 = 240
DUMP_PIXELS, DUMP_SEED = 1 << 21, 0        # 2M pixels x 3 channels x float32 = 24 MiB
_OUT_FD = 1


def emit(line: str) -> None:
    """The ONE JSON line of the contract goes to the real stdout; everything else this process or its libraries
    print on fd 1 (NCCL's version banner, the node's progress lines) is routed to stderr in main()."""
    os.write(_OUT_FD, (line + "\n").encode())


PARAMS = dict(mask_dilates=5, flow_mask_dilates=8, ref_stride=10, neighbor_length=10, subvideo_length=80, raft_iter=20,
              fp16="enable")
METRIC = "inpainted frames/sec at 640x360, 80-frame subvideo"
WORKLOAD = "configs[1]: 80-frame 640x360 synthetic clip, ref_stride=10 neighbor_length=10 raft_iter=20 fp16"
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tensor_burst=d["bf16_tflops"], tensor=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor=1400.0, source="fallback")


def ncu_traffic():
    """DRAM bytes per launch of the dominant kernels from the committed ncu pass (tools/ncu_traffic.py ->
    profiles/traffic.json); None when no capture of the current kernels is committed."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    return json.load(open(p)) if os.path.exists(p) else {}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [int(s[0]) for s in self.samples if s and s[0].isdigit()]
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples if len(s) >= 6 for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        return dict(sm_mhz=int(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(sm))


def synthetic_inputs(T=T_FRAMES):
    from comfyui_propainter_nodes_b200.synthetic import synthetic_clip, synthetic_mask
    return synthetic_clip(T, HEIGHT, WIDTH, 1234), synthetic_mask(T, HEIGHT, WIDTH)


def dump_outputs(out_dir, frames):
    """DIR/frames.npy: float32 [DUMP_PIXELS, 3], the pixels of `frames` ([T,H,W,3]) at fixed seeded positions."""
    os.makedirs(out_dir, exist_ok=True)
    rows = frames.reshape(-1, frames.shape[-1])
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(rows.shape[0], min(DUMP_PIXELS, rows.shape[0]), replace=False))
    sample = rows[torch.from_numpy(idx).to(rows.device)].float().cpu().numpy()
    np.save(os.path.join(out_dir, "frames.npy"), sample)


def synthetic_state_dicts():
    from comfyui_propainter_nodes_b200 import weights as Wt
    return Wt.synthetic_raft_state_dict(), Wt.synthetic_rfc_state_dict(), Wt.synthetic_generator_state_dict()


# ------------------------------------------------------------------------------------------------------------------
# the reference itself (baseline/_ref) and, when it is absent, the CPU oracle port
# ------------------------------------------------------------------------------------------------------------------
def host_threads():
    """Threads of the CPU arm: every host core up to PP_CPU_THREADS (default 32 -- beyond that the 1/8-resolution
    convolutions of the recurrent stages stop scaling on the 128-core host, profiles/r01_cpu_threads.log)."""
    return min(os.cpu_count() or 1, int(os.environ.get("PP_CPU_THREADS", 32)))


def load_reference():
    """Import the unmodified reference package from baseline/_ref with a stub ``comfy.model_management`` (the one
    ComfyUI module it imports).  Returns the package's modules or None when it was not installed."""
    pkg = os.path.join(REF_DIR, "comfyui_propainter_nodes")
    if not os.path.exists(os.path.join(pkg, "propainter_inference.py")):
        return None
    sys.dont_write_bytecode = True
    if "comfy" not in sys.modules:
        comfy, mm = types.ModuleType("comfy"), types.ModuleType("comfy.model_management")
        mm.get_torch_device = lambda: torch.device("cuda" if torch.cuda.is_available() else "cpu")
        comfy.model_management = mm
        sys.modules["comfy"], sys.modules["comfy.model_management"] = comfy, mm
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import importlib
    ns = types.SimpleNamespace()
    ns.RI = importlib.import_module("comfyui_propainter_nodes.propainter_inference")
    ns.RU = importlib.import_module("comfyui_propainter_nodes.utils.image_utils")
    ns.MU = importlib.import_module("comfyui_propainter_nodes.utils.model_utils")
    ns.RAFT_bi = importlib.import_module("comfyui_propainter_nodes.model.modules.flow_comp_raft").RAFT_bi
    ns.RFC = importlib.import_module("comfyui_propainter_nodes.model.recurrent_flow_completion").RecurrentFlowCompleteNet
    ns.GEN = importlib.import_module("comfyui_propainter_nodes.model.propainter").InpaintGenerator
    return ns


def reference_models(ref, device, use_half):
    """What the reference's initialize_models builds (utils/model_utils.py:49-59), from the synthetic checkpoints
    instead of the downloaded files."""
    raft_sd, rfc_sd, gen_sd = synthetic_state_dicts()
    path = os.path.join(tempfile.mkdtemp(), "raft-things.pth")
    torch.save(raft_sd, path)
    with contextlib.redirect_stdout(sys.stderr):
        raft = ref.RAFT_bi(path, device)
        rfc = ref.RFC()
        rfc.load_state_dict(rfc_sd, strict=True)
        for p in rfc.parameters():
            p.requires_grad = False
        rfc.to(device).eval()
        gen = ref.GEN()
        gen.load_state_dict(gen_sd, strict=True)
        gen.to(device).eval()
    if use_half == "enable":
        rfc, gen = rfc.half(), gen.half()
    return ref.MU.Models(raft, rfc, gen)


def reference_pass(ref, models, image, mask, device, fp16):
    """The reference's own hot path on one clip: process_inpainting + feature_propagation (SURVEY.md 8d), timed by
    wall clock with the device synchronised.  Returns (frames/s, seconds)."""
    T = image.shape[0]
    icfg = ref.RU.ImageConfig(WIDTH, HEIGHT, PARAMS["mask_dilates"], PARAMS["flow_mask_dilates"], (WIDTH, HEIGHT), T)
    ft, fm, md, orig = ref.RU.prepare_frames_and_masks(ref.RU.convert_image_to_frames(image), mask, icfg, device)
    cfg = ref.RI.ProPainterConfig(PARAMS["ref_stride"], PARAMS["neighbor_length"], PARAMS["subvideo_length"],
                                  PARAMS["raft_iter"], fp16, T, device, icfg.process_size)
    if device.type == "cuda":
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(sys.stderr), contextlib.redirect_stderr(open(os.devnull, "w")):
        uf, um, pf = ref.RI.process_inpainting(models, ft, fm, md, cfg)
        ref.RI.feature_propagation(models.inpaint_model, uf, um, md, pf, orig, cfg)
    if device.type == "cuda":
        torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return T / dt, dt


def oracle_pass(n_frames):
    """CPU oracle port on the first `n_frames` frames of the clip (only used when baseline/_ref is absent)."""
    from comfyui_propainter_nodes_b200.utils import image_utils as IU
    from oracle import propainter_oracle as O
    image, mask = synthetic_inputs()
    image, mask = image[:n_frames], mask[:n_frames]
    icfg = IU.ImageConfig(WIDTH, HEIGHT, PARAMS["mask_dilates"], PARAMS["flow_mask_dilates"], (WIDTH, HEIGHT), n_frames)
    ft, fm, md, orig = IU.prepare_frames_and_masks(IU.convert_image_to_frames(image), mask, icfg, torch.device("cpu"))
    t0 = time.perf_counter()
    O.run_pipeline(*synthetic_state_dicts(), ft, fm, md, orig, raft_iter=PARAMS["raft_iter"],
                   subvideo_length=PARAMS["subvideo_length"], neighbor_length=PARAMS["neighbor_length"],
                   ref_stride=PARAMS["ref_stride"])
    dt = time.perf_counter() - t0
    return n_frames / dt, dt


def cpu_sample(n_frames):
    """(frames/s, seconds, kind) of the CPU baseline on the first n_frames frames: the real reference when installed,
    else the oracle port."""
    cores = host_threads()
    torch.set_num_threads(cores)
    ref = load_reference()
    if ref is None:
        v, dt = oracle_pass(n_frames)
        return v, dt, "port", cores
    image, mask = synthetic_inputs()
    models = reference_models(ref, torch.device("cpu"), "disable")
    v, dt = reference_pass(ref, models, image[:n_frames], mask[:n_frames], torch.device("cpu"), "disable")
    return v, dt, "reference", cores


def run_reference(args, rank):
    if rank != 0:
        return
    n = int(os.environ.get("PP_REF_FRAMES", 16))
    if args.warmup > 0:
        cpu_sample(3)            # thread pools, allocator and first-touch of the weights
    v, dt, kind, cores = cpu_sample(n)
    what = "the unmodified reference (baseline/_ref), fp32, PyTorch CPU" if kind == "reference" else "CPU oracle port of the reference, fp32"
    sample = (f"ONE pass over the first {n} frames of the 80-frame 640x360 clip (raft_iter=20, all other parameters of the "
              f"workload), {what}, {cores} threads, {dt:.1f} s")
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "frames/s", "n_gpus": args.gpus, "steps": 1,
        "warmup": min(args.warmup, 1), "ms_per_step": 1000.0 * dt, "higher_is_better": True, "scaling": "strong" if args.gpus > 1 else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOAD + " (CPU arm: first %d frames)" % n},
        "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "timed once (a 16-frame pass is tens of seconds); --steps/--warmup of the command line are not repeated",
    }
    # second stated baseline: the reference's own PyTorch-CUDA fp16 path on this B200 at the full workload
    if kind == "reference" and torch.cuda.is_available() and not args.no_ref_cuda:
        try:
            ref = load_reference()
            dev = torch.device("cuda", 0)
            models = reference_models(ref, dev, PARAMS["fp16"])
            image, mask = synthetic_inputs()
            reference_pass(ref, models, image[:20], mask[:20], dev, PARAMS["fp16"])   # warm-up (cuDNN autotune, allocator)
            vals = [reference_pass(ref, models, image, mask, dev, PARAMS["fp16"]) for _ in range(2)]
            best = max(vals)
            line["reference_cuda"] = {"value": best[0], "unit": "frames/s", "seconds": best[1], "frames": T_FRAMES,
                                      "what": "unmodified reference, PyTorch eager CUDA, fp16=enable, same 80-frame clip and weights, best of 2 after warm-up, "
                                              "process_inpainting + feature_propagation (inputs resident on the device)",
                                      "torch": torch.__version__, "gpu": torch.cuda.get_device_name(0)}
        except Exception as ex:  # the CPU number above stands on its own
            line["reference_cuda"] = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}
    emit(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------------------------
def run_b200(args, rank, world):
    import torch.distributed as dist
    from comfyui_propainter_nodes_b200 import propainter_inference as PI
    from comfyui_propainter_nodes_b200.propainter_nodes import ProPainterInpaint, _to_host
    from comfyui_propainter_nodes_b200.utils import image_utils as IU
    from comfyui_propainter_nodes_b200.utils import model_utils as MU
    from comfyui_propainter_nodes_b200 import parallel as PAR

    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    models = MU.build_models(dev, *synthetic_state_dicts())      # arena sized per clip (the node path)
    MU.set_resident_models(dev, models)                           # the node's initialize_models() returns this engine
    eng = models.raft_model.engine
    strong = world > 1 and args.mode == "strong"
    if world > 1:
        PAR.init_engine_comm(eng)        # NCCL communicator inside the C library (pp_comm_init), id broadcast via torch

    def prepared(T):
        image, mask = synthetic_inputs(T)
        icfg = IU.ImageConfig(WIDTH, HEIGHT, PARAMS["mask_dilates"], PARAMS["flow_mask_dilates"], (WIDTH, HEIGHT), T)
        ft, fm, md, orig = IU.prepare_frames_and_masks(IU.convert_image_to_frames(image), mask, icfg, dev)
        cfg = PI.ProPainterConfig(PARAMS["ref_stride"], PARAMS["neighbor_length"], PARAMS["subvideo_length"],
                                  PARAMS["raft_iter"], PARAMS["fp16"], T, dev, icfg.process_size)
        return image, mask, ft, fm, md, torch.from_numpy(np.stack(orig)).to(dev), cfg

    image, mask, ft, fm, md, orig_dev, cfg = prepared(T_FRAMES)
    eng.reserve_for_clip(T_FRAMES, HEIGHT, WIDTH)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > L2 (126 MB)

    def run_clip(ft, fm, md, orig_dev, cfg):
        if strong:
            return PAR.inpaint_clip_distributed(models, ft, fm, md, orig_dev, cfg)
        uf, um, flows = PI.process_inpainting(models, ft, fm, md, cfg)
        return PI.feature_propagation_device(models.inpaint_model, uf, um, md, flows, orig_dev, cfg)

    last = [None]       # the output of the latest step, kept only for --dump-outputs

    def step():
        out = run_clip(ft, fm, md, orig_dev, cfg)
        if args.dump_outputs:
            last[0] = out
        return out

    def staged():
        """Same work as step() on one GPU, with CUDA events between the stages (reported as stage_ms)."""
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        ev[0].record()
        gt = PI.compute_flow(models.raft_model, ft, cfg)
        ev[1].record()
        pf = PI.complete_flow(models.flow_model, gt, fm, cfg.subvideo_length)
        ev[2].record()
        uf, um = PI.image_propagation(models.inpaint_model, ft, md, pf, cfg)
        ev[3].record()
        PI.feature_propagation_device(models.inpaint_model, uf, um, md, pf, orig_dev, cfg)
        ev[4].record()
        torch.cuda.synchronize()
        names = ["raft", "flow_completion", "image_propagation", "generator_windows"]
        return {n: round(ev[i].elapsed_time(ev[i + 1]), 2) for i, n in enumerate(names)}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """K steps, each bracketed by CUDA events on the launch stream, L2 flushed in between; max over ranks."""
        barrier()
        times = []
        for _ in range(steps):
            flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            times.append(a.elapsed_time(b))
        barrier()
        total = torch.tensor([sum(times)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(total, op=dist.ReduceOp.MAX)
        return float(total.item()) / steps

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = eng.launch_count
    ms_per_step = timed(step, args.steps)
    launches = (eng.launch_count - l0) // max(args.steps, 1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last[0])
    last[0] = None
    clips = 1 if (strong or world == 1) else world
    value = clips * T_FRAMES / (ms_per_step / 1000.0)

    # ---- end to end through the node API with (pageable) host tensors: pre-processing + H2D + D2H inside
    node = ProPainterInpaint()

    def e2e_step():
        if strong:   # host tensors -> device pre-processing on every rank -> sharded clip -> float IMAGE back on the
            # host of rank 0 (the caller's process); the other ranks hold the same result in HBM and return it there
            f, m1, m2, o = eng.preprocess(image, mask, PARAMS["flow_mask_dilates"], PARAMS["mask_dilates"])
            out = eng.postprocess(PAR.inpaint_clip_distributed(models, f, m1, m2, o, cfg))
            return _to_host(out) if rank == 0 else out
        with contextlib.redirect_stdout(sys.stderr):   # the node prints progress; stdout carries only the JSON line
            frames, _, _ = node.propainter_inpainting(image, mask, WIDTH, HEIGHT, **PARAMS)
        return frames
    e2e_value = None
    if not args.no_e2e:
        # two warm-up calls whose results are held the way a caller (ComfyUI's output cache) holds them
        res = e2e_step()
        res = e2e_step()
        barrier()
        t0 = time.perf_counter()
        n_e2e = max(1, min(args.steps, 3))
        for _ in range(n_e2e):
            res = e2e_step()
        torch.cuda.synchronize()
        e2e_s = torch.tensor([(time.perf_counter() - t0) / n_e2e], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
        e2e_value = clips * T_FRAMES / float(e2e_s.item())
        del res
    sampler.stop_flag = True
    sampler.join(timeout=2)
    h2d = image.numel() * 4 + mask.numel() * 4              # the node uploads the IMAGE / MASK float tensors
    d2h = T_FRAMES * HEIGHT * WIDTH * 3 * 4                  # and downloads the float32 IMAGE result

    # ---- BASELINE config[2]: 240 frames, subvideo_length 80 (3 sub-video chunks), same sharding
    c2 = None
    if not args.no_config2:
        _, _, ft2, fm2, md2, orig2, cfg2 = prepared(T_CONFIG2)
        eng.reserve_for_clip(T_CONFIG2, HEIGHT, WIDTH)
        fn2 = lambda: run_clip(ft2, fm2, md2, orig2, cfg2)
        fn2()
        ms2 = timed(fn2, 2)
        c2 = {"workload": "configs[2]: 240-frame 640x360 clip, subvideo_length=80", "frames": T_CONFIG2, "steps": 2,
              "ms_per_step": ms2, "value": clips * T_CONFIG2 / (ms2 / 1000.0), "unit": "frames/s"}
        del ft2, fm2, md2, orig2

    # ---- per-kernel timing of one extra step (CUDA events on the launch stream) for the roofline
    roof, extra, stage_ms = None, [], None
    if strong and not args.no_profile and rank != 0:
        step()                      # the profiled step below is collective in strong mode
    if rank == 0 and not args.no_profile:
        if world == 1:
            stage_ms = staged()
        pk = peaks()
        traffic = ncu_traffic()
        eng.profile_enable(True)
        step()
        prof = eng.profile_dump()
        eng.profile_enable(False)
        all_ms = sum(v["ms"] for v in prof.values())

        def conv_class(prefix, label):
            sel = {k: v for k, v in prof.items() if k.startswith(prefix)}
            ms = sum(v["ms"] for v in sel.values())
            fl = sum(v["flops"] for v in sel.values())
            n = sum(v["count"] for v in sel.values())
            a = fl / (ms / 1e3) / 1e12 if ms > 0 else 0.0
            return {"bound": "tensor", "kernel": label, "achieved": a, "peak": pk["tensor"], "unit": "TFLOP/s", "frac": a / pk["tensor"],
                    "peak_source": pk["source"] + " bf16 sustained", "share_of_profiled_step": ms / all_ms if all_ms else None,
                    "launches": n, "flops_per_launch": fl / max(n, 1), "ms_per_launch": ms / max(n, 1), "ms": ms}

        FL = ("flops are ALGORITHMIC: 2 x output pixels x Cout x kh x kw x Cin/groups of the reference layer "
              "(no padded channels, no block-diagonal zeros)")
        # the dominant kernel of the step: the TMA halo-tile tcgen05 convolution (every stride-1 conv and every linear)
        roof = conv_class("conv:halo:", "conv_halo_kernel (TMA halo-tile tcgen05 convolution: every stride-1 conv / linear launch of the step); " + FL)
        roof["traffic"] = traffic.get("conv_bytes_per_launch")
        roof["traffic_note"] = traffic.get("note")
        extra.append(conv_class("conv:", "ALL tcgen05 convolution launches (conv_halo_kernel + conv_igemm_kernel + conv_prog_kernel); " + FL))
        extra.append(conv_class("conv:igemm:", "conv_igemm_kernel (cp.async implicit GEMM: stride-2 / 7x7 / replicate-pad layers, all-pairs correlation)"))
        extra.append(conv_class("conv:prog:", "conv_prog_kernel (multi-layer program: one flow-completion propagation step = 8 dependent layers per launch, "
                                              "latency-bound by construction)"))
        for name in ("corr_lookup", "imgprop", "dcn_sample", "featprop_warp", "fold_ffn"):
            if name in prof and prof[name]["ms"] > 0:
                v = prof[name]
                gbs = v["bytes"] / (v["ms"] / 1e3) / 1e9
                extra.append({"kernel": name, "bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s",
                              "frac": gbs / pk["hbm"], "launches": v["count"], "ms": v["ms"],
                              "traffic": traffic.get(name + "_bytes_per_launch")})
        if "attention" in prof:
            v = prof["attention"]
            tf = v["flops"] / (v["ms"] / 1e3) / 1e12 if v["ms"] > 0 else 0.0
            extra.append({"kernel": "window_attention_tc (tcgen05, masked windows) + window_attention (unmasked windows)", "bound": "tensor",
                          "achieved": tf, "peak": pk["tensor"], "unit": "TFLOP/s", "frac": tf / pk["tensor"],
                          "flops": "4 x queries x keys x 128 per head of the windows that are actually masked / unmasked in this clip",
                          "ms": v["ms"], "launches": v["count"]})
        if args.profile_out:
            with open(args.profile_out, "w") as fh:
                json.dump({"stage_ms": stage_ms, "kernels": prof}, fh, indent=1, sort_keys=True)
        top = sorted(prof.items(), key=lambda kv: -kv[1]["ms"])[:12]
        extra.append({"top_by_time_ms": {k: round(v["ms"], 3) for k, v in top}, "profiled_step_kernel_ms": all_ms})

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        v, dt, kind, cores = cpu_sample(4)
        cpu = {"value": v, "unit": "frames/s", "cores": cores, "kind": kind,
               "sample": f"first 4 frames of the same clip and parameters ({'unmodified reference from baseline/_ref' if kind == 'reference' else 'CPU oracle port'}, fp32, {dt:.1f} s)"}
    if rank == 0:
        if strong:
            par = (f"ONE subvideo sharded over {world} GPUs: RAFT pairs, flow-completion encoder/decoder frames and direction passes, "
                   f"generator windows; NCCL all-gathers of flows / features / predictions (pp_comm_*)")
        elif world > 1:
            par = f"{world} independent subvideos, no data-path collective"
        else:
            par = "single GPU"
        emit(json.dumps({
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak" if (world > 1 and not strong) else "strong",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": WORKLOAD + (", ONE clip shared by all GPUs" if strong else ", 1 clip per B200"),
                       "frames_per_gpu": T_FRAMES / world if strong else T_FRAMES, "l2": "flushed between steps (256 MiB write)",
                       "weights": "seeded synthetic checkpoints", "parallelism": par,
                       "e2e_inputs": "pageable host tensors (what ComfyUI hands a node); result in a pinned block of torch's caching host allocator",
                       "roofline_timing": "one extra profiled step after the timed region"},
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches), "clocks": sampler.summary(), "roofline": roof, "roofline_other": extra,
            "stage_ms": stage_ms, "config2_240f": c2, "cpu_baseline": cpu, "workspace_peak_gb": eng.workspace_peak / 2 ** 30,
        }))
    if world > 1:
        PAR.destroy_engine_comm(eng)
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="strong", choices=["strong", "weak"],
                    help="N>1: strong = ONE 80-frame subvideo shared by all GPUs (default, north_star); weak = one subvideo per GPU")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline sample")
    ap.add_argument("--no-e2e", action="store_true", help="skip the node-level end-to-end leg (profiling runs)")
    ap.add_argument("--no-profile", action="store_true", help="skip the per-kernel timed extra step")
    ap.add_argument("--no-config2", action="store_true", help="skip the 240-frame config[2] leg")
    ap.add_argument("--no-ref-cuda", action="store_true", help="reference arm: skip the reference's PyTorch-CUDA leg")
    ap.add_argument("--profile-out", default=None, help="write the full per-kernel table (JSON) here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="b200 arm: write a fixed seeded sample of the last timed step's frames to DIR/frames.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    global _OUT_FD
    sys.stdout.flush()
    _OUT_FD = os.dup(1)      # keep the real stdout for the JSON line ...
    os.dup2(2, 1)            # ... and send every other write to fd 1 (C libraries included) to stderr
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_b200(args, rank, world)


if __name__ == "__main__":
    main()
