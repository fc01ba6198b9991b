#!/usr/bin/env python
"""bench.py -- frames/sec of the AOT mask-propagation hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--model r50_aotl] [--dump-outputs DIR]

One "step" = one propagated frame through the reference's timed span (networks/managers/
evaluator.py:325-446): match_propogate_one_frame + decode + softmax/argmax + nearest resize +
update_memory; the reference frame is excluded, as in the reference.  Workload = BASELINE
configs[1]: R50-AOTL, synthetic 480p (481x849 network input, 480x854 output), 10 objects, long-term
gap 5, fp32; K = 99 steps is exactly the 100-frame clip.  Warm-up runs W frames of a scratch clip,
then the engine is restarted so the timed clip starts from an empty memory bank.

--dump-outputs DIR writes what the timed value pass handed back at its last step K (rank 0), as float32 .npy:
label.npy (the 480x854 label map) and logits.npy (the decoder's low-resolution logits of the background and the 10
objects).  Weights and clip are seeded, so the same arguments give the same inputs on every run and build.

Prints ONE JSON line (rank 0).  `value`: inputs resident in HBM, fused mask path.  `e2e`: the
drop-in API exactly as the unedited evaluator drives it, with pinned HOST frames copied H2D and
the label map copied D2H inside the timed region every step.  `roofline`: the long-term attention
kernel (tensor bound).  `cpu_baseline`: the CPU oracle port of the same span on the host cores.
With N > 1 each rank propagates its own clip (video-level data parallelism, no collective on the
data path; weak scaling).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

H_IN, W_IN, H_OUT, W_OUT, OBJS = 481, 849, 480, 854, 10   # SURVEY 8: what MultiRestrictSize makes of 480x854


def set_workload(model_name):
    """Network input size per model family (SURVEY 8): align_corners models get (k*16+1) sizes -- 481x849 for 480p --
    and the Swin models (align_corners=False, BASELINE configs[3]) multiples of 16 at 1.3 x 480p = 592x1040."""
    global H_IN, W_IN
    if model_name.startswith("swinb"):
        H_IN, W_IN = 592, 1040


def _peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.idx = gpu_index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "500", "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm = sorted(float(r[1]) for r in rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) >= 9:
                for n, v in zip(names, r[5:9]):
                    if v.strip().lower() == "active":
                        reasons.add(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def build_model(model_name, device):
    from aot_benchmark_b200 import EngineConfig, build_engine, build_vos_model
    cfg = EngineConfig("bench", model_name)
    torch.manual_seed(0)
    model = build_vos_model(cfg.MODEL_VOS, cfg).to(device).eval()   # random init: no checkpoints offline
    eng = build_engine(cfg.MODEL_ENGINE, phase="eval", aot_model=model, gpu_id=device.index,
                       long_term_mem_gap=cfg.TEST_LONG_TERM_MEM_GAP,
                       short_term_mem_skip=cfg.TEST_SHORT_TERM_MEM_SKIP)
    eng.eval()
    return cfg, model, eng


def make_clip(n_frames, seed):
    from oracle.aot_oracle import synthetic_video   # input generator only (shared with tests)
    frames, mask = synthetic_video(n_frames, H_IN, W_IN, OBJS, seed=seed)
    return frames, mask


# ---------------------------------------------------------------------------------------------
def step_fused(eng, img):
    """value path: all-kernel span, label map produced by the fused upsample+argmax kernel."""
    from aot_benchmark_b200 import ops
    eng.match_propogate_one_frame(img)
    logits = eng.decode_current_logits(None)
    e0 = eng.aot_engines[0]
    label = torch.empty((1, 1, H_OUT, W_OUT), dtype=torch.float32, device=img.device)
    ops.logits_argmax(e0.pred_id_logits, label, e0.align_corners)
    small = torch.empty((1, 1) + tuple(eng.input_size_2d), dtype=torch.float32, device=img.device)
    ops.nearest_resize(label, small)
    eng.update_memory(small)
    return label, logits


def step_dropin(eng, img_host, label_host, stream_dev):
    """e2e path: exactly the evaluator's calls (evaluator.py:302-305,332-339,355-361,418-422)."""
    img = img_host.to(stream_dev, non_blocking=True)
    eng.match_propogate_one_frame(img)
    logit = eng.decode_current_logits((H_OUT, W_OUT))
    prob = torch.softmax(logit, dim=1)
    label = torch.argmax(prob, dim=1, keepdim=True).float()
    fb = F.interpolate(label, size=eng.input_size_2d, mode="nearest")
    eng.update_memory(fb)
    label_host.copy_(label.to(torch.uint8), non_blocking=True)   # the mask the evaluator writes out


def dump_outputs(out_dir, arrays):
    """arrays: {name: CPU float tensor} -> out_dir/<name>.npy"""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU path). Use --impl reference for the CPU baseline.")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    from aot_benchmark_b200 import _lib
    L = _lib.lib()
    K, Wm = args.steps, max(args.warmup, 3)
    cfg, model, eng = build_model(args.model, dev)
    shard = args.mode == "shard"
    if shard:
        # BASELINE configs[3] mechanism: every rank propagates the SAME clip; the long-term memory bank is sharded by
        # memory frame over the ranks and the attention partials are exchanged (NCCL all-gather + exact merge) per layer
        if world < 2:
            raise SystemExit("--mode shard needs torchrun with >= 2 ranks (the bank is sharded over ranks)")
        eng.enable_kv_sharding(rank, world)
    frames, mask = make_clip(K + 1, seed=1234 + (0 if shard else rank))
    frames_dev = [f.to(dev) for f in frames]          # ~4.9 MB each, 490 MB for the clip: larger than L2
    frames_host = [f.pin_memory() for f in frames]
    mask_dev = mask.to(dev)
    label_host = torch.empty((1, 1, H_OUT, W_OUT), dtype=torch.uint8).pin_memory()
    from aot_benchmark_b200 import engine as engine_mod
    from aot_benchmark_b200 import ops as ops_mod

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def run_clip(mode, n_steps, keep=None):
        """keep: a dict that receives, after the timed region, host copies of what the last fused step returned."""
        eng.restart_engine()
        with torch.no_grad():
            eng.add_reference_frame(frames_dev[0], mask_dev, obj_nums=[OBJS], frame_step=0)
            barrier()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = L.aotb_launch_count() + engine_mod.REPLAYED_KERNELS[0]
            ev0.record()
            for t in range(1, n_steps + 1):
                if mode == "fused":
                    res = step_fused(eng, frames_dev[t])
                else:
                    step_dropin(eng, frames_host[t], label_host, dev)
            ev1.record()
            barrier()
            l1 = L.aotb_launch_count() + engine_mod.REPLAYED_KERNELS[0]
            if keep is not None:
                label, logits = res
                keep["label"] = label[0, 0].float().cpu()
                keep["logits"] = logits[0, :OBJS + 1].float().cpu()
        ms = ev0.elapsed_time(ev1)
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms, l1 - l0

    with torch.no_grad():
        # warm-up passes (buffers, module load, CUDA-graph capture of every call variant incl. the every-5th-frame
        # bank append): >= W frames, at least 11 so both memory-update variants have been captured
        run_clip("fused", min(max(Wm, 11), K))
        run_clip("dropin", min(max(Wm, 11), K))
    peaks, how = _peaks()
    peak = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
    clips = 1 if shard else world            # shard mode: one clip, total work fixed -> strong scaling

    def measure(n_steps, sample_clocks, keep=None):
        """value pass (fused mask path, resident inputs, CUDA graphs), e2e pass (drop-in API, pinned host frames), probe pass
        (same clip, eager launches, CUDA events around every long-term attention and every tensor-core conv launch)."""
        sampler = ClockSampler(local)
        if sample_clocks and rank == 0:
            sampler.start()
        ms_value, launches = run_clip("fused", n_steps, keep)
        clocks = sampler.stop() if (sample_clocks and rank == 0) else None
        ms_e2e, _ = run_clip("dropin", n_steps)
        lt_probe, conv_probe = [], []
        engine_mod.LT_PROBE = lt_probe
        run_clip("fused", n_steps)
        engine_mod.LT_PROBE = None
        ops_mod.CONV_PROBE = conv_probe        # separate pass: events around ~75 short launches per frame perturb the LT timing
        engine_mod.LT_PROBE = []
        run_clip("fused", n_steps)
        engine_mod.LT_PROBE = None
        ops_mod.CONV_PROBE = None
        torch.cuda.synchronize()
        lt_flops = sum(f for (_, _, f) in lt_probe)
        lt_ms = sum(a.elapsed_time(b) for (a, b, _) in lt_probe)
        cv_flops = sum(f for (_, _, f) in conv_probe)
        cv_ms = sum(a.elapsed_time(b) for (a, b, _) in conv_probe)
        return {"ms_value": ms_value, "ms_e2e": ms_e2e, "launches": int(launches), "clocks": clocks,
                "lt": (lt_flops, lt_ms, len(lt_probe)), "conv": (cv_flops, cv_ms, len(conv_probe))}

    def lt_roofline(m, n_steps):
        flops, ms, n = m["lt"]
        achieved = flops / (ms / 1e3) / 1e12 if ms > 0 else 0.0
        return {"achieved": round(achieved, 2), "peak": peak, "unit": "TFLOP/s", "frac": round(achieved / peak, 4),
                "launches": n, "avg_launch_us": round(1e3 * ms / max(n, 1), 2)}

    def conv_roofline(m, n_steps):
        flops, ms, n = m["conv"]
        achieved = flops / (ms / 1e3) / 1e12 if ms > 0 else 0.0
        return {"kernel": "conv_tc_kernel family (tcgen05 implicit GEMM, fp16x2 split: every Conv2d / Linear of the frame)",
                "bound": "tensor", "achieved": round(achieved, 2), "peak": peak, "unit": "TFLOP/s",
                "frac": round(achieved / peak, 4), "launches_per_frame": round(n / max(n_steps, 1), 1),
                "gflop_per_frame": round(flops / max(n_steps, 1) / 1e9, 2), "ms_per_frame": round(ms / max(n_steps, 1), 4),
                "algorithmic": "FLOPs = 2*M*Cout*(KH*KW*Cin) per launch, summed over the launches of the clip",
                "timing": "CUDA events around every launch in an eager (graph-free, PDL-free) probe pass of the same clip"}

    def encoder_probe(reps=40):
        """The image encoder alone (ResNet-50 layers + projector: 53 tcgen05 convs, the 7x7 stem and the max-pool), replayed from
        its captured graph with PDL as in the real step: FLOPs from one eager pass with the conv probe, time from CUDA events
        around `reps` graph replays on distinct frames.  This is the accurate number for the conv family (the per-launch events
        of the probe pass break graph replay and PDL, so they overstate the conv time)."""
        e0 = eng.aot_engines[0]
        st = torch.cuda.current_stream().cuda_stream
        probe = []
        ops_mod.CONV_PROBE, engine_mod.LT_PROBE = probe, []          # LT_PROBE != None: eager launches
        chain, ops_mod.CONV_CHAIN = ops_mod.CONV_CHAIN, False          # FLOPs are counted on the per-layer path
        with torch.no_grad():
            e0._encode(frames_dev[1], st)
            ops_mod.CONV_PROBE, engine_mod.LT_PROBE, ops_mod.CONV_CHAIN = None, None, chain
            for i in range(3):
                e0._encode(frames_dev[1 + i % K], st)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(reps):
                e0._encode(frames_dev[1 + i % K], st)
            b.record()
            torch.cuda.synchronize()
        flops = sum(f for (_, _, f) in probe)
        ms = a.elapsed_time(b) / reps
        ach = flops / (ms / 1e3) / 1e12
        return {"what": "image encoder alone (ResNet-50 stages + projector), captured graph replayed with PDL"
                        + (", stages + projector as ONE persistent dataflow kernel (conv_chain.cu)" if chain else ""),
                "conv_launches": len(probe), "gflop": round(flops / 1e9, 2), "ms": round(ms, 4),
                "achieved": round(ach, 2), "unit": "TFLOP/s", "frac": round(ach / peak, 4)}

    last = {} if args.dump_outputs and rank == 0 else None
    m = measure(K, True, last)
    enc = encoder_probe() if cfg.MODEL_ENCODER == "resnet50" else None
    enc_hw = eng.aot_engines[0].enc_hw
    h2d_bytes = int(frames_host[1].numel() * 4)
    cfg4 = None
    if args.cfg4_frames > 0 and args.model == "r50_aotl" and not shard:
        del frames_dev, frames_host, frames                 # ~1 GB of cfg2 frames
        eng.restart_engine()
        torch.cuda.empty_cache()
        cfg4 = measure_cfg4(args.cfg4_frames, rank, world, dev, dist)
    if last is not None:
        dump_outputs(args.dump_outputs, last)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    fps = clips * K / (m["ms_value"] / 1e3)
    fps_e2e = clips * K / (m["ms_e2e"] / 1e3)
    traffic, traffic_note = None, None
    ncu_json = os.path.join(REPO, "profiles", "lt_attn_ncu_latest.json")
    if os.path.exists(ncu_json) and cfg.MODEL_VOS == "aot":
        nj = json.load(open(ncu_json))
        traffic = nj.get("traffic_bytes")
        traffic_note = f"{nj.get('launch')}: dram read+write of one ncu --set full capture ({nj.get('source')})"
    lt_name = engine_mod.LT_KERNEL_NAME if cfg.MODEL_VOS == "aot" else engine_mod.deaot_lt_kernel_name()
    rl = {"kernel": lt_name, "bound": "tensor"}
    rl.update(lt_roofline(m, K))
    rl.update({"traffic": traffic, "traffic_note": traffic_note,
               "peak_source": f"MEASURED_PEAKS.json bf16 sustained ({how})",
               "algorithmic": f"FLOPs = 4*N*Tk*C per launch (N={enc_hw}, C=256, Tk={enc_hw}*m); the exact fp16x2 mode executes 3.5x "
                              f"these on the tensor pipe (6+16 MMAs per 128x128 tile), the fast mode 1.75x (DESIGN.md 3.1)"
               if cfg.MODEL_VOS == "aot" else f"FLOPs = 2*N*Tk*(128+1024) per launch (N={enc_hw}, Tk={enc_hw}*m)",
               "timing": "CUDA events around every launch in an eager (graph-free) probe pass of the same clip"})
    out = {
        "metric": "frames/sec (480p, 10 obj)", "value": round(fps, 3), "unit": "frames/s", "n_gpus": world,
        "steps": K, "warmup": Wm, "ms_per_step": round(m["ms_value"] / K, 4), "higher_is_better": True,
        "scaling": "strong" if shard else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.model} inference, synthetic {'1.3x480p' if H_IN > 481 else '480p'} clip (net input {H_IN}x{W_IN}, output "
                               f"{H_OUT}x{W_OUT}), {OBJS} objects, 1 reference + {K} propagated frames, long-term gap "
                               f"{cfg.TEST_LONG_TERM_MEM_GAP}, batch 1/GPU, "
                               + ("one clip, long-term bank sharded over the GPUs" if shard else "one clip per GPU"),
                   "weights": "seeded random init (no checkpoints offline)",
                   "l2": "inputs larger than L2 (distinct 4.9 MB frame per step, >126 MB activations per frame)",
                   "parallelism": f"bank-shard{world}" if shard else f"video-dp{world}"},
        "e2e": {"value": round(fps_e2e, 3), "unit": "frames/s",
                "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": int(label_host.numel()),
                "path": "AOTInferEngine drop-in API as networks/managers/evaluator.py drives it, pinned host frames"},
        "gpu_launches": m["launches"],
        "roofline": rl,
        "roofline_conv": dict(conv_roofline(m, K), encoder=enc),
        "clocks": m["clocks"],
    }
    if cfg4 is not None:
        out["cfg4"] = cfg4
    if not args.skip_cpu_baseline:
        out["gpu_eager_baseline"] = gpu_eager_baseline(args.model, dev)
    out["cpu_baseline"] = None if args.skip_cpu_baseline else cpu_baseline(args.model, threads=os.cpu_count())
    print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


def measure_cfg4(n_prop, rank, world, dev, dist, distinct=48):
    """BASELINE configs[3]: SwinB-AOTL, ONE 1.3x480p clip (net input 592x1040) of 1 reference + n_prop propagated frames, long-term
    gap 5 (the bank reaches 1 + n_prop/5 memory frames).  One GPU: the bank lives on that GPU.  N > 1 GPUs: every rank propagates
    the same clip, memory frame f lives on rank f % N, each rank attends over its shard and the un-normalised (O | m | l)
    partials are exchanged once per layer per frame (one packed all-gather) and merged exactly -- strong scaling of the
    long-term attention, everything else replicated.  Inputs resident in HBM (48 distinct 7.4 MB frames, cycled: > L2)."""
    from aot_benchmark_b200 import EngineConfig, build_engine, build_vos_model, ops
    from oracle.aot_oracle import synthetic_video
    Hc, Wc = 592, 1040
    cfg = EngineConfig("bench4", "swinb_aotl")
    torch.manual_seed(0)
    model = build_vos_model(cfg.MODEL_VOS, cfg).to(dev).eval()
    eng = build_engine(cfg.MODEL_ENGINE, phase="eval", aot_model=model, gpu_id=dev.index,
                       long_term_mem_gap=cfg.TEST_LONG_TERM_MEM_GAP, short_term_mem_skip=cfg.TEST_SHORT_TERM_MEM_SKIP).eval()
    if world > 1:
        eng.enable_kv_sharding(rank, world)
    frames, mask = synthetic_video(distinct + 1, Hc, Wc, OBJS, seed=4321)          # the SAME clip on every rank
    frames = [f.to(dev) for f in frames]
    mask = mask.to(dev)

    def clip(n):
        eng.restart_engine()
        with torch.no_grad():
            eng.add_reference_frame(frames[0], mask, obj_nums=[OBJS], frame_step=0)
            if dist is not None:
                dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for t in range(1, n + 1):
                eng.match_propogate_one_frame(frames[1 + (t - 1) % distinct])
                eng.decode_current_logits(None)
                a0 = eng.aot_engines[0]
                label = torch.empty((1, 1, Hc, Wc), dtype=torch.float32, device=dev)
                ops.logits_argmax(a0.pred_id_logits, label, a0.align_corners)
                eng.update_memory(label)
            e1.record()
            if dist is not None:
                dist.barrier()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    clip(min(n_prop, 26))                     # warm-up: graph capture of both memory-update variants, first bank growth
    ms = clip(n_prop)
    a0 = eng.aot_engines[0]
    rec = {"workload": f"swinb_aotl inference, synthetic 1.3x480p clip (net input {Hc}x{Wc}), {OBJS} objects, 1 reference + "
                       f"{n_prop} propagated frames, long-term gap {cfg.TEST_LONG_TERM_MEM_GAP}, ONE clip on {world} GPU(s)",
           "n_gpus": world, "steps": n_prop, "value": round(n_prop / (ms / 1e3), 3), "unit": "frames/s",
           "ms_per_step": round(ms / n_prop, 4), "scaling": "strong",
           "mode": "bank on one GPU" if world == 1 else
                   f"long-term bank sharded by memory frame over {world} GPUs, " + (
                       "partials in symmetric memory, one device-side barrier per layer, merge reads the peers over NVLink"
                       if os.environ.get("AOTB_SHARD_XCHG", "nccl") == "p2p" else
                       "one packed (O|m|l) NCCL all-gather per layer per frame + exact merge"),
           "memory_frames_end": int(a0._mem_frames), "local_bank_rows_end": int(a0.bank_len), "tokens_per_frame": int(a0.enc_hw)}
    del eng, model, frames
    torch.cuda.empty_cache()
    return rec


def gpu_eager_baseline(model_name, dev, max_frames=12):
    """The reference's algorithm as eager PyTorch on the SAME B200 (SURVEY 0.1: the bar a rewrite has to clear): the
    oracle restatement with device='cuda', fp32, TF32 off, the evaluator's span, inputs resident; a bounded sample of the
    clip.  A baseline arm only -- nothing on the product path touches it."""
    from aot_benchmark_b200 import EngineConfig, build_vos_model
    from oracle import aot_oracle as O
    cfg = EngineConfig("eager", model_name)
    torch.manual_seed(0)
    sd = build_vos_model(cfg.MODEL_VOS, cfg).state_dict()
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        frames, mask = make_clip(max_frames + 1, seed=1234)
        frames = [f.to(dev) for f in frames]
        mask = mask.to(dev)
        oe = O.OracleEngine(sd, O.OracleConfig(model_name), device=dev)

        def one(t):
            oe.match_propogate_one_frame(frames[t])
            lg = oe.decode_current_logits((H_OUT, W_OUT))
            lab = torch.softmax(lg, 1).argmax(1, keepdim=True).float()
            oe.update_memory(F.interpolate(lab, size=oe.input_size_2d, mode="nearest"))

        with torch.no_grad():
            oe.add_reference_frame(frames[0], mask, [OBJS], 0)
            for t in range(1, 4):                      # warm-up (cuDNN autotune, allocator)
                one(t)
            oe.restart_engine()
            oe.add_reference_frame(frames[0], mask, [OBJS], 0)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for t in range(1, max_frames + 1):
                one(t)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        return {"value": round(max_frames / (ms / 1e3), 3), "unit": "frames/s", "kind": "port, eager PyTorch (cuDNN/cuBLAS fp32, TF32 off) on the same GPU",
                "sample": f"frames 1-{max_frames} of the same clip (bank holds <= {1 + max_frames // cfg.TEST_LONG_TERM_MEM_GAP} memory frames)"}
    except Exception as e:                              # a baseline arm must never take the bench line down
        return {"value": None, "error": f"{type(e).__name__}: {e}"[:300]}
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


# ---------------------------------------------------------------------------------------------
def _best_threads(step_fn, candidates):
    """Pick the torch intra-op thread count that runs one propagated frame fastest on this host."""
    best, best_t = candidates[0], float("inf")
    for n in candidates:
        torch.set_num_threads(n)
        t0 = time.perf_counter()
        step_fn()
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def _thread_candidates():
    n = os.cpu_count() or 1
    return sorted({n, max(1, n // 2), min(n, 32), min(n, 16), min(n, 8), min(n, 4)}, reverse=True)


def cpu_baseline(model_name, threads, max_frames=4, budget_s=40.0):
    """The CPU oracle port of the same span on the host cores, on a bounded sample of the clip."""
    from aot_benchmark_b200 import EngineConfig, build_vos_model
    from oracle import aot_oracle as O
    cfg = EngineConfig("cpu", model_name)
    torch.manual_seed(0)
    sd = build_vos_model(cfg.MODEL_VOS, cfg).state_dict()
    frames, mask = make_clip(max_frames + 1, seed=1234)
    oe = O.OracleEngine(sd, O.OracleConfig(model_name))
    n = 0

    def one(t):
        oe.match_propogate_one_frame(frames[t])
        lg = oe.decode_current_logits((H_OUT, W_OUT))
        lab = torch.softmax(lg, 1).argmax(1, keepdim=True).float()
        oe.update_memory(F.interpolate(lab, size=oe.input_size_2d, mode="nearest"))

    with torch.no_grad():
        torch.set_num_threads(threads)
        oe.add_reference_frame(frames[0], mask, [OBJS], 0)
        threads = _best_threads(lambda: one(1), _thread_candidates())
        oe.restart_engine()
        oe.add_reference_frame(frames[0], mask, [OBJS], 0)
        t0 = time.perf_counter()
        for t in range(1, max_frames + 1):
            one(t)
            n += 1
            if time.perf_counter() - t0 > budget_s:
                break
        dt = time.perf_counter() - t0
    return {"value": round(n / dt, 4), "unit": "frames/s", "cores": threads, "kind": "port",
            "sample": f"frames 1-{n} of the same clip (memory bank holds 1 frame; later frames are slower on CPU "
                      f"because long-term attention grows with the bank)"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The reference is pure
    Python and /root/reference does not exist on the GPU box, so this is the oracle port
    (oracle/aot_oracle.py, pinned to the reference by tests/golden) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    from aot_benchmark_b200 import EngineConfig, build_vos_model
    from oracle import aot_oracle as O
    threads = os.cpu_count()
    torch.set_num_threads(threads)
    cfg = EngineConfig("cpu", args.model)
    torch.manual_seed(0)
    sd = build_vos_model(cfg.MODEL_VOS, cfg).state_dict()
    K, Wm = args.steps, args.warmup
    budget = 150.0
    frames, mask = make_clip(min(K, 40) + 1, seed=1234)
    oe = O.OracleEngine(sd, O.OracleConfig(args.model))

    def step(t):
        oe.match_propogate_one_frame(frames[1 + (t - 1) % (len(frames) - 1)])
        lg = oe.decode_current_logits((H_OUT, W_OUT))
        lab = torch.softmax(lg, 1).argmax(1, keepdim=True).float()
        oe.update_memory(F.interpolate(lab, size=oe.input_size_2d, mode="nearest"))

    with torch.no_grad():
        oe.add_reference_frame(frames[0], mask, [OBJS], 0)
        threads = _best_threads(lambda: step(1), _thread_candidates())   # also the warm-up
        oe.restart_engine()
        oe.add_reference_frame(frames[0], mask, [OBJS], 0)
        n, t0 = 0, time.perf_counter()
        for t in range(1, K + 1):
            step(t)
            n += 1
            if time.perf_counter() - t0 > budget:
                break
        dt = time.perf_counter() - t0
    fps = n / dt
    sample = f"first {n} of {K} propagated frames of the same clip (time-capped at {budget:.0f} s), {threads} of {os.cpu_count()} host threads (fastest of the tried counts)"
    print(json.dumps({
        "impl": "reference", "metric": "frames/sec (480p, 10 obj)", "value": round(fps, 4), "unit": "frames/s",
        "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": round(1e3 / fps, 2), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.model} inference, synthetic {'1.3x480p' if H_IN > 481 else '480p'} clip (net input {H_IN}x{W_IN}, output "
                               f"{H_OUT}x{W_OUT}), {OBJS} objects, 1 reference + {K} propagated frames, long-term gap "
                               f"{cfg.TEST_LONG_TERM_MEM_GAP}, batch 1",
                   "weights": "seeded random init"},
        "cpu_baseline": {"value": round(fps, 4), "unit": "frames/s", "cores": threads, "kind": "port",
                         "sample": sample},
        "e2e": {"value": round(fps, 4), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=99)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="r50_aotl")
    ap.add_argument("--mode", default="dp", choices=["dp", "shard"],
                    help="dp: one clip per GPU (default, weak scaling); shard: one clip, long-term bank sharded over the "
                         "ranks with an NCCL exchange of the attention partials per layer (BASELINE configs[3], strong scaling)")
    ap.add_argument("--cfg4-frames", type=int, default=int(os.environ.get("AOTB_BENCH_CFG4_FRAMES", "500")),
                    help="propagated frames of the additional BASELINE configs[3] record (SwinB-AOTL, one clip, long-term bank "
                         "sharded over the GPUs when N > 1); 0 disables it")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the label map and logits of the value pass's last timed step to DIR/<name>.npy (float32)")
    ap.add_argument("--skip-cpu-baseline", action="store_true",
                    help="development only: omit the cpu_baseline leg (the driver's default run keeps it)")
    args = ap.parse_args()
    set_workload(args.model)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
