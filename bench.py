"""bench.py - images/sec of LMD+ (SD1.4/1.5 + GLIGEN shapes, fp16 activations / fp32 accumulate, 512x512, 50 steps,
4 boxes per prompt, 8 prompts per GPU) through lgd_b200.generation.lmd_plus.run_batch, plus the tensor-pipe roofline
of the cross-attention+loss op and the reference's CPU path timed on the host cores.

One "step" = one full batch of 8 images (Phase A: 32 per-box generations x 50 CFG steps with GLIGEN fusers for the first
40 %; composition; Phase B: 8 overall generations x 50 CFG steps + attention-guidance forward/backward iterations for
index < 30 + reference-attention transfer; every generation ends in the B200 VAE decode, `--vae 0` leaves it out).
Synthetic data: seeded random weights with the real layer shapes, seeded text embeddings, seeded layouts (no checkpoints,
vocabularies or datasets exist offline).  CLIP / SAM are outside the measured path (SURVEY.md section 8: out of scope /
"next"); the SAM mask is the box raster.  The headline `value` is
the fixed-iteration mode (B) of SURVEY.md section 8d - overall_loss_threshold=0, so every image runs all 65 guidance
iterations and the FLOPs behind the number are known; mode (A), the reference's data-dependent thresholds, is timed
beside it (`mode_a`) with its per-image iteration counts.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]
"""
import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOAD = "LMD+ SD1.5(+GLIGEN shapes) 512x512, 50 steps, 4 boxes/prompt, 8 prompts/GPU"
NAMES = ["a red ball", "a blue cube", "a green vase", "a yellow lamp", "a wooden chair", "a black cat", "a white dog",
         "a purple flower", "a silver car", "an orange bird"]


_T0 = time.time()


def log(msg):
    print(f"[bench +{time.time() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


def make_specs(batch, boxes, seed):
    rng = random.Random(seed)
    specs = []
    for _ in range(batch):
        names = rng.sample(NAMES, boxes)
        gb = []
        for n in names:
            w, h = rng.uniform(0.2, 0.5), rng.uniform(0.2, 0.5)
            x, y = rng.uniform(0, 1 - w), rng.uniform(0, 1 - h)
            gb.append((n, [int(x * 512), int(y * 512), int(w * 512), int(h * 512)]))
        specs.append(dict(prompt="", gen_boxes=gb, bg_prompt="a realistic photo of a living room", extra_neg_prompt=""))
    return specs


class Clocks(threading.Thread):
    """nvidia-smi sampler running during the timed region (B200_PROFILING.md recipe)"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.5)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = max([int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()] or [0])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": reasons}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["bf16_tflops"], d["hbm_gbs"], "measured"
    return 1590.0, 6650.0, "fallback"


def ncu_dram_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE xattn_fused_kernel launch at the roofline shape, read from the
    committed export of the `ncu --set full` capture (profiles/xattn_fused_ncu_raw.csv, written by
    profiles/ncu_extract.py from the .ncu-rep of `profiles/bench_xattn.py`); None when no capture is committed."""
    import csv
    path = os.path.join(ROOT, "profiles", "xattn_fused_ncu_raw.csv")
    if not os.path.exists(path):
        return None, None
    tot, n = 0.0, 0
    with open(path) as f:
        for row in csv.DictReader(f):
            if "xattn_fused_kernel" not in row.get("kernel", ""):
                continue
            tot += float(row["dram_bytes_read"]) + float(row["dram_bytes_write"])
            n += 1
    return (tot / n, os.path.relpath(path, ROOT)) if n else (None, None)


def xattn_roofline(dev, with_loss=True):
    """the fused cross-attention+loss kernel at the config's guidance shape (B=8, n=256, C=1280, heads 8, T=77):
    algorithmic FLOPs 2nC^2 (to_q) + 2nTC (QK^T) + 2nTC (PV) + 2nC^2 (to_out) per sample (SURVEY.md section 8d), one
    launch, timed with CUDA events on the launching stream, L2 flushed between repetitions."""
    from lgd_b200 import guidance as G, ops
    B, heads, d, n, T, ctx = 8, 8, 160, 256, 77, 768
    C = heads * d
    g = torch.Generator(device="cpu").manual_seed(0)
    x = torch.randn(B * n, C, generator=g).half().to(dev)
    text = torch.randn(B * T, ctx, generator=g).half().to(dev)
    wq = (torch.randn(C, C, generator=g) * 3 / C ** 0.5).half().to(dev)
    wkv = (torch.randn(2 * C, ctx, generator=g) * 2 / ctx ** 0.5).half().to(dev)
    wo = (torch.randn(C, C, generator=g) / C ** 0.5).half().to(dev)
    bo = torch.zeros(C, device=dev)
    dp, d16 = ops.round_dp(d), ops.round_d16(d)
    z = lambda *s: torch.zeros(*s, device=dev, dtype=torch.float16)
    q = z(B * heads, n, dp)
    k, v, kt, vt = z(B * heads, 80, dp), z(B * heads, 80, dp), z(B * heads, d16, 80), z(B * heads, d16, 80)
    ops.project_heads2(text, wkv, T, heads, d, 1, rm=(None, k, v), tr=(None, kt, vt))
    rng = random.Random(0)
    lay = []
    for b in range(B):
        bx, pos = [], []
        for o in range(4):
            w_, h_ = rng.uniform(0.2, 0.5), rng.uniform(0.2, 0.5)
            x0, y0 = rng.uniform(0, 1 - w_), rng.uniform(0, 1 - h_)
            bx.append([(x0, y0, x0 + w_, y0 + h_)])
            pos.append([2 * o + 1, 2 * o + 2])
        lay.append(G.SampleLayout(bx, pos, [p[-1] for p in pos]))
    params = G.LossParams(loss_scale=5.0, fg_weight=1.0, bg_weight=4.0)
    st, so = G.assign_slots(lay, params)
    kl = G.KeyLoss(lay, torch.from_numpy(st).to(dev), so, ("up", 1, 0, 0), n, heads, 4, params, dev, gscale=256.0)
    flush = torch.empty(1024 * 1024 * 1024, dtype=torch.uint8, device=dev)
    res = x.clone()

    def op():      # ONE launch: xattn_fused_kernel (to_q, QK^T, softmax, loss + dP, PV, to_out + bias + residual)
        return ops.xattn_fused(x, wq, k, vt, wo, bo, res, B, n, heads, d, T, d ** -0.5, loss=kl if with_loss else None)[0]

    for _ in range(3):
        op()
    torch.cuda.synchronize()
    # device time of the launch: the L2 flush (1 GiB memset, > 126 MB L2, ~300 us) is still running while the host
    # enqueues event / launch / event behind it, so the events bracket the kernel alone with no host launch latency in
    # between (the kernel's hand-shake counters reset themselves: nothing else is launched)
    def isolated(fn, reps=20):
        times = []
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        return sum(times) / reps, times

    ms, times = isolated(op)
    if os.environ.get("B200_BENCH_VERBOSE"):
        print("xattn reps (ms):", [round(t, 4) for t in times], file=sys.stderr)
    flops = B * (2 * n * C * C * 2 + 2 * n * T * C * 2)
    peak, _, how = peaks()
    ach = flops / (ms * 1e-3) / 1e12
    traffic, traffic_src = ncu_dram_traffic()
    out = {"bound": "tensor", "achieved": round(ach, 2), "peak": peak, "unit": "TFLOP/s", "frac": round(ach / peak, 4),
           "traffic": traffic, "traffic_source": traffic_src,
           "kernel": "xattn_fused_kernel (projections + attention + guidance loss)",
           "launches_per_op": 1, "ms_per_op": round(ms, 4),
           "peak_source": how + " (burst, kernel timed alone before the step loop)",
           "shape": {"B": B, "n": n, "C": C, "heads": heads, "T": T}}
    if not with_loss:
        return out
    # context for the floor model (DESIGN.md), not the headline: (1) an EMPTY kernel with the same launch configuration,
    # bracketed the same way = the launch + drain share of ms_per_op; (2) the kernel launched back to back over rotating
    # input sets larger than L2 (8 x (x, Wq, Wo, residual) = 136 MB; outputs from the caching allocator), one event pair
    # around one CUDA-graph replay of 96 launches = its duration inside a stream of kernels (how the step runs it)
    import ctypes
    from lgd_b200._lib import check, cur_stream, lib
    n_ctas = B * n // 128 * heads

    def null_launch():
        check(lib().b200lmd_xattn_fused_launch_floor(ctypes.c_int(d), ctypes.c_int(n_ctas), cur_stream()))

    floor_ms, _ = isolated(null_launch)
    sets = [(x.clone(), wq.clone(), wo.clone(), res.clone()) for _ in range(8)]

    def run(i):
        xs, wqs, wos, rs = sets[i % 8]
        return ops.xattn_fused(xs, wqs, k, vt, wos, bo, rs, B, n, heads, d, T, d ** -0.5, loss=kl)

    for i in range(8):
        run(i)
    torch.cuda.synchronize()
    R = 96
    gr = torch.cuda.CUDAGraph()          # the step runs its kernels from CUDA graphs too: no host gaps between launches
    with torch.cuda.graph(gr):
        for i in range(R):
            run(i)
    gr.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    flush.zero_()
    e0.record()
    gr.replay()
    e1.record()
    torch.cuda.synchronize()
    bb = e0.elapsed_time(e1) / R
    out["launch_floor_ms"] = round(floor_ms, 4)
    out["back_to_back"] = {"ms_per_op": round(bb, 4), "frac": round(flops / (bb * 1e-3) / 1e12 / peak, 4), "launches": R,
                           "inputs": "8 rotating sets of (x, Wq, Wo, residual), 136 MB > L2"}
    return out


# forward passes of ONE LMD+ image at the bench configuration (4 boxes, 50 steps, GLIGEN fusers on for the first 40 % of
# the steps, models/pipelines.py:408) in fixed-iteration mode: Phase A 4 x 50 CFG passes, Phase B 50 CFG passes and
# sum(max_iter[:30]) = 65 guidance iterations (55 of them in the steps with the fusers on)
N_CFG_ON, N_CFG_OFF, N_GUID_ON, N_GUID_OFF = 5 * 20, 5 * 30, 55, 10
FUSER_OFF_RATIO = 803.0 / 1137.0      # FLOPs of a forward without / with the GLIGEN fusers (SURVEY.md section 8d)


class CpuArm:
    """the reference's CPU path (oracle restatement of its UNet / loss / autograd guidance step in fp32 PyTorch, pinned
    to the unmodified reference in the build container) on this box's host cores, at SD1.5+GLIGEN shapes"""

    def __init__(self):
        from oracle import unet_ref
        self.cores = min(os.cpu_count() or 1, 64)       # beyond ~64 threads the fp32 conv/GEMM kernels stop scaling
        torch.set_num_threads(self.cores)
        self.cfg = unet_ref.UNetConfig.sd15(gligen=True)
        self.w = unet_ref.make_weights(self.cfg, seed=0)
        g = torch.Generator().manual_seed(0)
        self.z = torch.randn(1, 4, 64, 64, generator=g)
        self.ctx = torch.randn(2, 77, 768, generator=g)
        self.gl = dict(boxes=torch.rand(2, 30, 4, generator=g), masks=torch.zeros(2, 30),
                       positive_embeddings=torch.randn(2, 30, 768, generator=g))
        self.gl["masks"][1, :4] = 1
        self.keys = [("mid", 0, 0, 0), ("up", 1, 0, 0), ("up", 1, 1, 0), ("up", 1, 2, 0)]

    def cond_forward(self):
        """one conditional batch-1 forward (fusers on)"""
        from oracle import unet_ref
        t0 = time.time()
        with torch.no_grad():
            unet_ref.unet_forward(self.w, self.cfg, self.z, 500, self.ctx[1:], gligen={k: v[1:] for k, v in self.gl.items()})
        return time.time() - t0

    def cfg_forward(self):
        """one classifier-free-guidance pass: batch 2 = [uncond; cond] (models/pipelines.py:420)"""
        from oracle import unet_ref
        t0 = time.time()
        with torch.no_grad():
            unet_ref.unet_forward(self.w, self.cfg, torch.cat([self.z, self.z]), 500, self.ctx, gligen=self.gl)
        return time.time() - t0

    def guidance_iteration(self):
        """one guidance iteration the way the reference runs it (models/pipelines.py:30-69): full cond-only forward
        with the 4 guidance maps saved, compute_ca_lossv3 with 4 phrases, autograd to the latent, latent update"""
        from oracle import guidance_ref, unet_ref
        t0 = time.time()
        zz = self.z.clone().requires_grad_(True)
        saved = {}
        unet_ref.unet_forward(self.w, self.cfg, zz, 500, self.ctx[1:], gligen={k: v[:1] for k, v in self.gl.items()},
                              saved=saved, save_keys=self.keys)
        bboxes = [[(0.1, 0.1, 0.4, 0.5)], [(0.5, 0.1, 0.9, 0.4)], [(0.1, 0.6, 0.45, 0.95)], [(0.55, 0.5, 0.95, 0.9)]]
        pos = [[1, 2], [3, 4], [5, 6], [7, 8]]
        L = guidance_ref.ca_loss({k: v[0] for k, v in saved.items()}, bboxes, pos, self.keys, 0.2, 0.2, 1.0, 4.0) * 5.0
        grad = torch.autograd.grad(L, [zz])[0]
        _ = (zz - 0.5 * grad).detach()
        return time.time() - t0


def cpu_image_seconds(t_cfg, t_guid):
    """extrapolation of the timed samples to one LMD+ image (fusers-off passes scaled by the FLOP ratio)"""
    return (N_CFG_ON + N_CFG_OFF * FUSER_OFF_RATIO) * t_cfg + (N_GUID_ON + N_GUID_OFF * FUSER_OFF_RATIO) * t_guid


def cpu_baseline():
    """bounded sample on the host cores: ONE CFG pass (batch 2) and ONE real guidance iteration (forward + autograd
    backward + update), after one warm-up forward; extrapolated to one image by the pass counts of the workload."""
    arm = CpuArm()
    arm.cond_forward()                               # warm-up (thread pool, allocator)
    t_cfg = arm.cfg_forward()
    t_guid = arm.guidance_iteration()
    sec = cpu_image_seconds(t_cfg, t_guid)
    return {"value": 1.0 / sec, "unit": "images/s", "cores": arm.cores, "kind": "port",
            "extrapolated": True, "t_cfg_pass_s": round(t_cfg, 3), "t_guidance_iteration_s": round(t_guid, 3),
            "sample": f"1 CFG pass (batch 2, {t_cfg:.2f} s) + 1 guidance iteration (forward + autograd backward, "
                      f"{t_guid:.2f} s) of the fp32 oracle at SD1.5+GLIGEN shapes; EXTRAPOLATED to one LMD+ image = "
                      f"{N_CFG_ON}+{N_CFG_OFF} CFG passes and {N_GUID_ON}+{N_GUID_OFF} guidance iterations with / without "
                      f"fusers (fusers-off passes scaled by the FLOP ratio {FUSER_OFF_RATIO:.3f}) = {sec:.0f} s"}


def reference_arm(args, config):
    """--impl reference: the reference's CPU implementation of the path (oracle port - the reference is Python and
    its third-party model code cannot be installed here, DESIGN.md section 1) on the host cores.  Each timed step is a
    bounded sample of the workload - one conditional UNet forward at SD1.5+GLIGEN shapes - and the per-image figure
    uses the MEASURED cost ratios of a CFG pass and of a real guidance iteration (timed once) to that sample."""
    arm = CpuArm()
    for _ in range(max(1, min(args.warmup, 3))):
        arm.cond_forward()
    t_cfg = arm.cfg_forward()
    t_guid = arm.guidance_iteration()
    t1 = arm.cond_forward()
    r_cfg, r_guid = t_cfg / t1, t_guid / t1
    budget_s = 240.0
    k = max(1, min(args.steps, int(budget_s / max(t1, 1e-3))))
    ts = [arm.cond_forward() for _ in range(k)]
    t_fwd = sum(ts) / k
    sec = cpu_image_seconds(r_cfg * t_fwd, r_guid * t_fwd)
    base = {"value": 1.0 / sec, "unit": "images/s", "cores": arm.cores, "kind": "port", "extrapolated": True,
            "sample": f"{k} timed batch-1 conditional forwards ({t_fwd:.2f} s each); a CFG pass costs {r_cfg:.2f} and a "
                      f"guidance iteration (forward + autograd backward) {r_guid:.2f} of those (both timed once); "
                      f"EXTRAPOLATED to one LMD+ image = {sec:.0f} s"}
    line = {"metric": "images/sec (LMD+ SD1.5, 50 steps, 512^2)", "value": base["value"], "unit": "images/s",
            "n_gpus": args.gpus, "steps": k, "warmup": args.warmup, "ms_per_step": t_fwd * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "impl": "reference", "config": config, "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


DUMP_BYTES = 64 << 20          # --dump-outputs budget
IMAGE_VALUES = 8 << 20         # decoded images up to this many values are written whole (32 MB as float32) ...
IMAGE_SAMPLE = 2 << 20         # ... larger ones as a sample of this many (value + index: 24 MB)
SO_IMAGE_SAMPLE = 1 << 20      # the per-box images are always sampled (all of them: 32 x 512 x 512 x 3 values)


def seeded_sample(name, a, n_whole, n_sample, out):
    """out[name] = a as float32 when it has at most n_whole values, else a fixed seeded sample of n_sample values in
    out[name + "_sample"] with their flat indices in out[name + "_index"]: same arguments, same indices"""
    import numpy as np
    flat = np.ascontiguousarray(a).reshape(-1)
    if flat.size <= n_whole:
        out[name] = flat.reshape(a.shape).astype(np.float32)
        return
    idx = np.sort(np.random.default_rng(0).choice(flat.size, min(n_sample, flat.size), replace=False))
    out[name + "_sample"] = flat[idx].astype(np.float32)
    out[name + "_index"] = idx.astype(np.float64)


def step_outputs(outs, iters):
    """what one step's run_batch call handed back, on the host: the final latents [B, 4, h, w], the decoded images
    [B, H, W, 3] (0..255), the per-box images of phase A (sampled) and the guidance iterations of every image"""
    import numpy as np
    d = {"latents": torch.cat([o["latents"] for o in outs], 0).float().cpu().numpy(),
         "guidance_iterations": np.asarray(iters, dtype=np.float64)}
    if outs[0].image is not None:
        seeded_sample("images", np.stack([o.image for o in outs]), IMAGE_VALUES, IMAGE_SAMPLE, d)
    so = [im for o in outs for im in (o.so_img_list or [])]
    if so:
        seeded_sample("so_images", np.stack(so), 0, SO_IMAGE_SAMPLE, d)
    return d


def write_outputs(path, arrays):
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_BYTES, f"--dump-outputs: {total} bytes > {DUMP_BYTES}"
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--boxes", type=int, default=4)
    ap.add_argument("--denoise-steps", type=int, default=50)
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-mode-a", action="store_true")
    ap.add_argument("--workload", default="lmd_plus", choices=["lmd_plus", "backward_guidance_sd21", "boxdiff"],
                    help="lmd_plus = BASELINE config 2 (the headline, default); backward_guidance_sd21 = config 3 (SD2.1 "
                         "shapes, 768x768, v-prediction, batch 4); boxdiff = config 4 (SD1.5, 25 guided steps, batch 8)")
    ap.add_argument("--vae", type=int, default=int(os.environ.get("B200_BENCH_VAE", "1")),
                    help="1: decode every per-box and overall generation with the B200 VAE decoder (synthetic weights) "
                         "inside the timed step, as models/pipelines.py:233,461,591 do")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (final latents, decoded images, a seeded sample of "
                         "the per-box images, guidance iteration counts) as DIR/<name>.npy, float32/float64, <= 64 MB")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the B200 path computed; --impl reference times a sample of the CPU path")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    config = {"workload": WORKLOAD, "batch_per_gpu": args.batch, "boxes_per_prompt": args.boxes,
              "denoise_steps": args.denoise_steps,
              "guidance": "mode B (SURVEY 8d): overall_loss_threshold=0 -> fixed sum(max_iter[:30]) = 65 guidance "
                          "iterations per image; mode A (reference thresholds, data-dependent counts) in `mode_a`",
              "l2": "inputs exceed L2 (per-step activations >> 126 MB)", "parallelism": f"dp{world}",
              "unit_note": "an 'image' is the final latent [4,64,64] of one prompt: CLIP/VAE/SAM are outside the "
                           "measured path (SAM mask = box raster)"}

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, config)
        return

    import lgd_b200
    from lgd_b200 import _lib, weights as Wt
    from lgd_b200.env import SyntheticEnv
    from lgd_b200.generation import common, lmd_plus
    from lgd_b200.unet import B200UNet, UNetConfig
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    from lgd_b200 import parallel
    import torch.distributed as dist
    parallel.init("nccl", dev)
    pin = parallel.pin_host_threads(local, min(world, torch.cuda.device_count()))
    wl = args.workload
    cfg = {"lmd_plus": UNetConfig.sd15(gligen=True), "backward_guidance_sd21": UNetConfig.sd21(),
           "boxdiff": UNetConfig.sd15()}[wl]
    if wl == "backward_guidance_sd21":
        if args.batch == 8:
            args.batch = 4
        config.update(workload="backward guidance (ratio energy) SD2.1 shapes 768x768 v-prediction, 50 steps, 5 guidance "
                               "iterations x 10 steps, 4 boxes/prompt, 4 prompts/GPU (BASELINE config 3)",
                      guidance="overall_loss_threshold=0: fixed 5 x 10 = 50 guidance iterations per image")
    elif wl == "boxdiff":
        config.update(workload="BoxDiff SD1.5 512x512, 50 steps, 25 guided steps x 1 iteration, 4 boxes/prompt, 8 "
                               "prompts/GPU (BASELINE config 4)", guidance="fixed 25 BoxDiff steps per image")
    # the only collective on the path: start-up NCCL broadcast of the frozen weights from rank 0
    w = parallel.broadcast_weights(Wt.parameter_shapes(cfg), lambda: Wt.synthetic_weights(cfg, seed=0, device=dev), dev)
    log("weights ready")
    net = B200UNet(cfg, w, dev)
    del w
    log("unet prepared")
    specs = make_specs(args.batch, args.boxes, seed=1000 + rank)
    seeds = [rank * 1000 + i for i in range(args.batch)]
    fgs = [s + 123456789 for s in seeds]
    io = {"h2d": 0, "d2h": 0}
    last = {}

    def step(env, fixed=True):
        common.configure(net, env)
        kw = dict(overall_loss_threshold=0.0) if fixed else {}
        if wl == "lmd_plus":
            outs = lmd_plus.run_batch(specs, seeds, fgs, num_inference_steps=args.denoise_steps, return_latents=True, **kw)
        elif wl == "backward_guidance_sd21":
            from lgd_b200.generation import backward_guidance
            outs = backward_guidance.run_batch(specs, seeds, num_inference_steps=args.denoise_steps, height=768, width=768,
                                               prediction_type="v_prediction", return_latents=True, **kw)
        else:
            from lgd_b200.generation import boxdiff as boxdiff_plugin
            outs = boxdiff_plugin.run_batch(specs, seeds, num_inference_steps=args.denoise_steps, return_latents=True)
        lat = torch.cat([o["latents"] for o in outs], 0)
        host = lat.cpu()                                  # device -> host read of the step's result
        io["d2h"] = host.numel() * host.element_size()
        if outs[0].image is not None:                     # decoded pictures already crossed to the host in env.decode
            io["d2h"] += sum(o.image.nbytes + sum(im.nbytes for im in (o.so_img_list or [])) for o in outs)
        if args.dump_outputs:
            last["outs"] = outs
        st = outs[0]["guidance_state"]
        if wl == "boxdiff":
            last["iters"] = [len(getattr(st, "boxdiff_losses", []))] * len(outs)
        else:
            last["iters"] = [int(sum(it[b] for it in st.iters)) for b in range(len(outs))]
        return host

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(env, k, fixed=True):
        barrier()
        # only rank 0 samples clocks (its own GPU): eight ranks each forking nvidia-smi five times a second is host
        # load that competes with the ranks' launch loops
        clk = Clocks(local)
        if rank == 0:
            clk.start()
        n0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            step(env, fixed)
        e1.record()
        barrier()
        clk.stop_flag = True
        ms = e0.elapsed_time(e1)
        return parallel.max_over_ranks(ms, dev), _lib.launch_count() - n0, clk.summary()

    vae = None
    ctx_dim = cfg.cross_attention_dim
    if args.vae:
        from lgd_b200.vae import B200VAEDecoder, VAEConfig
        vae = B200VAEDecoder(VAEConfig(), Wt.synthetic_vae_weights(VAEConfig(), seed=0, device=dev), dev)
        config["unit_note"] = ("an 'image' is the decoded uint8 512x512x3 picture: every per-box and overall generation "
                               "ends in the B200 VAE decode (synthetic weights); CLIP / SAM are outside the measured path")
    env_res = SyntheticEnv(ctx_dim=ctx_dim, cache_device=dev, vae_decoder=vae)    # inputs resident in HBM
    env_host = SyntheticEnv(ctx_dim=ctx_dim, cache_device=None, vae_decoder=vae)  # inputs produced on the host (pinned)
    roofline = None
    if rank == 0 and not args.no_roofline and wl == "lmd_plus":
        # the kernel-alone measurement runs BEFORE the step loop: its denominator is the burst peak (a kernel timed
        # alone on an idle GPU); after 90 s of sustained load the same launch measures 5-10 % slower (power state)
        roofline = xattn_roofline(dev)
        log("roofline micro-benchmark done")
    for i in range(args.warmup):
        step(env_res)
        torch.cuda.synchronize()
        log(f"warm-up step {i} done")
    ms, launches, clocks = timed(env_res, args.steps)
    iters_b = list(last["iters"])
    dump = step_outputs(last.pop("outs"), iters_b) if args.dump_outputs else None
    log(f"timed (resident inputs, fixed 65 iterations): {ms:.1f} ms for {args.steps} step(s)")
    env_host.bytes_out = 0
    k_e2e = min(args.steps, 8)             # bounded: the end-to-end leg repeats the same step with host inputs
    ms_e2e, _, _ = timed(env_host, k_e2e)
    log(f"timed (host inputs, e2e): {ms_e2e:.1f} ms for {k_e2e} step(s)")
    io["h2d"] = env_host.bytes_out // max(1, k_e2e)
    imgs = args.batch * world * args.steps
    metric = {"lmd_plus": "images/sec (LMD+ SD1.5, 50 steps, 512^2)",
              "backward_guidance_sd21": "images/sec (backward guidance SD2.1 shapes, 50 steps, 768^2)",
              "boxdiff": "images/sec (BoxDiff SD1.5, 50 steps, 512^2)"}[wl]
    line = {"metric": metric, "value": imgs / (ms * 1e-3), "unit": "images/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": config, "clocks": clocks, "gpu_launches": launches,
            "guidance_iterations_per_image": iters_b, "host_threads": pin,
            "e2e": {"value": args.batch * world * k_e2e / (ms_e2e * 1e-3), "unit": "images/s", "steps": k_e2e,
                    "h2d_bytes_per_step": io["h2d"], "d2h_bytes_per_step": io["d2h"]}}
    if not args.no_mode_a and wl == "lmd_plus":
        step(env_res, fixed=False)                  # graphs / tables of the data-dependent variant
        ms_a, _, _ = timed(env_res, 1, fixed=False)
        line["mode_a"] = {"value": args.batch * world / (ms_a * 1e-3), "unit": "images/s", "ms_per_step": ms_a,
                          "steps": 1, "guidance_iterations_per_image": list(last["iters"]),
                          "note": "reference thresholds (overall_loss_threshold 5.0): data-dependent iteration counts"}
        log(f"timed (mode A): {ms_a:.1f} ms")
    if rank == 0:
        if roofline is not None:
            line["roofline"] = roofline
        if world == 1 and not args.no_cpu_baseline and wl == "lmd_plus":
            line["cpu_baseline"] = cpu_baseline()
            log("cpu baseline done")
        print(json.dumps(line))
        if dump is not None:
            write_outputs(args.dump_outputs, dump)
            log(f"outputs of the last timed step written to {args.dump_outputs}")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
