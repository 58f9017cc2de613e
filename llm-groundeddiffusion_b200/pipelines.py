"""Host mirror of the reference's denoising loops (models/pipelines.py) over the B200 UNet.

One batched, timestep-synchronous `denoise` covers generate_semantic_guidance (:129-247), generate_gligen (:324-473) and
generate_partial_frozen (:541-599); `latent_backward_guidance` (:16-82) becomes a per-image-predicated loop around
B200UNet.guidance_gradient (no autograd).  The reference is batch-1 (utils/guidance.py:264 squeezes the batch); here B
independent (prompt, layout) pairs advance together and every data-dependent decision of the reference is kept PER
IMAGE:
  * stale-loss loop entry and permanent stop below threshold            pipelines.py:30,161,375,552
  * max_iter list indexed by step, last element reused                  pipelines.py:21-25
  * step scale sqrt(1 - alpha_bar_t) (DDIM has no sigmas)               pipelines.py:60-69
  * CFG batch order [uncond; cond]; guidance pass is cond-only          pipelines.py:44,420; models/models.py:85
  * GLIGEN: fuser on for index < int(beta*steps); the guidance pass sees the zeroed grounding-mask half
                                                                        pipelines.py:317,382-384,408-414
  * frozen blend with latents_all_input[index+1]                        pipelines.py:445-446
The only host<->device traffic inside a step is the per-image loss read-back that the reference also performs
(loss.item(), pipelines.py:30).
"""
import ctypes
import gc
import os
import sys
import time
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import guidance as G
from ._lib import check, cur_stream, lib, ptr

_i, _f = ctypes.c_int, ctypes.c_float

DEFAULT_GUIDANCE_ATTN_KEYS = [("mid", 0, 0, 0), ("up", 1, 0, 0), ("up", 1, 1, 0), ("up", 1, 2, 0)]


class DDIMSchedule:
    """diffusers 0.18 DDIMScheduler arithmetic (scaled_linear 0.00085..0.012, 1000 steps, steps_offset 1,
    set_alpha_to_one False, eta 0) - host scalars only; the update itself runs in cfg_ddim_blend_kernel."""

    def __init__(self, prediction_type="epsilon"):
        betas = np.linspace(0.00085 ** 0.5, 0.012 ** 0.5, 1000, dtype=np.float32) ** 2
        self.alphas_cumprod = np.cumprod((1.0 - betas).astype(np.float32), dtype=np.float32)
        self.final_alpha_cumprod = self.alphas_cumprod[0]
        self.prediction_type = prediction_type
        self.init_noise_sigma = 1.0
        self.num_inference_steps = None
        self.timesteps = None
        self.sigmas = None       # set to an array to take the sigma branch of the guidance step (pipelines.py:60-61)

    def set_timesteps(self, n):
        self.num_inference_steps = n
        self.timesteps = (np.arange(0, n) * (1000 // n)).round()[::-1].astype(np.int64) + 1

    def apply_fast_schedule(self, fast_after_steps, fast_rate=2):
        """utils/schedule.py:4-9 get_fast_schedule: keep the first `fast_after_steps` timesteps, then every
        `fast_rate`-th of the rest (starting one past the cut)."""
        ts = self.timesteps
        if fast_after_steps >= len(ts) - 1:
            return
        self.timesteps = np.concatenate([ts[:fast_after_steps], ts[fast_after_steps + 1::fast_rate]])

    def adjust(self, index, t):
        """utils/schedule.py:11-19 dynamically_adjust_inference_steps: the DDIM step lands on the next listed timestep
        (prev_timestep = t - 1000 // num_inference_steps), -1 past the end."""
        prev_t = int(self.timesteps[index + 1]) if index + 1 < len(self.timesteps) else -1
        self.num_inference_steps = 1000 // (int(t) - prev_t)

    def coefs(self, t):
        prev_t = int(t) - 1000 // self.num_inference_steps
        a_t = float(self.alphas_cumprod[int(t)])
        a_p = float(self.alphas_cumprod[prev_t]) if prev_t >= 0 else float(self.final_alpha_cumprod)
        return a_t ** 0.5, (1 - a_t) ** 0.5, a_p ** 0.5, (1 - a_p) ** 0.5


@dataclass
class GuidanceSpec:
    """semantic_guidance_kwargs of the reference for a batch of images (generation/lmd_plus.py:477-497)"""
    layouts: List[G.SampleLayout]              # per image: bboxes / object_positions / word tokens
    keys: list = field(default_factory=lambda: list(DEFAULT_GUIDANCE_ATTN_KEYS))
    loss_scale: float = 30.0
    loss_threshold: float = 0.2
    max_iter: object = 5
    max_index_step: int = 10
    fg_top_p: float = 0.2
    bg_top_p: float = 0.2
    fg_weight: float = 1.0
    bg_weight: float = 1.0
    ref_ca_loss_weight: float = 1.0
    ref_word_token_only: bool = False
    use_ratio_based_loss: bool = False     # utils/guidance.py:122-128 (what backward_guidance.py runs)
    # ref_maps[b][phrase][box][step] -> {key: array/tensor [heads, n]} or None
    ref_maps: Optional[list] = None


class CudaGraph:
    """capture a launch-only callable once (after an eager warm-up run) and replay it; all tensors it touches must be
    static (updated in place between replays)"""

    capture_seconds = 0.0      # wall time spent warming + capturing (B200_TIMING bookkeeping)

    def __init__(self, fn, key=None, owner=None):
        """key: identifies the launch sequence; owner: the object whose one-time state the sequence initialises (the
        B200UNet).  The warm-up record lives ON the owner (not in a process-wide set keyed by id(), which a new object
        can alias after garbage collection): first use of a sequence always runs once eagerly, so kernel attributes,
        the fused kernel's scratch and the slab cache are set up outside capture."""
        t0 = time.perf_counter()
        warmed = owner.__dict__.setdefault("_graph_warm_keys", set()) if owner is not None else None
        if warmed is None or key is None or key not in warmed:
            fn()                               # first use of this launch sequence: eager run (one-time kernel
            torch.cuda.synchronize()           # attributes, driver entry points, allocator warm-up)
            if warmed is not None and key is not None:
                warmed.add(key)
        self.graph = torch.cuda.CUDAGraph()
        # one memory pool per owner for all of its live graphs: a capture then reuses the blocks earlier captures left in
        # the pool instead of cudaMalloc-ing every intermediate again (the graphs replay on one stream, never
        # concurrently, and their outputs stay referenced, so sharing is safe).  A pool handle is only valid while at
        # least one graph captured into it is alive, so the owner tracks its live graphs and takes a fresh handle when
        # the last one has gone.
        pool = None
        if owner is not None:
            import weakref
            rec = owner.__dict__.get("_graph_pool")
            if rec is None or len(rec[1]) == 0:
                rec = owner.__dict__["_graph_pool"] = (torch.cuda.graph_pool_handle(), weakref.WeakSet())
            pool = rec[0]
            rec[1].add(self)
        # no garbage collection while capturing: torch.cuda.graph does not collect before capture_begin, so a collection
        # triggered inside the capture would run the finalizers of dead objects (graphs and buffers of earlier nets),
        # and their CUDA calls invalidate the capture
        gc_was_enabled = gc.isenabled()
        gc.disable()
        try:
            with torch.cuda.graph(self.graph, pool=pool):
                self.out = fn()
        finally:
            if gc_was_enabled:
                gc.enable()
        CudaGraph.capture_seconds += time.perf_counter() - t0

    def __call__(self):
        self.graph.replay()
        return self.out


class GuidanceState:
    """loss carried across steps per image (the reference's `loss` variable, initialised to 10000.)"""

    def __init__(self, B):
        self.loss = np.full(B, 10000.0, dtype=np.float64)
        self.trace = []          # (index, iteration, [loss per image], [active per image])
        self.iters = []
        self.losses = None       # device loss tables, built at the first guided iteration and reused
        self.graphs = {}         # fuser_on -> CudaGraph of the guidance forward+backward
        self.t_dev = None
        self.ctx = None          # DenoiseCtx: static buffers + captured graphs that survive across denoise() calls


def _heads_of(net, key):
    cfg = net.cfg
    if key[0] == "mid":
        return cfg.heads[-1]
    if key[0] == "down":
        return cfg.heads[key[1]]
    return list(reversed(cfg.heads))[key[1]]


def _tokens_of(net, key, H, W):
    cfg = net.cfg
    nb = len(cfg.block_out_channels)
    level = {"down": key[1], "mid": nb - 1, "up": nb - 1 - key[1]}[key[0]]
    return (H >> level) * (W >> level)


def build_losses(net, spec: GuidanceSpec, index, H, W, dev, reuse=None):
    """device loss tables of every guidance key (KeyLoss.set_step refreshes the per-step reference maps in place).
    reuse: (losses dict, slot_tok_dev) of an earlier batch with the same shape - refilled in place when the new tables
    fit, so the CUDA graphs that captured their addresses stay valid.  Returns (losses, slot_tok_dev, reused)."""
    B = len(spec.layouts)
    use_ref = spec.ref_maps is not None
    layouts = []
    for b, lay in enumerate(spec.layouts):
        refs = spec.ref_maps[b] if use_ref else None       # [phrase][box] -> list over steps of {key: [heads, n]}
        layouts.append(G.SampleLayout(lay.bboxes, lay.object_positions, lay.word_token_indices, refs))
    params = G.LossParams(spec.loss_scale, spec.fg_top_p, spec.bg_top_p, spec.fg_weight, spec.bg_weight,
                          spec.ref_ca_loss_weight, spec.ref_word_token_only, use_ref, spec.use_ratio_based_loss)
    slot_tok, slot_of = G.assign_slots(layouts, params)
    if reuse is not None:
        old, slot_dev = reuse
        if set(old) == set(spec.keys) and slot_dev.shape == slot_tok.shape and all(
                old[k].update(layouts, slot_of, len(spec.keys), params) for k in spec.keys):
            slot_dev.copy_(torch.from_numpy(slot_tok))
            for kl in old.values():
                kl.c.gscale = net.gscale
                kl.set_step(index)
            return old, slot_dev, True
    slot_dev = torch.from_numpy(slot_tok).to(dev)
    out = {k: G.KeyLoss(layouts, slot_dev, slot_of, k, _tokens_of(net, k, H, W), _heads_of(net, k), len(spec.keys),
                        params, dev, gscale=net.gscale) for k in spec.keys}
    for kl in out.values():
        kl.set_step(index)
    return out, slot_dev, False


def guidance_step_scale(sched, index, t):
    """models/pipelines.py:60-69: schedulers that carry `sigmas` (Euler / LMS family) scale the guidance step by
    sigmas[index]**2, DDIM-style schedulers by sqrt(1 - alpha_bar_t) (classifier-guidance scaling)"""
    sig = getattr(sched, "sigmas", None)
    if sig is not None:
        return float(sig[index]) ** 2
    return float((1.0 - sched.alphas_cumprod[int(t)]) ** 0.5)


class _LoopState:
    """device-resident per-image loop state of latent_backward_guidance (loss carried across steps, iteration counters,
    active mask, trace rows of the current step) + a pinned host mirror for the one small read-back per iteration"""

    def __init__(self, B, has_boxes, dev, cap=64):
        self.B, self.cap = B, cap
        self.loss = torch.full((B,), 10000.0, dtype=torch.float64, device=dev)
        self.it = torch.zeros(B, dtype=torch.int32, device=dev)
        self.active = torch.zeros(B, dtype=torch.int32, device=dev)
        self.has_boxes = torch.from_numpy(has_boxes.astype(np.int32)).to(dev)
        self.trace_loss = torch.zeros(cap, B, dtype=torch.float64, device=dev)
        self.trace_active = torch.zeros(cap, B, dtype=torch.int32, device=dev)
        self.any = torch.zeros(1, dtype=torch.int32, device=dev)
        self.any_host = torch.zeros(1, dtype=torch.int32).pin_memory()


def latent_backward_guidance(net, sched: DDIMSchedule, z, t, index, kv_cond, spec: GuidanceSpec, state: GuidanceState,
                             objs=None, fuser_on=False, use_graphs=False):
    """models/pipelines.py:16-82, batched with per-image predicates evaluated ON THE DEVICE
    (b200lmd_guidance_loop_begin / _advance): no active mask is uploaded and the loss partials are not read back; per
    iteration the host reads one int (does any image continue?), per step one trace block.
    z: device fp32 [B,4,H,W], updated in place."""
    B, Cz, H, W = z.shape
    it = np.zeros(B, dtype=np.int64)
    if index >= spec.max_index_step or all(len(l.bboxes) == 0 for l in spec.layouts):
        state.iters.append(it.tolist())
        return
    mi = spec.max_iter
    if isinstance(mi, list):
        mi = mi[index] if len(mi) > index else mi[-1]
    mi = int(mi)
    has_boxes = np.array([len(l.bboxes) > 0 for l in spec.layouts])
    # the host mirrors the carried loss (refreshed from the trace block at the end of every guided step), so whether the
    # loop is entered at all needs no device round trip
    if not (has_boxes & (state.loss / spec.loss_scale > spec.loss_threshold) & (0 < mi)).any():
        state.iters.append(it.tolist())
        return
    ls = state.__dict__.get("loop")
    if ls is None:
        ls = state.loop = _LoopState(B, has_boxes, z.device)
    if mi > ls.cap:
        raise ValueError(f"max_iter {mi} exceeds the trace capacity {ls.cap}")
    losses = state.losses
    if losses is not None:
        for kl in losses.values():
            kl.set_step(index)
    if state.t_dev is None:
        state.t_dev = torch.empty(B, device=z.device, dtype=torch.float32)
    t_dev = state.t_dev
    t_dev.fill_(float(t))
    step_scale = guidance_step_scale(sched, index, t)
    S = cur_stream()
    _d = ctypes.c_double
    check(lib().b200lmd_guidance_loop_begin(ptr(ls.loss), ptr(ls.it), ptr(ls.active), ptr(ls.has_boxes), ptr(ls.any),
                                            _i(B), _d(spec.loss_scale), _d(spec.loss_threshold), _i(mi), S))
    n_done, go = 0, True
    while go and n_done < mi:
        if losses is None:
            ctx = state.ctx
            reuse = (ctx.losses, ctx.slot_dev) if (ctx is not None and ctx.losses is not None) else None
            losses, slot_dev, reused = build_losses(net, spec, index, H, W, z.device, reuse=reuse)
            state.losses = losses
            if ctx is not None:
                if not reused:
                    ctx.guid_graphs.clear()          # graphs captured over the old tables are dead
                ctx.losses, ctx.slot_dev = losses, slot_dev
                state.graphs = ctx.guid_graphs
        if use_graphs:
            if fuser_on not in state.graphs:
                state.graphs[fuser_on] = CudaGraph(lambda: net.guidance_gradient_launch(
                    z, t_dev, kv_cond, losses, objs=objs, fuser_on=fuser_on),
                    key=("guid", tuple(z.shape), fuser_on, objs is not None), owner=net)
            grad, parts = state.graphs[fuser_on]()
        else:
            grad, parts = net.guidance_gradient_launch(z, t_dev, kv_cond, losses, objs=objs, fuser_on=fuser_on)
        check(lib().b200lmd_latent_update(ptr(z), ptr(grad), _i(grad.shape[2]), _i(B), _i(Cz), _i(H * W),
                                          _f(step_scale), _f(1.0 / net.gscale), ptr(ls.active), S))
        check(lib().b200lmd_guidance_loop_advance(
            ptr(ls.loss), ptr(ls.it), ptr(ls.active), ptr(ls.has_boxes), ptr(ls.trace_loss), ptr(ls.trace_active),
            ptr(ls.any), ptr(parts), _i(parts.shape[0]), _i(B), _i(parts.shape[1] // B), _d(spec.loss_scale),
            _d(spec.loss_threshold), _i(mi), _i(n_done), S))
        n_done += 1
        if n_done < mi:                         # does any image continue? (one int; the reference reads loss.item())
            ls.any_host.copy_(ls.any, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            go = bool(ls.any_host[0])
    # one read-back per guided step: the trace rows of this step
    tl = ls.trace_loss[:n_done].cpu().numpy()
    ta = ls.trace_active[:n_done].cpu().numpy().astype(bool)
    for j in range(n_done):
        it[ta[j]] += 1
        state.loss = np.where(ta[j], tl[j], state.loss)
        state.trace.append((index, j + 1, tl[j].tolist(), ta[j].tolist()))
    state.iters.append(it.tolist())


class DenoiseCtx:
    """static device state of one denoise() shape: latents, timestep vectors, text K/V slabs, GLIGEN object tokens, loss
    tables and the CUDA graphs captured over them.  Cached on the net (`net._denoise_ctx[key]`), so a later denoise()
    call of the same shape copies its inputs into these buffers and REPLAYS the graphs instead of re-capturing them
    (a capture of one CFG forward at batch 64 costs more than the 50 replays it serves)."""

    def __init__(self):
        self.z = self.t2 = self.tok_dev = self.kv = self.objs_main = None
        self.fwd_graphs, self.guid_graphs, self.bd_graphs = {}, {}, {}
        self.losses = self.slot_dev = self.bd = self.t_dev = None


def _denoise_ctx(net, key):
    cache = net.__dict__.setdefault("_denoise_ctx", {})
    if key not in cache:
        if len(cache) >= 6:                      # bound the number of live graph sets (shapes seen by one process)
            cache.pop(next(iter(cache)))
        cache[key] = DenoiseCtx()
    return cache[key]


def denoise(net, z0, uncond, cond, steps, guidance_scale=7.5, guidance: Optional[GuidanceSpec] = None,
            frozen_mask=None, frozen_latents=None, frozen_steps=0, gligen=None, gligen_beta=0.3, save_keys=None,
            save_tok: Optional[Sequence[int]] = None, save_latents=False, prediction_type="epsilon", use_graphs=True,
            fast_after_steps=None, fast_rate=2, dynamic_num_inference_steps=False, boxdiff=None):
    """B images in lock-step.  z0 [B,4,H,W] fp32 (any device); uncond [1 or B,T,ctx]; cond [B,T,ctx];
    frozen_mask [B,H,W] or [H,W] (1 = take the frozen latent), frozen_latents [steps+1,B,4,H,W];
    gligen: dict(boxes [B,30,4], masks [B,30], positive_embeddings [B,30,768]) of the conditional half;
    save_keys/save_tok: per step keep the cond-half map column tok[b] of those keys (return_cond_ca_only +
    return_token_ca_only).  fast_after_steps / fast_rate / dynamic_num_inference_steps: the reference's fast schedule
    (models/pipelines.py:358-362,439-440,449): thinned timestep list after `fast_after_steps`, DDIM step size
    re-derived per step, latents kept only for index < fast_after_steps.
    boxdiff: a boxdiff.BoxDiffSpec - one BoxDiff guidance step per denoising step for index < max_index_step
    (utils/boxdiff.py:190-259, models/pipelines.py:186-188) instead of the attention-energy guidance.
    Returns dict(latents, latents_all, saved, state)."""
    dev = net.dev
    timing = os.environ.get("B200_TIMING")
    if timing:
        torch.cuda.synchronize()
        t_start, cap0 = time.perf_counter(), CudaGraph.capture_seconds
    B, Cz, H, W = z0.shape
    ctx = None
    if use_graphs:
        key = (B, Cz, H, W, tuple(uncond.shape[1:]), tuple(cond.shape[1:]), gligen is not None,
               tuple(save_keys) if save_keys is not None else None, save_tok is not None,
               tuple(guidance.keys) if guidance is not None else None, prediction_type,
               ("boxdiff",) + tuple(boxdiff.keys) if boxdiff is not None else None)
        ctx = _denoise_ctx(net, key)
    if ctx is not None and ctx.z is not None:
        z = ctx.z
        z.copy_(z0.to(dev, torch.float32))
    else:
        z = z0.to(dev, torch.float32).contiguous().clone()
        if ctx is not None:
            ctx.z = z
    sched = DDIMSchedule(prediction_type)
    sched.set_timesteps(steps)
    if fast_after_steps is not None:
        sched.apply_fast_schedule(fast_after_steps, fast_rate)
    if uncond.shape[0] == 1:
        uncond = uncond.expand(B, -1, -1)
    text = torch.cat([uncond, cond], dim=0)
    kv = net.set_text(text, kv=ctx.kv if ctx is not None else None)
    if ctx is not None:
        ctx.kv = kv
    heads_of = lambda p: kv.slabs[p][0].shape[0] // (2 * B)
    kv_cond = lambda p: tuple(s[B * heads_of(p):] for s in kv.slabs[p])
    objs_main = objs_guid = None
    n_ground = int(gligen_beta * len(sched.timesteps))       # models/pipelines.py:408
    if gligen is not None:
        rep2 = lambda x: torch.cat([x, x], dim=0)
        masks2 = rep2(gligen["masks"]).clone()
        masks2[:B] = 0                                   # pipelines.py:317 (unconditional half sees null tokens)
        objs_main = net.position_net(rep2(gligen["boxes"]), masks2, rep2(gligen["positive_embeddings"]))
        if ctx is not None:
            if ctx.objs_main is not None and ctx.objs_main.shape == objs_main.shape:
                ctx.objs_main.copy_(objs_main)
                objs_main = ctx.objs_main
            else:
                ctx.objs_main = objs_main
                ctx.fwd_graphs.clear()
                ctx.guid_graphs.clear()
        n_obj = objs_main.shape[0] // (2 * B)
        objs_guid = objs_main[:B * n_obj]                # pipelines.py:382-384: the zeroed-mask half
    fm = fl = None
    if frozen_mask is not None:
        fm = frozen_mask.to(dev, torch.float32).clamp(0.0, 1.0)
        fm = fm.reshape(1, H * W).expand(B, -1).contiguous() if fm.ndim == 2 else fm.reshape(B, H * W).contiguous()
        fl = frozen_latents.to(dev, torch.float32).contiguous()
    tok_dev = None
    if save_tok is not None:
        tok_dev = torch.tensor([-1] * B + list(save_tok), dtype=torch.int32, device=dev)
        if ctx is not None:
            if ctx.tok_dev is None:
                ctx.tok_dev = tok_dev
            else:
                ctx.tok_dev.copy_(tok_dev)
                tok_dev = ctx.tok_dev
    state = GuidanceState(B)
    state.ctx = ctx
    fwd_graphs = ctx.fwd_graphs if ctx is not None else {}
    if ctx is not None:
        state.graphs = ctx.guid_graphs
        if ctx.t2 is None:
            ctx.t2 = torch.empty(2 * B, device=dev, dtype=torch.float32)
            ctx.t_dev = torch.empty(B, device=dev, dtype=torch.float32)
        t2, state.t_dev = ctx.t2, ctx.t_dev
    else:
        t2 = torch.empty(2 * B, device=dev, dtype=torch.float32)
    latents_all = [z.clone()] if save_latents else None
    saved_all = []
    if timing:
        torch.cuda.synchronize()
        t_loop = time.perf_counter()
    bd = bd_active = None
    bd_graphs = ctx.bd_graphs if ctx is not None else {}
    for index, t in enumerate(sched.timesteps):
        fuser_on = gligen is not None and index < n_ground
        if boxdiff is not None and index < boxdiff.max_index_step and any(len(l.bboxes) for l in boxdiff.layouts):
            from . import boxdiff as BD
            if bd is None:
                if ctx is not None and ctx.bd is not None and ctx.bd.update(boxdiff):
                    bd = ctx.bd                          # tables refilled in place: the captured graphs stay valid
                else:
                    bd = BD.BoxDiffLoss(net, boxdiff, H, W, kv.T)
                    bd_graphs.clear()
                    if ctx is not None:
                        ctx.bd = bd
                bd_active = torch.tensor([int(len(l.bboxes) > 0) for l in boxdiff.layouts], dtype=torch.int32, device=dev)
                if state.t_dev is None:
                    state.t_dev = torch.empty(B, device=dev, dtype=torch.float32)
                state.boxdiff_losses = []
            state.t_dev.fill_(float(t))
            if use_graphs:
                if fuser_on not in bd_graphs:
                    bd_graphs[fuser_on] = CudaGraph(lambda: bd.gradient_launch(z, state.t_dev, kv_cond, objs=objs_guid,
                                                                               fuser_on=fuser_on),
                                                    key=("boxdiff", tuple(z.shape), fuser_on, objs_guid is not None),
                                                    owner=net)
                grad, bl = bd_graphs[fuser_on]()
            else:
                grad, bl = bd.gradient_launch(z, state.t_dev, kv_cond, objs=objs_guid, fuser_on=fuser_on)
            check(lib().b200lmd_latent_update(ptr(z), ptr(grad), _i(grad.shape[2]), _i(B), _i(Cz), _i(H * W),
                                              _f(BD.step_scale(boxdiff, index, len(sched.timesteps))),
                                              _f(1.0 / net.gscale), ptr(bd_active), cur_stream()))
            state.boxdiff_losses.append(bl.clone())
        if guidance is not None:
            latent_backward_guidance(net, sched, z, t, index, kv_cond, guidance, state, objs=objs_guid,
                                     fuser_on=fuser_on, use_graphs=use_graphs)
        t2.fill_(float(t))
        if use_graphs:
            if fuser_on not in fwd_graphs:
                fwd_graphs[fuser_on] = CudaGraph(lambda: net.forward(
                    z, t2, kv, rep=2, objs=objs_main, fuser_on=fuser_on, save_keys=save_keys, save_tok=tok_dev),
                    key=("fwd", tuple(z.shape), fuser_on, objs_main is not None, save_keys is not None), owner=net)
            eps, saved = fwd_graphs[fuser_on]()
        else:
            eps, saved = net.forward(z, t2, kv, rep=2, objs=objs_main, fuser_on=fuser_on, save_keys=save_keys,
                                     save_tok=tok_dev)
        if save_keys is not None:       # graph outputs are static buffers: keep a copy of this step's maps
            saved_all.append({k: v["tok"][B:].clone() for k, v in saved.items()})
        if dynamic_num_inference_steps:
            sched.adjust(index, t)
        sa_t, sb_t, sa_p, sb_p = sched.coefs(t)
        use_frozen = fm is not None and index < frozen_steps
        check(lib().b200lmd_cfg_ddim_blend(ptr(z), ptr(eps), _i(eps.shape[3]), _i(B), _i(Cz), _i(H * W),
                                           _f(guidance_scale), _f(sa_t), _f(sb_t), _f(sa_p), _f(sb_p),
                                           _i(int(prediction_type == "v_prediction")),
                                           ptr(fl[index + 1]) if use_frozen else None, ptr(fm) if use_frozen else None,
                                           cur_stream()))
        if save_latents and (fast_after_steps is None or index < fast_after_steps):
            latents_all.append(z.clone())
    if timing:
        torch.cuda.synchronize()
        t_end = time.perf_counter()
        print(f"[timing] denoise B={B}: setup {1e3 * (t_loop - t_start):.0f} ms, loop {1e3 * (t_end - t_loop):.0f} ms "
              f"(of which graph warm-up+capture {1e3 * (CudaGraph.capture_seconds - cap0):.0f} ms), guidance "
              f"iterations {int(np.sum(state.iters)) if state.iters else 0}", file=sys.stderr)
    # z may be a static buffer of the cached context: hand out a copy
    return dict(latents=z.clone() if ctx is not None else z,
                latents_all=torch.stack(latents_all, 0) if save_latents else None, saved=saved_all, state=state)
