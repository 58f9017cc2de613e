"""Pins the oracle restatement (oracle/*.py) against outputs of the UNMODIFIED reference.

CPU only.  The reference has no tests or golden vectors of its own (SURVEY.md section 4), so outputs of the reference
itself, run on seeded synthetic weights and inputs, are the pin.  `python -m oracle.make_goldens vs_reference` runs
the reference on exactly the inputs built here and stores what each test compares against in
tests/golden/oracle_vs_reference.npz (with tests/golden/pipeline_reference.npz for the semantic-guidance latents), so
the comparison runs wherever the repository does.  Exact reference outputs (integers, masks, shifted tensors) are
stored as sha256 digests of dtype, shape and bytes; floating-point tensors too large to store whole are stored at a
fixed sample of positions (all nonzero entries up to a count, plus seeded positions anywhere) and compared there with
the same tolerance.
"""
import functools
import hashlib
import os
import random

import numpy as np
import pytest
import torch

from oracle import guidance_ref, pipeline_ref, unet_ref

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
KEYS = [("mid", 0, 0, 0), ("up", 1, 0, 0), ("up", 1, 1, 0), ("up", 1, 2, 0)]


def digest(x):
    """sha256 (first 128 bits) of an array's dtype, shape and bytes (tensor or array-like)"""
    a = x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()[:32]


def sample_index(ref, k):
    """flat positions at which a large reference tensor is stored: up to k of its nonzero entries and k // 4 positions
    anywhere, both drawn with a fixed seed"""
    flat = np.asarray(ref).reshape(-1)
    if flat.size <= k:
        return np.arange(flat.size, dtype=np.int64)
    rng = np.random.RandomState(0)
    nz = np.flatnonzero(flat)
    pick = nz if nz.size <= k else rng.choice(nz, k, replace=False)
    return np.unique(np.concatenate([pick, rng.choice(flat.size, k // 4, replace=False)]))


def _shapes(shapes):
    out = np.full((len(shapes), 6), -1, dtype=np.int64)
    for i, s in enumerate(shapes):
        out[i, :len(s)] = s
    return out


def _shape(row):
    return tuple(int(v) for v in row if v >= 0)


def pack(values, samples, texts):
    """stored reference outputs as a few flat arrays (one .npz member per output would outweigh the outputs):
    values {name: array} (float64), samples {name: (shape, flat positions, float32 values)}, texts {name: str}"""
    vn, sn, tn = list(values), list(samples), list(texts)
    va = [np.asarray(values[n], dtype=np.float64) for n in vn]
    return dict(
        value_names=np.array(vn), value_shapes=_shapes([a.shape for a in va]),
        value_offsets=np.cumsum([0] + [a.size for a in va]), value_data=np.concatenate([a.reshape(-1) for a in va]),
        sample_names=np.array(sn), sample_shapes=_shapes([samples[n][0] for n in sn]),
        sample_offsets=np.cumsum([0] + [len(samples[n][1]) for n in sn]),
        sample_idx=np.concatenate([samples[n][1] for n in sn]).astype(np.int32),
        sample_val=np.concatenate([samples[n][2] for n in sn]).astype(np.float32),
        text_names=np.array(tn), text_values=np.array([texts[n].encode() for n in tn]))


def unpack(f):
    g = {}
    o = f["value_offsets"]
    for i, n in enumerate(f["value_names"]):
        g[str(n)] = f["value_data"][o[i]:o[i + 1]].reshape(_shape(f["value_shapes"][i]))
    o = f["sample_offsets"]
    for i, n in enumerate(f["sample_names"]):
        g[str(n)] = (_shape(f["sample_shapes"][i]), f["sample_idx"][o[i]:o[i + 1]], f["sample_val"][o[i]:o[i + 1]])
    for n, t in zip(f["text_names"], f["text_values"]):
        g[str(n)] = t.decode()
    return g


@functools.lru_cache(maxsize=None)
def _golden(name="oracle_vs_reference.npz"):
    with np.load(os.path.join(GOLDEN, name)) as f:
        d = {k: f[k] for k in f.files}
    return unpack(d) if "value_names" in d else d


def gold(key):
    return _golden()[key]


def key_name(k):
    return "_".join(map(str, k))


def sampled(name, mine):
    """(mine, reference) at the stored positions of reference tensor `name`; the shapes must agree"""
    mine = mine.detach().cpu().numpy() if torch.is_tensor(mine) else np.asarray(mine)
    shape, idx, val = gold(name)
    assert tuple(mine.shape) == shape, (mine.shape, shape)
    return mine.reshape(-1)[idx], val


def test_scale_proportion_matches_reference():
    rng = random.Random(0)
    out = []
    for _ in range(3000):
        x0, y0 = rng.uniform(-0.1, 0.9), rng.uniform(-0.1, 0.9)
        box = (x0, y0, x0 + rng.uniform(0, 0.8), y0 + rng.uniform(0, 0.8))
        for side in (8, 16, 24, 64):
            out.append(guidance_ref.scale_proportion(box, side, side))
    # .5 cases (banker's rounding)
    for box in [(0.0625, 0.1875, 0.5625, 0.8125), (0.03125, 0.09375, 0.15625, 0.21875)]:
        for side in (8, 16):
            out.append(guidance_ref.scale_proportion(box, side, side))
    assert digest(np.array(out, dtype=np.int64)) == gold("scale_proportion")


def _random_case(seed, heads=8, with_ref=True):
    g = torch.Generator().manual_seed(seed)
    rng = random.Random(seed)
    saved = {}
    for k in KEYS:
        n = 64 if k[0] == "mid" else 256
        saved[k] = torch.softmax(3 * torch.randn(1, heads, n, 77, generator=g), dim=-1)
    n_obj = rng.randint(1, 3)
    bboxes, positions, words, refs = [], [], [], []
    tok = 1
    for o in range(n_obj):
        nb = rng.randint(1, 2)
        boxes = []
        for _ in range(nb):
            w_, h_ = rng.uniform(0.15, 0.6), rng.uniform(0.15, 0.6)
            x, y = rng.uniform(0, 1 - w_), rng.uniform(0, 1 - h_)
            boxes.append((x, y, x + w_, y + h_))
        bboxes.append(boxes)
        nt = rng.randint(1, 3)
        positions.append(list(range(tok, tok + nt)))
        words.append(tok + nt - 1)
        tok += nt + 1
        refs.append([[{k: torch.softmax(3 * torch.randn(1, heads, saved[k].shape[2], 1, generator=g), dim=2)
                       for k in KEYS}] for _ in range(nb)])   # [box][step=0][key]
    return saved, bboxes, positions, words, (refs if with_ref else None)


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
@pytest.mark.parametrize("with_ref", [False, True])
def test_ca_loss_and_grad_match_reference(seed, with_ref):
    """utils/guidance.py compute_ca_lossv3 (+ autograd w.r.t. every saved map) vs ca_loss / ca_loss_and_grad"""
    saved, bboxes, positions, words, refs = _random_case(seed, with_ref=with_ref)
    tag = f"ca_s{seed}_r{int(with_ref)}"
    L_ref = float(gold(tag + "_loss"))
    one = {k: v[0] for k, v in saved.items()}
    ref_maps = None
    if refs is not None:
        ref_maps = [[{k: box[0][k][0, :, :, 0] for k in KEYS} for box in obj] for obj in refs]
    L = guidance_ref.ca_loss(one, bboxes, positions, KEYS, 0.2, 0.2, 1.0, 4.0, ref_maps, words, 2.0, True)
    assert abs(float(L) - L_ref) < 2e-6 * max(1.0, abs(L_ref))
    L2, grads = guidance_ref.ca_loss_and_grad({k: v.numpy() for k, v in one.items()}, bboxes, positions, KEYS, 0.2,
                                              0.2, 1.0, 4.0,
                                              None if ref_maps is None else
                                              [[{k: m[k].numpy() for k in KEYS} for m in obj] for obj in ref_maps],
                                              words, 2.0, True)
    assert abs(L2 - L_ref) < 5e-6 * max(1.0, abs(L_ref))
    for k in KEYS:
        mine, ref = sampled(f"{tag}_g_{key_name(k)}", grads[k][None])
        np.testing.assert_allclose(mine, ref, rtol=2e-4, atol=2e-7)


def _unet_case(gligen):
    cfg = unet_ref.UNetConfig.tiny(gligen=gligen)
    w = unet_ref.make_weights(cfg, seed=0)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 4, 16, 16, generator=g)
    ctx = torch.randn(2, 77, 768, generator=g)
    gl = None
    if gligen:
        gl = dict(boxes=torch.rand(2, 30, 4, generator=g), masks=(torch.rand(2, 30, generator=g) > 0.8).float(),
                  positive_embeddings=torch.randn(2, 30, 768, generator=g))
    return cfg, w, x, ctx, gl


@pytest.mark.parametrize("gligen", [False, True])
def test_unet_forward_matches_reference(gligen):
    cfg, w, x, ctx, gl = _unet_case(gligen)
    with torch.no_grad():
        saved = {}
        mine = unet_ref.unet_forward(w, cfg, x, 481, ctx, gligen=gl, saved=saved)
    tag = f"unet_g{int(gligen)}"
    assert np.abs(np.subtract(*sampled(tag + "_eps", mine))).max() < 2e-5
    assert len(saved) == 16
    ref_keys = gold(tag + "_keys").split(",")
    assert len(ref_keys) == 16
    for k, v in saved.items():
        assert key_name(k) in ref_keys
    for ks in ref_keys:
        k = tuple(int(p) if p.isdigit() else p for p in ks.split("_"))
        a, b = sampled(f"{tag}_saved_{ks}", saved[k])
        assert np.abs(a - b).max() < 1e-4


def _pipeline_inputs(gligen):
    cfg = unet_ref.UNetConfig.tiny(gligen=gligen)
    w = unet_ref.make_weights(cfg, seed=0)
    g = torch.Generator().manual_seed(5)
    z0 = torch.randn(1, 4, 32, 32, generator=g)
    uncond = torch.randn(1, 77, 768, generator=g)
    cond = torch.randn(1, 77, 768, generator=g)
    table = torch.randn(4, 768, generator=g)
    return cfg, w, z0, uncond, cond, table


def _check_saved(tag, saved):
    """per-step maps saved by a denoising loop vs the reference's (return_saved_cross_attn)"""
    assert len(saved) == int(gold(tag + "_nsteps"))
    for i, s in enumerate(saved):
        ref_keys = sorted(gold(f"{tag}_{i}_keys").split(","))
        assert sorted(key_name(k) for k in s) == ref_keys
        for k in s:
            a, b = sampled(f"{tag}_{i}_{key_name(k)}", s[k])
            assert np.abs(a - b).max() < 1e-3


def test_semantic_guidance_loop_matches_reference():
    """generate_semantic_guidance (LMD per-box phase, backward_guidance): guidance + CFG + DDIM, attention saving"""
    cfg, w, z0, uncond, cond, _ = _pipeline_inputs(False)
    bboxes = [[(0.1, 0.2, 0.6, 0.7)], [(0.5, 0.4, 0.95, 0.9)]]
    positions = [[2, 3], [6]]
    steps = 4
    all_ref = torch.from_numpy(_golden("pipeline_reference.npz")["semantic_latents_all"])
    lat_ref = all_ref[-1]
    g = pipeline_ref.GuidanceCfg(bboxes, positions, KEYS, 30, 0.2, [2, 1, 1], 3, 0.2, 0.2, 1.0, 4.0)
    res = pipeline_ref.denoise(w, cfg, z0, uncond, cond, steps, g=g, save_keys=[("down", 2, 1, 0)] + KEYS,
                               save_token=3)
    assert res["iters"] == [2, 1, 1, 0]
    assert (res["latents"] - lat_ref).abs().max() < 5e-3
    assert (res["latents_all"] - all_ref).abs().max() < 5e-3
    _check_saved("semantic_saved", res["saved"])


def test_partial_frozen_loop_matches_reference():
    """generate_partial_frozen (LMD overall phase, models/pipelines.py:541-599): guidance + CFG + DDIM with the frozen
    blend z = z_ref[i+1] m + z (1 - m) for index < frozen_steps"""
    cfg, w, z0, uncond, cond, _ = _pipeline_inputs(False)
    steps = 4
    g0 = torch.Generator().manual_seed(21)
    latents_all = torch.randn(steps + 1, 1, 4, 32, 32, generator=g0)
    latents_all[0] = z0
    frozen_mask = (torch.rand(32, 32, generator=g0) > 0.4).float()
    bboxes = [[(0.1, 0.2, 0.6, 0.7)], [(0.5, 0.4, 0.95, 0.9)]]
    positions = [[2, 3], [6]]
    g = pipeline_ref.GuidanceCfg(bboxes, positions, KEYS, 30, 0.2, [2, 1], 3, 0.2, 0.2, 1.0, 4.0)
    res = pipeline_ref.denoise(w, cfg, z0, uncond, cond, steps, g=g, frozen_mask=frozen_mask,
                               frozen_latents=latents_all, frozen_steps=2)
    assert res["iters"] == [2, 1, 1, 0]
    assert np.abs(np.subtract(*sampled("partial_frozen_latents", res["latents"]))).max() < 5e-3


def _gligen_ref_case():
    steps = 4
    cfg, w, z0, uncond, cond, table = _pipeline_inputs(True)
    g0 = torch.Generator().manual_seed(9)
    frozen_latents = torch.randn(steps + 1, 1, 4, 32, 32, generator=g0)
    frozen_latents[0] = z0
    frozen_mask = (torch.rand(32, 32, generator=g0) > 0.5).float()
    heads = 8
    refs = [[[{k: torch.softmax(3 * torch.randn(1, heads, 16 if k[0] == "mid" else 64, 1, generator=g0), dim=2)
               for k in KEYS} for _ in range(steps)]] for _ in range(2)]   # [obj][box][step][key]
    return steps, frozen_latents, frozen_mask, refs


def _gligen_cond(table, bboxes_flat):
    n = len(bboxes_flat)
    boxes = torch.zeros(1, 30, 4)
    boxes[0, :n] = torch.tensor(bboxes_flat)
    emb = torch.zeros(1, 30, 768)
    emb[0, :n] = table[:n]
    masks = torch.zeros(1, 30)
    masks[0, :n] = 1
    return dict(boxes=boxes, masks=masks, positive_embeddings=emb)


def test_gligen_loop_with_ref_attention_matches_reference():
    """generate_gligen (LMD+ overall phase): fuser schedule, null-mask guidance pass, ref-attention loss, frozen blend"""
    cfg, w, z0, uncond, cond, table = _pipeline_inputs(True)
    steps, frozen_latents, frozen_mask, refs = _gligen_ref_case()
    bboxes_flat = [(0.1, 0.2, 0.6, 0.7), (0.5, 0.4, 0.95, 0.9)]
    sg_bboxes = [[bboxes_flat[0]], [bboxes_flat[1]]]
    positions = [[2, 3], [6]]
    words = [3, 6]
    ref_maps = [[[{k: st[k][0, :, :, 0] for k in KEYS} for st in box] for box in obj] for obj in refs]
    g = pipeline_ref.GuidanceCfg(sg_bboxes, positions, KEYS, 5, 0.01, [2, 1], 3, 0.2, 0.2, 1.0, 4.0, ref_maps, words,
                                 2.0, True)
    res = pipeline_ref.denoise(w, cfg, z0, uncond, cond, steps, g=g, frozen_mask=frozen_mask,
                               frozen_latents=frozen_latents, frozen_steps=2,
                               gligen=_gligen_cond(table, bboxes_flat), gligen_beta=0.5)
    assert res["iters"] == [2, 1, 1, 0]
    assert np.abs(np.subtract(*sampled("gligen_ref_latents", res["latents"]))).max() < 5e-3


def _boxdiff_case(seed):
    g = torch.Generator().manual_seed(100 + seed)
    heads, n, T = 8, 256, 77
    keys = [("down", 2, 0, 0), ("down", 2, 1, 0), ("up", 1, 0, 0), ("up", 1, 1, 0), ("up", 1, 2, 0)]
    bboxes = [[(0.1, 0.2, 0.6, 0.7)], [(0.5, 0.4, 0.95, 0.9), (0.0, 0.0, 0.3, 0.3)]]
    positions = [[2, 3], [6]]
    maps = {k: torch.softmax(2 * torch.randn(heads, n, T, generator=g), dim=-1) for k in keys}
    return g, keys, bboxes, positions, maps


@pytest.mark.parametrize("seed,smooth", [(0, True), (1, True), (2, False)])
def test_boxdiff_loss_and_grad_match_reference(seed, smooth):
    """utils/boxdiff.py compute_ca_loss_boxdiff (no reference-attention term) vs oracle/boxdiff_ref.py: loss and the
    gradient with respect to every saved map (groundwork for SURVEY section 8 row a14)"""
    from oracle import boxdiff_ref
    g, keys, bboxes, positions, maps = _boxdiff_case(seed)
    ours_in = {k: v.clone().requires_grad_(True) for k, v in maps.items()}
    ours = boxdiff_ref.boxdiff_loss(ours_in, bboxes, positions, keys, smooth_attentions=smooth)
    g_ours = torch.autograd.grad(ours, [ours_in[k] for k in keys])
    tag = f"boxdiff_s{seed}"
    ref = float(gold(tag + "_loss"))
    assert abs(float(ours) - ref) < 1e-5 * max(1.0, abs(ref)), (float(ours), ref)
    for k, a in zip(keys, g_ours):
        name = f"{tag}_g_{key_name(k)}"
        mine, b = sampled(name, a[None])
        assert np.abs(mine - b).max() < 1e-6 + 1e-4 * float(gold(name + "_absmax"))
    # update rule (boxdiff.py:228-232)
    z, gr = torch.randn(1, 4, 8, 8, generator=g), torch.randn(1, 4, 8, 8, generator=g)
    for index in (0, 7, 24):
        scale = (1.0 + (0.5 - 1.0) * index / 49) ** 0.5
        assert torch.allclose(boxdiff_ref.boxdiff_update(z, gr, index, 50), z - 20 * scale / 10 * gr)


def test_gligen_loop_fast_schedule_matches_reference():
    """generate_gligen with the thinned timestep list and per-step DDIM step size (fast_after_steps, fast_rate,
    dynamic_num_inference_steps; models/pipelines.py:358-362,439-440)"""
    cfg, w, z0, uncond, cond, table = _pipeline_inputs(True)
    steps = 8
    res = pipeline_ref.denoise(w, cfg, z0, uncond, cond, steps, gligen=_gligen_cond(table, [(0.1, 0.2, 0.6, 0.7)]),
                               gligen_beta=0.5, fast_after_steps=3, fast_rate=2, dynamic_num_inference_steps=True)
    assert res["latents_all"].shape[0] == 4            # initial + the three steps before the fast part
    assert np.abs(np.subtract(*sampled("gligen_fast_latents", res["latents"]))).max() < 5e-3


def fast_schedule_cases():
    for steps in (10, 20, 50):
        for fast_after in (0, 3, steps // 2, steps - 2, steps - 1, steps + 5):
            for rate in (2, 3):
                yield steps, fast_after, rate


def test_fast_schedule_matches_reference():
    """utils/schedule.py (get_fast_schedule, dynamically_adjust_inference_steps) vs pipelines.DDIMSchedule"""
    import lgd_b200  # noqa: F401
    from lgd_b200.pipelines import DDIMSchedule
    for steps, fast_after, rate in fast_schedule_cases():
        tag = f"sched_{steps}_{fast_after}_{rate}"
        ours = DDIMSchedule()
        ours.set_timesteps(steps)
        ours.apply_fast_schedule(fast_after, rate)
        assert ours.timesteps.tolist() == gold(tag + "_timesteps").tolist()
        nis = []
        for index, t in enumerate(ours.timesteps.tolist()):
            ours.adjust(index, t)
            nis.append(ours.num_inference_steps)
        assert nis == gold(tag + "_num_inference_steps").tolist()


def test_callshape_loop_matches_reference_pipeline():
    """oracle/callshape_ref.generate (the loop used to test the B200UNetAdapter on the GPU box) over `OracleUNet` (the
    CPU oracle behind the reference's UNet call shape) must reproduce the unmodified pipelines.generate_gligen: same
    iteration counts, same latents, same saved maps"""
    from oracle import callshape_ref
    cfg, w, z0, uncond, cond, table = _pipeline_inputs(True)
    steps = 4
    bboxes_flat = [(0.1, 0.2, 0.6, 0.7), (0.5, 0.4, 0.95, 0.9)]
    sg_bboxes = [[bboxes_flat[0]], [bboxes_flat[1]]]
    positions = [[2, 3], [6]]
    g = pipeline_ref.GuidanceCfg(sg_bboxes, positions, KEYS, 5, 0.01, [2, 1], 3, 0.2, 0.2, 1.0, 4.0)
    res = callshape_ref.generate(callshape_ref.OracleUNet(w, cfg), z0, uncond, cond, steps, g=g,
                                 gligen=_gligen_cond(table, bboxes_flat), gligen_beta=0.5,
                                 saved_cross_attn_keys=[("down", 2, 1, 0)] + KEYS, return_token_ca_only=3)
    assert res["iters"] == [2, 1, 1, 0]
    assert np.abs(np.subtract(*sampled("callshape_latents", res["latents"]))).max() < 5e-3
    _check_saved("callshape_saved", res["saved"])


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_ratio_based_loss_matches_reference(seed):
    """compute_ca_lossv3 with its DEFAULT use_ratio_based_loss=True (what generation/backward_guidance.py runs,
    utils/guidance.py:122-128): loss and gradient w.r.t. every saved map vs oracle ca_loss(use_ratio_based_loss=True)"""
    saved, bboxes, positions, words, _ = _random_case(seed, with_ref=False)
    ours_in = {k: v[0].clone().requires_grad_(True) for k, v in saved.items()}
    ours = guidance_ref.ca_loss(ours_in, bboxes, positions, KEYS, use_ratio_based_loss=True)
    g_ours = torch.autograd.grad(ours, [ours_in[k] for k in KEYS])
    tag = f"ratio_s{seed}"
    ref = float(gold(tag + "_loss"))
    assert abs(float(ours) - ref) < 1e-6 * max(1.0, abs(ref))
    for k, a in zip(KEYS, g_ours):
        name = f"{tag}_g_{key_name(k)}"
        mine, b = sampled(name, a[None])
        assert np.abs(mine - b).max() < 1e-7 + 1e-4 * float(gold(name + "_absmax"))


def test_boxdiff_loop_matches_reference():
    """generate_semantic_guidance(use_boxdiff=True) (generation/boxdiff.py:126-137 -> utils/boxdiff.py:190-259): one
    BoxDiff step per denoising step with the sqrt step schedule, vs oracle pipeline_ref.denoise(boxdiff=...)"""
    cfg, w, z0, uncond, cond, _ = _pipeline_inputs(False)
    keys = [("down", 2, 0, 0), ("down", 2, 1, 0), ("up", 1, 0, 0), ("up", 1, 1, 0), ("up", 1, 2, 0)]
    bboxes = [[(0.1, 0.2, 0.6, 0.7)], [(0.5, 0.4, 0.95, 0.9), (0.0, 0.0, 0.4, 0.4)]]
    positions = [[2, 3], [6]]
    steps = 4
    res = pipeline_ref.denoise(w, cfg, z0, uncond, cond, steps,
                               boxdiff=dict(bboxes=bboxes, object_positions=positions, keys=keys, max_index_step=3))
    assert len(res["boxdiff_losses"]) == 3
    assert np.abs(np.subtract(*sampled("boxdiff_loop_latents", res["latents"]))).max() < 5e-3


# ---------------------------------------------------------------------------------------------------------------------
# mask refinement around the SAM network (SURVEY.md 8 f-3): lgd_b200.mask_refine vs the UNMODIFIED models/sam.py, both
# driven by the same synthetic "SAM network" (three candidate masks + predicted IoUs as a function of the prompt)
def _fake_prompt(input_boxes, input_points):
    if input_boxes is not None:          # [[[4]]] from sam_refine_boxes, [[4]] from sam_refine_attn (models/sam.py:141-142)
        b = input_boxes[0]
        return "box", (b if np.ndim(b) == 1 else b[0])
    return "point", input_points[0][0]


def _fake_sam_candidates(prompt_kind, prompt, size=512, seed=0):
    """deterministic stand-in for facebook/sam-vit-base: candidates grown from the prompt (whole / part / over-grown
    object, the usual three granularities), scores from a seeded generator"""
    rng = np.random.RandomState(seed + int(sum(np.ravel(prompt))) % 9973)
    yy, xx = np.mgrid[0:size, 0:size]
    if prompt_kind == "box":
        x0, y0, x1, y1 = [float(v) for v in prompt]
    else:
        px, py = [float(v) for v in prompt]
        w, h = rng.uniform(60, 200), rng.uniform(60, 200)
        x0, y0, x1, y1 = px - w / 2, py - h / 2, px + w / 2, py + h / 2
    cx, cy, rx, ry = (x0 + x1) / 2, (y0 + y1) / 2, max((x1 - x0) / 2, 2.0), max((y1 - y0) / 2, 2.0)
    ell = lambda s: (((xx - cx) / (rx * s)) ** 2 + ((yy - cy) / (ry * s)) ** 2) <= 1.0
    masks = np.stack([ell(0.9), ell(0.45) & (yy < cy), ell(rng.uniform(1.3, 2.5))])
    scores = rng.uniform(0.7, 1.0, size=3).astype(np.float32)
    return masks, scores


class _FakeSamInputs(dict):
    def to(self, device):
        return self


class _FakeSamProcessor:
    def __init__(self, seed):
        self.seed = seed
        self.image_processor = self

    def __call__(self, image, input_points=None, input_boxes=None, return_tensors="pt"):
        kind, prompt = _fake_prompt(input_boxes, input_points)
        if isinstance(image, list):                      # sam_refine_boxes hands over a list of images
            image = image[0]
        masks, scores = _fake_sam_candidates(kind, prompt, size=np.asarray(image).shape[0], seed=self.seed)
        return _FakeSamInputs(masks=torch.from_numpy(masks), scores=torch.from_numpy(scores),
                              original_sizes=torch.tensor([[masks.shape[1], masks.shape[2]]]),
                              reshaped_input_sizes=torch.tensor([[1024, 1024]]))

    def post_process_masks(self, pred_masks, original_sizes, reshaped_input_sizes):
        return [pred_masks[0] > 0]                       # [n_prompts = 1, 3, h, w] bool per image


class _FakeSamModel:
    def __call__(self, masks, scores, original_sizes, reshaped_input_sizes):
        import types
        return types.SimpleNamespace(pred_masks=(masks.float() * 2 - 1)[None, None], iou_scores=scores[None, None])


def _fake_predict(seed):
    def predict(image, input_boxes=None, input_points=None):
        kind, prompt = _fake_prompt(input_boxes, input_points)
        return _fake_sam_candidates(kind, prompt, size=np.asarray(image).shape[0], seed=seed)
    return predict


def mask_refine_box_cases(seed):
    """(image, [(box, conf_th, iou_th)] x 6) of one seed"""
    rng = np.random.RandomState(seed)
    image = rng.randint(0, 255, size=(512, 512, 3)).astype(np.uint8)
    cases = []
    for _ in range(6):
        x0, y0 = rng.uniform(0, 0.6, size=2)
        box = (x0, y0, x0 + rng.uniform(0.08, 0.4), y0 + rng.uniform(0.08, 0.4))
        cases.append((box, rng.choice([0.85, 0.8, 0.95]), rng.choice([0.2, 0.25, 0.6])))
    return image, cases


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_mask_refine_box_matches_reference_sam(seed):
    from lgd_b200 import mask_refine as MR
    image, cases = mask_refine_box_cases(seed)
    for i, (box, conf_th, iou_th) in enumerate(cases):
        m, c = MR.refine_box(_fake_predict(seed), image, box, 512, 512, 64, 64, discourage_mask_below_confidence=conf_th,
                             discourage_mask_below_coarse_iou=iou_th)
        assert m.dtype == np.bool_ and m.shape == (64, 64)
        tag = f"sam_box_s{seed}_{i}"
        assert digest(m) == gold(tag + "_mask") and float(c) == float(gold(tag + "_conf"))


def mask_refine_attn_cases(use_box_input, side):
    """(image, [token-attention map] x 6): a blob plus noise, like utils/attn.py get_token_attnv2 hands over"""
    rng = np.random.RandomState(10 + side + int(use_box_input))
    image = rng.randint(0, 255, size=(512, 512, 3)).astype(np.uint8)
    attns = []
    for _ in range(6):
        yy, xx = np.mgrid[0:side, 0:side] / side
        cx, cy, s = rng.uniform(0.25, 0.75), rng.uniform(0.25, 0.75), rng.uniform(0.08, 0.2)
        attns.append((np.exp(-((xx - cx) ** 2 + (yy - cy) ** 2) / (2 * s * s)) + 0.05 * rng.rand(side, side))
                     .astype(np.float32))
    return image, attns


def mask_refine_attn_kwargs(use_box_input):
    from lgd_b200 import mask_refine as MR
    sigma = MR.GAUSSIAN_SIGMA_BOX_INPUT if use_box_input else MR.GAUSSIAN_SIGMA_POINT_INPUT
    return dict(use_box_input=use_box_input, gaussian_sigma=sigma, mask_th_for_box=0.05, n_erode_dilate_mask_for_box=1,
                mask_th_for_point=0.25, discourage_mask_below_confidence=0.85, discourage_mask_below_coarse_iou=0.25)


@pytest.mark.parametrize("use_box_input", [False, True])
@pytest.mark.parametrize("side", [16, 64])
def test_mask_refine_attn_matches_reference_sam(use_box_input, side):
    from lgd_b200 import mask_refine as MR
    image, attns = mask_refine_attn_cases(use_box_input, side)
    kw = mask_refine_attn_kwargs(use_box_input)
    for i, attn in enumerate(attns):
        m, c = MR.refine_attn(_fake_predict(5), image, attn.copy(), 512, 512, 64, 64, **kw)
        tag = f"sam_attn_b{int(use_box_input)}_{side}_{i}"
        assert digest(m) == gold(tag + "_mask") and float(c) == float(gold(tag + "_conf"))
        mb, prompt = MR.attn_prompt(attn, 512, 512, use_box_input, kw["gaussian_sigma"])
        assert mb.shape == (side, side) and (("input_boxes" in prompt) == use_box_input)


def select_mask_cases():
    rng = np.random.RandomState(0)
    for _ in range(50):
        masks = rng.rand(3, 32, 32) > rng.uniform(0.2, 0.9, size=(3, 1, 1))
        conf = rng.uniform(0.6, 1.0, size=3)
        ious = rng.uniform(0.0, 0.6, size=3) if rng.rand() < 0.7 else None
        yield masks, conf, ious


def test_select_mask_rule_matches_reference():
    from lgd_b200 import mask_refine as MR
    for i, (masks, conf, ious) in enumerate(select_mask_cases()):
        b, cb = MR.select_mask(masks, conf, ious, 0.85, 0.2)
        assert digest(b) == gold(f"select_mask_{i}_mask") and cb == float(gold(f"select_mask_{i}_conf"))
