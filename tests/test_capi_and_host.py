"""CPU-side checks: the C-ABI library loads and exports every symbol include/b200lmd.h declares; host logic (loss
tables, latents bookkeeping, spec conversion, DDIM scalars, synthetic env) agrees with the oracle / reference."""
import ctypes
import os
import random
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    import __graft_entry__ as ge
    ge.build()
    return ctypes.CDLL(os.path.join(ROOT, "llm-groundeddiffusion_b200", "libb200lmd.so"))


def test_library_exports_every_declared_symbol():
    lib = _lib()
    hdr = open(os.path.join(ROOT, "include", "b200lmd.h")).read()
    names = set(re.findall(r"\b(b200lmd_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 30
    for n in sorted(names):
        assert hasattr(lib, n), f"missing export {n}"
    assert lib.b200lmd_version() >= 100
    assert lib.b200lmd_round_dp(40) == 64 and lib.b200lmd_round_dp(160) == 192
    assert lib.b200lmd_round_d16(40) == 48 and lib.b200lmd_round_d16(160) == 160


def test_struct_sizes_match_c_abi():
    from lgd_b200 import guidance as G
    from lgd_b200.unet import GemmDesc
    assert G.TERM_DTYPE.itemsize == 36
    assert ctypes.sizeof(G.XattnLossC) == 9 * 8 + 3 * 4 + 4       # 9 pointers, int, 2 floats, tail padding
    assert ctypes.sizeof(GemmDesc) > 200


def test_no_cpu_fallback(tmp_path, monkeypatch):
    from lgd_b200 import _lib as L
    monkeypatch.setattr(L, "_lib", None)
    monkeypatch.setattr(L, "LIB_PATH", str(tmp_path / "missing.so"))
    with pytest.raises(L.B200Error):
        L.lib()


def test_loss_tables_match_oracle_integers():
    from lgd_b200 import guidance as G
    from oracle import guidance_ref
    rng = random.Random(0)
    for _ in range(300):
        x0, y0 = rng.uniform(-0.1, 0.9), rng.uniform(-0.1, 0.9)
        box = (x0, y0, x0 + rng.uniform(0, 0.8), y0 + rng.uniform(0, 0.8))
        for side in (8, 16, 24, 64):
            assert G.scale_proportion(box, side, side) == guidance_ref.scale_proportion(box, side, side)
            m1, m2 = G.box_mask([box], side), guidance_ref.box_mask([box], side)
            assert np.array_equal(m1.astype(np.float32), m2)
            assert G.topk_sizes(m1, 0.2, 0.2) == guidance_ref.topk_sizes(m2, 0.2, 0.2)


def test_term_weights_and_slots():
    from lgd_b200 import guidance as G
    lay = [G.SampleLayout([[(0.1, 0.1, 0.5, 0.5)], [(0.5, 0.5, 0.9, 0.9), (0.0, 0.6, 0.3, 1.0)]], [[2, 3], [5]], [3, 5],
                          [[{("mid", 0, 0, 0): np.ones((8, 64), np.float32)}],
                           [{("mid", 0, 0, 0): np.ones((8, 64), np.float32)}] * 2])]
    p = G.LossParams(loss_scale=5.0, fg_weight=1.0, bg_weight=4.0, ref_ca_loss_weight=2.0, ref_word_token_only=True,
                     use_ref=True)
    from lgd_b200._lib import lib
    try:
        lib()
    except Exception:
        pytest.skip("library not built")
    slot_tok, slot_of = G.assign_slots(lay, p)
    assert slot_tok[0, :3].tolist() == [2, 3, 5] and slot_tok[0, 3] == -1
    off, terms, masks, refs = G.build_key_tables(lay, slot_of, ("mid", 0, 0, 0), 64, 8, 4, p)
    assert off.tolist() == [0, 6]           # 3 energy terms + 3 reference terms (1 + 2 boxes)
    e = terms[terms["type"] == 0]
    np.testing.assert_allclose(e["w_fg"], [5 / (2 * 2 * 4), 5 / (2 * 2 * 4), 5 / (1 * 2 * 4)], rtol=1e-6)
    np.testing.assert_allclose(e["w_bg"], 4 * e["w_fg"], rtol=1e-6)
    rterm = terms[terms["type"] == 1]
    np.testing.assert_allclose(rterm["w_ref"], [5 * 2 / 1 / 8 / 8, 5 * 2 / 2 / 8 / 8, 5 * 2 / 2 / 8 / 8], rtol=1e-6)
    assert len(refs) == 3 and masks.shape == (5, 64)


def test_ddim_schedule_matches_oracle():
    from lgd_b200.pipelines import DDIMSchedule
    from oracle.pipeline_ref import DDIM
    a, b = DDIMSchedule(), DDIM()
    for n in (4, 10, 50):
        a.set_timesteps(n)
        b.set_timesteps(n)
        assert a.timesteps.tolist() == b.timesteps.tolist()
        for t in a.timesteps:
            sa_t, sb_t, sa_p, sb_p = a.coefs(t)
            x = torch.randn(1, 4, 8, 8, generator=torch.Generator().manual_seed(int(t)))
            e = torch.randn(1, 4, 8, 8, generator=torch.Generator().manual_seed(int(t) + 1))
            mine = sa_p * (x - sb_t * e) / sa_t + sb_p * e
            assert (mine - b.step(e, t, x)).abs().max() < 2e-5


def latents_helper_cases():
    """(tensor, dx, dy, box) x 50"""
    rng = random.Random(1)
    g = torch.Generator().manual_seed(1)
    for _ in range(50):
        t = torch.randn(3, 2, 16, 16, generator=g)
        dx, dy = rng.uniform(-0.6, 0.6), rng.uniform(-0.6, 0.6)
        box = (0.1, 0.2, 0.1 + rng.uniform(0.1, 0.7), 0.2 + rng.uniform(0.1, 0.7))
        yield t, dx, dy, box


def test_latents_helpers_match_reference():
    """utils/utils.py shift_tensor, proportion_to_mask, binary_mask_to_box_mask, binary_mask_to_center, get_centered_box
    vs latents.py; the reference's outputs are stored in tests/golden/oracle_vs_reference.npz (exact results as
    digests, see oracle/make_goldens.py vs_reference)"""
    import test_oracle_vs_reference as T
    from lgd_b200 import latents as L
    from lgd_b200.generation.common import centered_box
    for i, (t, dx, dy, box) in enumerate(latents_helper_cases()):
        tag = f"latents_{i}"
        assert T.digest(L.shift(t, dx, dy)) == T.gold(tag + "_shift")
        assert T.digest(L.box_to_mask(box, 64, 64)) == T.gold(tag + "_box_mask")
        m = L.box_to_mask(box, 16, 16).bool()
        assert T.digest(L.mask_to_box_mask(m)) == T.gold(tag + "_mask_to_box")
        cx, cy = L.mask_center(m)
        rx, ry = T.gold(tag + "_center")
        assert abs(cx - rx) < 1e-6 and abs(cy - ry) < 1e-6
        np.testing.assert_allclose(centered_box(box, False, "floor_padding", 0.2), T.gold(tag + "_centered_box"),
                                   rtol=1e-12)


def test_convert_spec_and_synthetic_env():
    from lgd_b200.env import SyntheticEnv
    from lgd_b200.generation.common import convert_spec
    spec = dict(prompt="", bg_prompt="a photo of a room", extra_neg_prompt="",
                gen_boxes=[("a dog", [10, 20, 100, 120]), ("a cat", [200, 220, 150, 100]), ("a dog", [300, 30, 80, 90])])
    so, prompt, overall = convert_spec(spec)
    assert [s[1] for s in so] == ["a cat", "a dog", "a dog"]
    assert prompt == "a photo of a room with a cat, two dogs"
    assert overall[1][0] == "two dogs" and len(overall[1][2]) == 2
    np.testing.assert_allclose(so[0][3], (200 / 512, 220 / 512, 350 / 512, 320 / 512))
    env = SyntheticEnv()
    pos, widx, p2 = env.phrase_indices(prompt, ["a cat", "two dogs"], ["cat", "dogs"])
    toks = env.tokens(p2)
    assert [toks[i] for i in pos[0]] == ["a", "cat"] and toks[widx[1]] == "dogs"
    pos, widx, p3 = env.phrase_indices("a room", ["a bird"], ["bird"])
    assert p3 == "a room| a bird" and env.tokens(p3)[widx[0]] == "bird"
    u, c = env.encode_prompts(["x", "y"], "neg")
    assert u.shape == (1, 77, 768) and c.shape == (2, 77, 768) and not torch.equal(c[0], c[1])


def test_fast_schedule_host_logic():
    """utils/schedule.py:4-19 semantics on the host scheduler (known-answer: 10 steps, cut after 5, every 2nd)"""
    from lgd_b200.pipelines import DDIMSchedule
    s = DDIMSchedule()
    s.set_timesteps(10)
    assert s.timesteps.tolist() == [901, 801, 701, 601, 501, 401, 301, 201, 101, 1]
    s.apply_fast_schedule(5, 2)
    assert s.timesteps.tolist() == [901, 801, 701, 601, 501, 301, 101]
    nis = []
    for i, t in enumerate(s.timesteps.tolist()):
        s.adjust(i, t)
        nis.append(s.num_inference_steps)
    assert nis == [10, 10, 10, 10, 5, 5, 9]          # 1000 // (t - next t), last: 1000 // (101 + 1)
    s2 = DDIMSchedule()
    s2.set_timesteps(10)
    s2.apply_fast_schedule(9, 2)                     # cut at or past the end: unchanged
    assert len(s2.timesteps) == 10


def compose_cases():
    """(per-box latents [steps + 1, 1, 4, 16, 16] x 3, masks, background latents, steps, boxes)"""
    g = torch.Generator().manual_seed(0)
    steps = 6
    lat = [torch.randn(steps + 1, 1, 4, 16, 16, generator=g) for _ in range(3)]
    masks = []
    for i in range(3):
        m = torch.zeros(16, 16, dtype=torch.bool)
        m[2 + i:9 + i, 1 + 2 * i:8 + 2 * i] = True
        masks.append(m)
    bg = torch.randn(1, 4, 16, 16, generator=g)
    boxes = [(0.05, 0.1, 0.5, 0.6), (0.4, 0.3, 0.9, 0.8), (0.2, 0.5, 0.7, 0.95)]
    return lat, masks, bg, steps, boxes


def test_compose_and_align_match_reference():
    """utils/latents.py compose_latents (all steps and the fast-schedule prefix) and align_with_bboxes vs latents.py;
    the reference's outputs are stored in tests/golden/oracle_vs_reference.npz"""
    import test_oracle_vs_reference as T
    from lgd_b200 import latents as L
    lat, masks, bg, steps, boxes = compose_cases()
    for fast in (None, 3):
        n = steps if fast is None else fast
        mine_c, mine_fg = L.compose([x[:n + 1] for x in lat], masks, bg, n)
        assert T.digest(mine_c) == T.gold(f"compose_fast{fast}_latents")
        assert T.digest(mine_fg) == T.gold(f"compose_fast{fast}_owner")
    for horizontal_only in (False, True):
        ml, mm, mo = L.align_to_boxes([x.clone() for x in lat], [m.clone() for m in masks], boxes,
                                      horizontal_only=horizontal_only)
        tag = f"align_h{int(horizontal_only)}"
        assert [T.digest(a) for a in ml] == T.gold(tag + "_latents").split(",")
        assert [T.digest(a) for a in mm] == T.gold(tag + "_masks").split(",")
        np.testing.assert_allclose(np.array(mo, dtype=np.float64), T.gold(tag + "_offsets"), rtol=0, atol=1e-7)


def test_boxdiff_tables_and_struct():
    """integer artefacts of the BoxDiff tables (cell masks, corner masks, k = floor(count * P) without clamp) against a
    direct restatement of utils/boxdiff.py:48-87, and the C-ABI struct sizes"""
    from lgd_b200 import boxdiff as BD, guidance as G
    from oracle import guidance_ref
    assert BD.TERM_DTYPE.itemsize == 20
    assert ctypes.sizeof(BD.BoxdiffC) == 256      # 16 + 7 pointers, 6 + 1 ints, 9 + 1 floats, tail padding
    rng = random.Random(1)
    for _ in range(50):
        side = rng.choice([8, 16, 24])
        lay = []
        for b in range(2):
            boxes = []
            for _o in range(rng.randint(1, 3)):
                w_, h_ = rng.uniform(0.35, 0.6), rng.uniform(0.35, 0.6)
                x, y = rng.uniform(0, 1 - w_), rng.uniform(0, 1 - h_)
                boxes.append([(x, y, x + w_, y + h_)])
            lay.append(G.SampleLayout(boxes, [[1 + 2 * i, 2 + 2 * i] for i in range(len(boxes))]))
        off, terms, masks, corner = BD.build_tables(lay, side, 0.2, 1)
        assert off.tolist() == [0, 2 * len(lay[0].bboxes), 2 * (len(lay[0].bboxes) + len(lay[1].bboxes))]
        ti = 0
        for s in lay:
            for o, obj in enumerate(s.bboxes):
                m = torch.zeros(side, side)
                cx, cy = torch.zeros(side), torch.zeros(side)
                for box in obj:
                    x0, y0, x1, y1 = guidance_ref.scale_proportion(box, side, side)
                    m[y0:y1, x0:x1] = 1
                    cx[max(x0 - 1, 0):min(x0 + 2, side)] = 1.
                    cx[max(x1 - 1, 0):min(x1 + 2, side)] = 1.
                    cy[max(y0 - 1, 0):min(y0 + 2, side)] = 1.
                    cy[max(y1 - 1, 0):min(y1 + 2, side)] = 1.
                for tok in s.object_positions[o]:
                    t = terms[ti]
                    assert t["tok"] == tok
                    assert np.array_equal(masks[t["mask"]], m.reshape(-1).numpy().astype(np.uint8))
                    assert np.array_equal(corner[t["corner"]], torch.cat([cx, cy]).numpy().astype(np.uint8))
                    assert t["k_fg"] == int((m.sum() * 0.2).long()) and t["k_bg"] == int(((1 - m).sum() * 0.2).long())
                    ti += 1
    with pytest.raises(ValueError):
        BD.build_tables([G.SampleLayout([[(0.1, 0.1, 0.2, 0.2)]], [[1]])], 16, 0.2, 1)


def test_compose_owners_match_host_compose():
    import lgd_b200.latents as L
    g = torch.Generator().manual_seed(3)
    for trial in range(10):
        H = W = 64
        boxes = [(0.1 + 0.05 * trial % 0.3, 0.2, 0.5, 0.7), (0.4, 0.3, 0.95, 0.9), (0.3, 0.05, 0.6, 0.35)]
        masks = [L.box_to_mask(b, H, W).bool() for b in boxes]
        lat = [torch.randn(3, 1, 4, H, W, generator=g) for _ in boxes]
        _, fg_idx = L.compose(lat, masks, torch.randn(1, 4, H, W, generator=g), 2)
        ow, bow = L.compose_owners(masks)
        assert torch.equal(ow.long(), fg_idx)
        assert int((bow > 0).sum()) >= int((ow > 0).sum())
    assert L.shift_cells(0.26, -0.13, 64, 64) == (16, -8)


def test_guidance_step_scale_branches():
    """models/pipelines.py:60-69: sigmas[index]**2 when the scheduler carries sigmas, sqrt(1 - alpha_bar_t) otherwise"""
    from lgd_b200.pipelines import DDIMSchedule, guidance_step_scale
    s = DDIMSchedule()
    s.set_timesteps(50)
    t = int(s.timesteps[3])
    assert abs(guidance_step_scale(s, 3, t) - float((1 - s.alphas_cumprod[t]) ** 0.5)) < 1e-12
    s.sigmas = np.linspace(14.6, 0.0, 51)
    assert abs(guidance_step_scale(s, 3, t) - float(s.sigmas[3]) ** 2) < 1e-12


def test_env_refine_mask_with_sam_predict_hook():
    """ReferenceEnv(sam_predict=...): prompt construction and candidate selection run in mask_refine, only the network
    call is the hook (models/sam.py; the bit-exact comparison with the reference lives in test_oracle_vs_reference.py)"""
    import numpy as np
    import torch
    from lgd_b200 import mask_refine as MR
    from lgd_b200.env import ReferenceEnv
    calls = []

    def predict(image, input_boxes=None, input_points=None):
        calls.append((input_boxes, input_points))
        yy, xx = np.mgrid[0:512, 0:512]
        if input_boxes is not None:
            b = input_boxes[0]
            x0, y0, x1, y1 = b if np.ndim(b) == 1 else b[0]
        else:
            px, py = input_points[0][0]
            x0, y0, x1, y1 = px - 64, py - 64, px + 64, py + 64
        inside = (xx >= x0) & (xx < x1) & (yy >= y0) & (yy < y1)
        small = inside & (xx < (x0 + x1) / 2)
        return np.stack([inside, small, np.ones_like(inside)]), np.array([0.95, 0.99, 0.5], dtype=np.float32)

    env = ReferenceEnv(model_dict=None, sam_predict=predict)
    image = np.zeros((512, 512, 3), dtype=np.uint8)
    box = (0.25, 0.25, 0.75, 0.5)
    m = env.refine_mask(image, box, 64, 64)                       # LMD+: box prompt in pixels
    assert calls[-1][0] == [[[128, 128, 384, 256]]] and calls[-1][1] is None
    assert m.dtype == torch.bool and m.shape == (64, 64)
    # candidate 2 (everything) has confidence 0.5 < 0.85 and is pushed back; candidate 0 (the box) is the largest left
    assert int(m.sum()) >= 32 * 16 and not bool(m[0, 0])
    attn = np.zeros((16, 16), dtype=np.float32)
    attn[8, 4] = 1.0
    m2 = env.refine_mask(image, box, 64, 64, token_attn=torch.from_numpy(attn))     # LMD: point prompt at the arg-max
    assert calls[-1][0] is None and calls[-1][1] == [[[4 * 32, 8 * 32]]]
    assert m2.shape == (64, 64) and bool(m2[8 * 4, 4 * 4])
    attn[6:11, 3:9] = 1.0                                         # a blob survives the binary opening of the box path
    mb, prompt = MR.attn_prompt(attn, 512, 512, use_box_input=True)
    assert list(prompt) == ["input_boxes"] and len(prompt["input_boxes"][0]) == 4
    with __import__("pytest").raises(ValueError):
        MR.binary_mask_to_box(np.zeros((4, 4), dtype=bool))


def test_measurement_helpers_read_committed_profiles():
    """bench.py takes `roofline.traffic` from the committed ncu export (not a literal), and the launch-list summariser
    parses the committed ncu CSV of the final tree"""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    traffic, src = bench.ncu_dram_traffic()
    assert src == os.path.join("profiles", "xattn_fused_ncu_raw.csv")
    assert 15e6 < traffic < 40e6          # x + Wq + Wo + K/V + residual of the roofline shape: ~20.8 MB per launch
    out = subprocess.run([sys.executable, os.path.join(root, "profiles", "launches_summary.py"),
                          os.path.join(root, "profiles", "r2", "launches_step_call12.csv")],
                         capture_output=True, text=True, check=True).stdout
    assert "b200::xattn_fused_kernel<160>" in out and "b200::gemm2_tc_kernel" in out
    assert "this library's kernels" in out.splitlines()[0]


def test_product_path_never_touches_the_oracle():
    """only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may use oracle/: no module
    of the package imports it, and bench.py imports it only inside the CPU arm (class CpuArm)"""
    import ast
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def oracle_imports(path):
        tree = ast.parse(open(path).read())
        hits = []
        for node in ast.walk(tree):
            names = []
            if isinstance(node, ast.Import):
                names = [a.name for a in node.names]
            elif isinstance(node, ast.ImportFrom):
                names = [node.module or ""]
            hits += [(node.lineno, n) for n in names if n == "oracle" or n.startswith("oracle.")]
        return tree, hits

    pkg = os.path.join(root, "llm-groundeddiffusion_b200")
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                assert oracle_imports(os.path.join(d, f))[1] == [], os.path.join(d, f)
    tree, hits = oracle_imports(os.path.join(root, "bench.py"))
    arm = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "CpuArm"][0]
    lo, hi = arm.lineno, max(getattr(n, "end_lineno", arm.lineno) for n in ast.walk(arm) if hasattr(n, "end_lineno"))
    assert hits and all(lo <= line <= hi for line, _ in hits), (hits, lo, hi)


def test_bench_dump_outputs_host_side(tmp_path):
    """bench.py --dump-outputs: float32/float64 .npy files within 64 MB, large outputs as the same seeded sample on
    every call"""
    import bench
    from lgd_b200.generation.common import Output
    rng = np.random.RandomState(0)

    def outs():
        res = []
        for b in range(2):
            o = Output(image=rng.randint(0, 255, size=(64, 64, 3)).astype(np.uint8),
                       so_img_list=[rng.randint(0, 255, size=(64, 64, 3)).astype(np.uint8) for _ in range(2)])
            o["latents"] = torch.from_numpy(rng.randn(1, 4, 8, 8).astype(np.float32)).half()
            res.append(o)
        return res

    first = outs()
    a = bench.step_outputs(first, [3, 4])
    assert a["latents"].shape == (2, 4, 8, 8) and a["images"].shape == (2, 64, 64, 3)
    assert a["guidance_iterations"].tolist() == [3.0, 4.0]
    so = np.stack([im for o in first for im in o.so_img_list]).reshape(-1)
    assert a["so_images_sample"].size == min(so.size, bench.SO_IMAGE_SAMPLE)
    np.testing.assert_array_equal(a["so_images_sample"], so[a["so_images_index"].astype(np.int64)])
    b = bench.step_outputs(outs(), [3, 4])
    np.testing.assert_array_equal(a["so_images_index"], b["so_images_index"])
    bench.write_outputs(str(tmp_path / "d"), a)
    for name, v in a.items():
        got = np.load(tmp_path / "d" / (name + ".npy"))
        assert got.dtype in (np.float32, np.float64) and np.array_equal(got, v)
    with pytest.raises(AssertionError):
        bench.write_outputs(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_BYTES // 4 + 1, np.float32)})
