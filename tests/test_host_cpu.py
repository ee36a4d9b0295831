"""CPU tests of the host-side logic: C-ABI surface, weight packing, scheduler tables, shard planning and the
world_size-2 gloo path of the temporal K/V gather."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_c_abi_library_exports_every_declared_symbol():
    import __graft_entry__ as g
    g.build()
    hdr = open(os.path.join(ROOT, "include", "hallo_b200.h")).read()
    names = sorted(set(re.findall(r"\b(hallo_b200_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 15
    cdll = ctypes.CDLL(os.path.join(ROOT, "hallo_b200", "libhallo_b200.so"))
    missing = [n for n in names if not hasattr(cdll, n)]
    assert not missing, missing
    cdll.hallo_b200_abi_version.restype = ctypes.c_int
    assert cdll.hallo_b200_abi_version() == 3
    assert not any("ubench" in n for n in names), "micro-benchmarks are not part of the public ABI"


def test_ctypes_structs_match_the_compiled_header():
    """The ctypes mirrors in hallo_b200/lib.py (and the copy shown in INTEGRATION.md) must have exactly the size the
    library was compiled with; a short struct would make the library read past the caller's memory."""
    import __graft_entry__ as g
    g.build()
    from hallo_b200 import lib
    h = lib.load()
    assert ctypes.sizeof(lib.GemmParams) == h.hallo_b200_sizeof_gemm_params()
    assert ctypes.sizeof(lib.AttentionParams) == h.hallo_b200_sizeof_attention_params()
    # the struct printed in INTEGRATION.md: same field names, in the same order, as the binding the repo itself uses
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    block = doc[doc.index("class GemmParams"):doc.index("def linear")]
    doc_fields = re.findall(r'\("([A-Za-z0-9_]+)",\s*C\.c_', block)
    assert doc_fields == [f[0] for f in lib.GemmParams._fields_], doc_fields


def test_no_undefined_names_in_gpu_only_code():
    """GPU-only branches (tests marked gpu, bench.py, the engine) cannot run here; at least every global name they
    load must be bound (a missing import in a GPU test fixture would otherwise only surface on the box)."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "lint_names.py")], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:]


def test_kernel_selection_options_roundtrip():
    """hallo_b200_set_option / get_option are host-only; the defaults are the kernels promoted after their hardware
    A/B runs (profiles/r2_first_call_summary.txt), everything still experimental stays off."""
    import __graft_entry__ as g
    g.build()
    from hallo_b200 import lib
    defaults = {"gemm_tepi": 1, "gemm_1cta": 0, "gemm_fill": 1, "attn_occ2": 1, "attn_poly": 0, "attn_v1": 0,
                "xattn_tc": 1, "tattn_mma": 1, "gn_fused": 1, "gemm_splitk": 1, "pdl": 0}
    for name, dflt in defaults.items():
        if os.environ.get("HALLO_B200_" + name.upper()) is None:
            assert lib.get_option(name) == dflt, name
        old = lib.get_option(name)
        lib.set_option(name, 3)
        assert lib.get_option(name) == 3
        lib.set_option(name, old)
    with pytest.raises(RuntimeError):
        lib.set_option("no_such_option", 1)
    for gone in ("no_such_option", "attn_chunk", "attn_v3"):          # losers of the A/B runs were deleted
        with pytest.raises(KeyError):
            lib.get_option(gone)


def test_no_cpu_fallback_in_product_path():
    """The product must fail loudly without CUDA, and must not import the oracle."""
    from hallo_b200.models.unet_3d import UNet3DConditionModel
    for dirpath, _, files in os.walk(os.path.join(ROOT, "hallo_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f
    if not torch.cuda.is_available():
        from hallo_b200.spec import HALLO_UNET_KWARGS, SD15_UNET_CONFIG
        tiny = dict(SD15_UNET_CONFIG)
        m = UNet3DConditionModel.from_config(tiny, **HALLO_UNET_KWARGS)
        m.set_banks({"x": torch.zeros(1)})
        with pytest.raises(RuntimeError):
            m(torch.zeros(2, 4, 1, 8, 8), 1, torch.zeros(2, 4, 768), audio_embedding=torch.zeros(2, 1, 32, 768),
              mask_cond_fea=None, full_mask=[torch.zeros(2, 64)], face_mask=[torch.zeros(2, 64)],
              lip_mask=[torch.zeros(2, 64)])


def test_weight_packing_layouts():
    from hallo_b200 import ops
    g = torch.Generator().manual_seed(0)
    w = torch.randn(16, 8, 3, 3, generator=g)
    x = torch.randn(2, 8, 5, 5, generator=g)
    wp = ops.pack_conv3x3_weight(w)                                   # [cout, (kh kw cin)]
    cols = F.unfold(x, 3, padding=1).view(2, 8, 9, 25).permute(0, 3, 2, 1).reshape(50, 72)   # (tap, cin) order
    ref = F.conv2d(x, w, padding=1).permute(0, 2, 3, 1).reshape(50, 16)
    assert torch.allclose(cols @ wp.t(), ref, atol=1e-4)
    w1 = torch.randn(32, 4, generator=g)
    b1 = torch.randn(32, generator=g)
    wi, bi = ops.pack_geglu_weight(w1, b1)
    h = torch.randn(3, 4, generator=g)
    full = h @ w1.t() + b1
    inter = h @ wi.t() + bi
    assert torch.allclose(inter[:, 0::2], full[:, :16]) and torch.allclose(inter[:, 1::2], full[:, 16:])


def test_scheduler_tables():
    from hallo_b200.scheduler import DDIMScheduler
    s = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="linear", clip_sample=False, steps_offset=1,
                      prediction_type="v_prediction", rescale_betas_zero_snr=True, timestep_spacing="trailing")
    s.set_timesteps(40)
    assert s.timesteps.tolist()[:2] == [999, 974] and s.timesteps.tolist()[-1] == 24
    c = s.coef_table()
    assert c.shape == (40, 4) and abs(float(c[0, 0])) < 1e-6 and abs(float(c[-1, 2]) - 1.0) < 1e-7
    assert torch.allclose(c[:, 0] ** 2 + c[:, 1] ** 2, torch.ones(40), atol=1e-6)
    assert torch.allclose(c[1:, 0], c[:-1, 2], atol=1e-6)            # a_prev of step i == a_t of step i+1


def test_shard_layout():
    from hallo_b200.dist import shard_layout
    for world in (1, 2, 4, 8, 16):
        lay = shard_layout(world, 16)
        rows = sorted((b, g) for halves, frames in lay for b in halves for g in frames)
        assert rows == [(b, g) for b in (0, 1) for g in range(16)]    # every (half, frame) owned exactly once
        assert all(halves == (0, 1) and len(frames) == 16 // world for halves, frames in lay)   # balanced, CFG-local
    with pytest.raises(ValueError):
        shard_layout(3, 16)


def test_row_scatter_matches_the_frame_owner_layout():
    """The proj_out epilogue's hb_row_scatter parameters (engine._motion_px): GEMM row (global frame g, pixel p of rank
    me's slice) of half b must land at row (b*fl + g % fl)*L + me*Lg + p of rank g // fl; the GroupNorm scatter's
    (frame n = b*fl + j, pixel p) at row (b*F18 + nm + me*fl + j)*Lg + p % Lg of rank p // Lg."""
    from hallo_b200.dist import scatter_row_destination
    nb, nm, f, R, L = 2, 2, 16, 4, 64
    fl, Lg, F18 = f // R, L // R, nm + f
    for me in range(R):
        for b in range(nb):
            for g in range(f):
                for pp in (0, 1, Lg - 1):
                    d, row = scatter_row_destination(g * Lg + pp, seg=Lg, segs_per_dest=fl, seg_stride=L,
                                                     row0=b * fl * L + me * Lg)
                    assert d == g // fl and row == (b * fl + g % fl) * L + me * Lg + pp
    # GroupNorm scatter (csrc/aux.cu gn_apply_kernel): n_out = (n // fpb_in) * fpb_out + frame_off + n % fpb_in
    for me in range(R):
        for n in range(nb * fl):
            n_out = (n // fl) * F18 + (nm + me * fl) + n % fl
            b, j = divmod(n, fl)
            assert n_out == b * F18 + nm + me * fl + j


WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.environ["HB_ROOT"])
from hallo_b200.dist import plan_shard, frames_to_pixels, pixels_to_frames
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
n_frames, nb = 8, 2
sh = plan_shard(rank, world, n_frames, exchange="nccl")
fl = n_frames // world
assert sh.halves == (0, 1) and sh.frames == tuple(range(rank * fl, (rank + 1) * fl)) and sh.group_size == world
# frame<->pixel exchange around a motion module (engine._motion_px): a per-pixel op that mixes ALL frames (a cumulative
# sum over the frame axis + a per-frame scale) computed on pixel slices must equal the unsharded result, both halves
L, C = 6, 4
xg = (torch.arange(nb * n_frames * L * C, dtype=torch.float32).reshape(nb, n_frames, L, C) / 7.0).sin()   # global
x_loc = xg[:, rank * fl:(rank + 1) * fl].contiguous()                                   # my frames, both halves
Lg = L // world
allf = frames_to_pixels(x_loc, nb, fl, world, sh.group)
assert torch.equal(allf, xg[:, :, rank * Lg:(rank + 1) * Lg]), rank                      # my pixel slice of all frames
scale = torch.arange(1, n_frames + 1, dtype=torch.float32).view(1, n_frames, 1, 1)
y = (allf.cumsum(1) * scale).contiguous()
back = pixels_to_frames(y, nb, fl, world, sh.group) + x_loc
ref = (xg.cumsum(1) * scale + xg)[:, rank * fl:(rank + 1) * fl]
assert torch.allclose(back, ref), rank
dist.destroy_process_group()
print("ok", rank)
'''


def test_gloo_world2_frame_pixel_exchange(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(WORKER)
    env = dict(os.environ, HB_ROOT=ROOT, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29577", str(script)],
                       env=env, capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stdout.count("ok") == 2


def test_layernorm_fold_algebra():
    """ops.fold_layernorm: rstd * (x W'^T - mu * colsum) + b' == Linear(LayerNorm(x)) (checked in fp32 on the host)."""
    from hallo_b200 import ops
    g = torch.Generator().manual_seed(3)
    M, C, N = 37, 64, 48
    x = torch.randn(M, C, generator=g) * 3 + 1.5
    w = torch.randn(N, C, generator=g) / 8
    b = torch.randn(N, generator=g)
    gamma = 1 + 0.3 * torch.randn(C, generator=g)
    beta = 0.3 * torch.randn(C, generator=g)
    wg, cs, bb = ops.fold_layernorm(w, b, gamma, beta, torch.float32)
    mu = x.mean(1, keepdim=True)
    var = (x * x).mean(1, keepdim=True) - mu * mu              # the kernel's E[x^2] - mu^2 form
    rstd = torch.rsqrt(var + 1e-5)
    out = rstd * (x @ wg.t() - mu * cs[None, :]) + bb
    ref = F.linear(F.layer_norm(x, (C,), gamma, beta, 1e-5), w, b)
    assert torch.allclose(out, ref, atol=2e-4, rtol=1e-4)


def test_scheduler_step_matches_oracle_ddim():
    """DDIMScheduler.step (the call at face_animate.py:420) against the oracle's independent restatement, and against the
    coefficient table the device kernel consumes -- the three forms of the same v-prediction update must agree."""
    from hallo_b200.scheduler import DDIMScheduler
    from oracle import port
    s = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="linear", clip_sample=False, steps_offset=1,
                      prediction_type="v_prediction", rescale_betas_zero_snr=True, timestep_spacing="trailing")
    s.set_timesteps(40)
    o = port.DDIM()
    assert o.timesteps(40) == s.timesteps.tolist()
    g = torch.Generator().manual_seed(5)
    x = torch.randn(1, 4, 3, 8, 8, generator=g)
    c = s.coef_table()
    for i, t in enumerate(s.timesteps.tolist()):
        v = torch.randn(1, 4, 3, 8, 8, generator=g)
        mine = s.step(v, t, x).prev_sample
        assert torch.allclose(mine, o.step(v, t, x, 40), atol=2e-6)
        sa, sb, pa, pb = [float(z) for z in c[i]]
        assert torch.allclose(mine, pa * (sa * x - sb * v) + pb * (sa * v + sb * x), atol=2e-6)
        assert s.step(v, t, x, return_dict=False)[0].equal(mine)
        x = mine
    with pytest.raises(NotImplementedError):
        s.step(v, 24, x, eta=0.5)
    # a diffusers-style scheduler object (attributes only, no coef_table): same table through coef_table_of
    from types import SimpleNamespace
    from hallo_b200.scheduler import coef_table_of
    fake = SimpleNamespace(config=SimpleNamespace(num_train_timesteps=1000, prediction_type="v_prediction"),
                           num_inference_steps=40, timesteps=s.timesteps, alphas_cumprod=s.alphas_cumprod,
                           final_alpha_cumprod=s.final_alpha_cumprod)
    assert torch.equal(coef_table_of(fake), c) and torch.equal(coef_table_of(s), c)


def test_hallo_overlay_package_resolves_hot_path_to_b200_and_rest_to_reference(tmp_path):
    """scripts/inference.py:38-47 must run unchanged: with this repo ahead of the reference checkout on sys.path,
    `hallo.models.unet_3d / audio_proj / mutual_self_attention` and `hallo.animate.face_animate` are the B200 classes and
    every other hallo.* module still comes from the reference tree.  The checkout is a stub with the reference's package
    layout whose hot-path modules fail on import.  Run in a subprocess (clean sys.modules)."""
    ref = tmp_path / "reference"
    stub = {"__init__.py": "", "utils/__init__.py": "", "utils/config.py": "", "animate/__init__.py": "",
            "animate/face_animate_static.py": "", "models/__init__.py": "",
            "models/face_locator.py": "class FaceLocator:\n    pass\n",
            "models/image_proj.py": "class ImageProjModel:\n    pass\n"}
    for mod in ("animate/face_animate", "models/audio_proj", "models/unet_3d", "models/mutual_self_attention"):
        stub[mod + ".py"] = "raise ImportError('hot-path module resolved to the reference checkout')\n"
    for name, text in stub.items():
        (ref / "hallo" / name).parent.mkdir(parents=True, exist_ok=True)
        (ref / "hallo" / name).write_text(text)
    code = r'''
import os, sys
root, ref = sys.argv[1], sys.argv[2]
sys.path[:0] = [root, ref]
from hallo.animate.face_animate import FaceAnimatePipeline
from hallo.models.audio_proj import AudioProjModel
from hallo.models.unet_3d import UNet3DConditionModel
from hallo.models.mutual_self_attention import ReferenceAttentionControl
for cls in (FaceAnimatePipeline, AudioProjModel, UNet3DConditionModel, ReferenceAttentionControl):
    assert cls.__module__.startswith("hallo_b200."), cls.__module__
import hallo.utils.config as cfgmod                      # reference-only modules still resolve
assert os.path.abspath(cfgmod.__file__).startswith(os.path.abspath(ref)), cfgmod.__file__
import hallo.animate.face_animate_static as static
assert os.path.abspath(static.__file__).startswith(os.path.abspath(ref)), static.__file__
from hallo.models.face_locator import FaceLocator
from hallo.models.image_proj import ImageProjModel
assert os.path.abspath(sys.modules[FaceLocator.__module__].__file__).startswith(os.path.abspath(ref))
assert os.path.abspath(sys.modules[ImageProjModel.__module__].__file__).startswith(os.path.abspath(ref))
print("OK")
'''
    r = subprocess.run([sys.executable, "-c", code, ROOT, str(ref)], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout[-1500:] + r.stderr[-3000:]


def test_driver_window_logic_matches_reference_functions():
    """hallo_b200.driver restates three pieces of scripts/inference.py / audio_processor.py; process_audio_emb is also
    compared with what the unmodified script's function returned for the same input (tests/golden/process_audio_emb.pt,
    made by oracle/make_golden.py)."""
    from hallo_b200.driver import audio_frames, padded_sequence_length, process_audio_emb, window_reference_stack
    g = torch.Generator().manual_seed(0)
    emb = torch.randn(37, 12, 8, generator=g)
    mine = process_audio_emb(emb)
    # scripts/inference.py:95-114, restated literally
    ref = torch.stack([torch.stack([emb[max(min(i + j, emb.shape[0] - 1), 0)] for j in range(-2, 3)], 0)
                       for i in range(emb.shape[0])], 0)
    assert torch.equal(mine, ref)
    assert audio_frames(30 * 16000) == 750 and padded_sequence_length(750, 16) == 752 and 752 // 16 == 47   # configs[4]
    assert padded_sequence_length(752, 16) == 752
    src = torch.rand(1, 3, 8, 8, generator=g) * 2 - 1
    first = window_reference_stack(src, None, 2)
    assert first.shape == (1, 3, 3, 8, 8) and torch.equal(first[0, 1], src[0]) and torch.equal(first[0, 2], src[0])
    prev = torch.rand(1, 3, 16, 8, 8, generator=g)
    nxt = window_reference_stack(src, prev, 2)
    assert torch.equal(nxt[0, 0], src[0])
    assert torch.allclose(nxt[0, 1], prev[0, :, 14] * 2 - 1) and torch.allclose(nxt[0, 2], prev[0, :, 15] * 2 - 1)
    fx = torch.load(os.path.join(ROOT, "tests", "golden", "process_audio_emb.pt"), weights_only=False)
    assert fx["case"] == dict(shape=(37, 12, 8), seed=0) and torch.equal(fx["out"], mine)


def test_vae_architecture_contract():
    """hallo_b200.models.vae.AutoencoderKL: diffusers' SD-1.5 VAE key grammar and sizes (83,653,863 parameters, 248
    tensors), 8x spatial factor, encode().latent_dist.mean / decode().sample contract the pipeline uses."""
    from hallo_b200.models.vae import AutoencoderKL
    v = AutoencoderKL()
    sd = v.state_dict()
    assert len(sd) == 248 and sum(p.numel() for p in v.parameters()) == 83653863
    for k in ("encoder.down_blocks.0.downsamplers.0.conv.weight", "encoder.mid_block.attentions.0.to_q.bias",
              "decoder.up_blocks.0.upsamplers.0.conv.weight", "decoder.up_blocks.3.resnets.2.conv2.weight",
              "decoder.up_blocks.2.resnets.0.conv_shortcut.weight", "quant_conv.weight", "post_quant_conv.bias"):
        assert k in sd, k
    assert "decoder.up_blocks.3.upsamplers.0.conv.weight" not in sd and "encoder.down_blocks.3.downsamplers.0.conv.weight" not in sd
    assert len(v.config.block_out_channels) == 4
    x = torch.randn(2, 3, 32, 32)
    z = v.encode(x).latent_dist.mean
    assert tuple(z.shape) == (2, 4, 4, 4) and tuple(v.decode(z).sample.shape) == (2, 3, 32, 32)
    # per-sample independence (what lets the driver encode the source image once and decode frames in chunks)
    assert torch.allclose(v.encode(x[:1]).latent_dist.mean, z[:1], atol=1e-5)


def test_from_pretrained_2d_on_a_synthetic_checkpoint(tmp_path):
    """UNet3DConditionModel.from_pretrained_2d (hallo/models/unet_3d.py:717-839, scripts/inference.py:198-205) on a tiny
    SD-style directory: <base>/unet/config.json + 2-D weights, an AnimateDiff-style motion checkpoint, non-strict load,
    shape-mismatched tensors silently keep the model's own initialisation (:824-830)."""
    import json
    from hallo_b200.models.unet_3d import UNet3DConditionModel
    from hallo_b200.spec import HALLO_UNET_KWARGS, UNetConfig, param_spec, param_spec_2d
    base = tmp_path / "sd"
    (base / "unet").mkdir(parents=True)
    cfg_json = dict(_class_name="UNet2DConditionModel", _diffusers_version="0.6.0", sample_size=8, in_channels=4, out_channels=4,
                    center_input_sample=False, flip_sin_to_cos=True, freq_shift=0,
                    down_block_types=["CrossAttnDownBlock2D"] * 3 + ["DownBlock2D"],
                    up_block_types=["UpBlock2D"] + ["CrossAttnUpBlock2D"] * 3, block_out_channels=[32, 64, 128, 128],
                    layers_per_block=2, downsample_padding=1, mid_block_scale_factor=1, act_fn="silu", norm_num_groups=32,
                    norm_eps=1e-5, cross_attention_dim=768, attention_head_dim=8)
    json.dump(cfg_json, open(base / "unet" / "config.json", "w"))
    arch = UNetConfig(block_out_channels=(32, 64, 128, 128))
    g = torch.Generator().manual_seed(0)
    sd2d = {k: torch.randn(shape, generator=g) for k, shape, _ in param_spec_2d(arch)}
    sd2d["conv_norm_out.weight"] = torch.randn(32, generator=g)           # SD checkpoints carry the output head too
    sd2d["conv_in.weight"] = torch.randn(32, 9, 3, 3, generator=g)        # wrong shape on purpose (4 -> 9 input channels)
    torch.save(sd2d, base / "unet" / "diffusion_pytorch_model.bin")
    motion = {k: torch.randn(shape, generator=g) for k, shape, kind in param_spec(arch)
              if "motion_modules" in k and kind != "pe"}
    torch.save(motion, tmp_path / "mm.ckpt")
    m = UNet3DConditionModel.from_pretrained_2d(str(base), str(tmp_path / "mm.ckpt"), subfolder="unet",
                                                unet_additional_kwargs=dict(HALLO_UNET_KWARGS), use_landmark=False)
    own = m.state_dict()
    assert len(own) == len(param_spec(arch))
    k2 = "down_blocks.1.attentions.0.transformer_blocks.0.attn1.to_q.weight"
    km = "up_blocks.2.motion_modules.1.temporal_transformer.proj_in.weight"
    assert torch.equal(own[k2], sd2d[k2]) and torch.equal(own[km], motion[km])
    assert torch.equal(own["conv_norm_out.weight"], sd2d["conv_norm_out.weight"])
    assert own["conv_in.weight"].shape == (32, 4, 3, 3)                   # mismatched tensor: own init kept, no error
    ka = "mid_block.audio_modules.0.transformer_blocks.0.attn2_1.to_k.weight"
    assert ka in own and ka not in sd2d                                   # absent keys: non-strict load
    with pytest.raises(RuntimeError):
        UNet3DConditionModel.from_pretrained_2d(str(tmp_path / "nope"), str(tmp_path / "mm.ckpt"), subfolder="unet")
    with pytest.raises(RuntimeError):
        (tmp_path / "mm.bad").write_bytes(b"x")
        UNet3DConditionModel.from_pretrained_2d(str(base), str(tmp_path / "mm.bad"), subfolder="unet",
                                                unet_additional_kwargs=dict(HALLO_UNET_KWARGS), use_landmark=False)


def test_split_k_decision_is_host_arithmetic():
    """hallo_b200_gemm_choose_splits (include/hallo_b200.h): which launches divide their K loop, and how far.  Pure host
    arithmetic of the library, callable without a device."""
    import __graft_entry__ as g
    g.build()
    from hallo_b200 import lib
    h = lib.load()
    f = h.hallo_b200_gemm_choose_splits
    f.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_int]
    ws = int(h.hallo_b200_gemm_workspace_bytes())
    pairs = 74
    # level-3 conv of one rank of an 8-way shard: 5 tiles, K = 9 * 1280 -> 180 k-blocks -> ~sqrt(180 / 4) = 7 splits
    assert f(5, pairs, 11520, 2, 256, ws, 1) == 7
    # the FF-out GEMM of the same rank (K = 5120): 4 splits; the K = 1280 linears stay whole at the default threshold ...
    assert f(5, pairs, 5120, 2, 256, ws, 1) == 4
    assert f(5, pairs, 1280, 2, 256, ws, 1) == 1
    # ... and split in two when the option lowers the threshold to 16 k-blocks (the GPU tests use that)
    assert f(5, pairs, 1280, 2, 256, ws, 16) == 2
    # never more CTAs than SM pairs, never when the tiles already cover half of them, never without a workspace
    assert f(20, pairs, 11520, 2, 256, ws, 1) == 3
    assert f(40, pairs, 11520, 2, 256, ws, 1) == 1
    assert f(5, pairs, 11520, 2, 256, 0, 1) == 1
    assert f(5, pairs, 11520, 2, 256, ws, 0) == 1
    # a workspace with room for 8 partial tiles (pairs of 128 x 256 fp32) caps the split count: 5 tiles * (S - 1) <= 8
    small = 8192 + 8 * 2 * 256 * 128 * 4
    assert f(5, pairs, 11520, 2, 256, small, 1) == 2
    # every split owns at least one k-block: 33 k-blocks in 3 splits of 11 is fine, S is reduced where the last would be empty
    for kb in range(32, 400, 7):
        S = f(2, pairs, kb * 64, 2, 256, ws, 1)
        per = -(-kb // S)
        assert S >= 1 and (S - 1) * per < kb, (kb, S)
