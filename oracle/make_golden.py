"""Generates tests/golden/* by running the UNMODIFIED reference (through oracle/compat) in THIS container.

    python oracle/make_golden.py

Fixtures (small, committed):
  unet3d_state_dict_keys.json     key -> shape of the reference UNet3D (1946 entries)  [SURVEY.md 8b]
  unet_fwd_h{H}_f{F}.pt           reference UNet3D forward output on hallo_b200.synth inputs/weights
                                  (fp32, shipped branch, read-mode reader with synthetic fp16 banks)
                                  + per-block output statistics + input checksums
  refnet_h16_f32.pt               reference UNet2D + write-mode control at latent 16x16, fp32 (see make_refnet_h16)
  process_audio_emb.pt            scripts/inference.py process_audio_emb on a seeded embedding
The weights/inputs are NOT stored: they are regenerated from seeds by hallo_b200/synth.py; the stored
checksums detect generator drift.
"""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from hallo_b200.spec import UNetConfig  # noqa: E402
from hallo_b200.synth import (host_threads, synth_inputs, synth_refnet_inputs, synth_state_dict,  # noqa: E402
                              synth_state_dict_2d)
from oracle import ref_host  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
CASES = [dict(h=8, f=2, seed=42, t=999, ms=(1.0, 0.9, 1.1)),
         dict(h=16, f=3, seed=43, t=499, ms=(1.0, 1.0, 1.0)),
         dict(h=16, f=16, seed=44, t=24, ms=(1.2, 0.8, 1.0)),
         # round 2: the shapes the bench actually times (L0 = 4096 with the 8192-key reference concat) and config-4's
         # level sizes (L = 9216, 2304, 576, 144); run with `--only h64_f2 h64_f16 h96_f2` (f=16 takes ~3 min on 8 cores)
         dict(h=64, f=2, seed=45, t=777, ms=(1.0, 0.7, 1.3)),
         dict(h=64, f=16, seed=46, t=499, ms=(1.1, 0.9, 1.0)),
         dict(h=96, f=2, seed=47, t=261, ms=(0.9, 1.1, 1.0)),
         # fp32 cross-check of the port against the reference at a third timestep and uneven motion scales
         dict(h=8, f=3, seed=7, t=123, ms=(0.7, 1.3, 1.0))]


def checksum(t: torch.Tensor) -> float:
    return float(t.double().abs().sum())


def make_refnet():
    """ReferenceNet fixtures: the unmodified reference UNet2D (hallo/models/unet_2d_condition.py) with the reference's
    own write-mode ReferenceAttentionControl, on hallo_b200.synth weights / inputs at latent 8x8:
      unet2d_state_dict_keys.json   key -> shape (682 entries)
      refnet_h8.pt                  last-up-block features (fp16), the control's bank pairing order, per-bank
                                    statistics and three full banks (one per width + the mid block)"""
    cfg = UNetConfig()
    unet = ref_host.build_reference_unet2d()
    with open(os.path.join(GOLD, "unet2d_state_dict_keys.json"), "w") as f:
        json.dump({k: list(v.shape) for k, v in unet.state_dict().items()}, f, indent=0, sort_keys=True)
    sd = synth_state_dict_2d(cfg)
    unet.load_state_dict(sd, strict=True)
    c = dict(h=8, seed=7)
    inp = synth_refnet_inputs(cfg, c["h"], c["h"], seed=c["seed"])
    out, banks, names = ref_host.run_reference_net(unet, inp)
    keep = ("down_blocks.0.attentions.0", "up_blocks.2.attentions.1", "mid_block.attentions.0")
    fx = dict(case=c, out=out.half(), bank_order=names,
              bank_stats={n: dict(shape=list(b.shape), mean=float(b.mean()), std=float(b.std()), abs_sum=checksum(b))
                          for n, b in zip(names, banks)},
              banks={n: b.half() for n, b in zip(names, banks) if n in keep},
              input_checksums=dict(sample=checksum(inp["sample"]), ehs=checksum(inp["encoder_hidden_states"])),
              weight_checksums={k: checksum(sd[k]) for k in ("conv_in.weight", "mid_block.attentions.0.proj_in.weight")},
              torch_version=torch.__version__)
    path = os.path.join(GOLD, "refnet_h8.pt")
    torch.save(fx, path)
    print("wrote", path, tuple(out.shape), "std", float(out.std()))


def make_refnet_h16():
    """refnet_h16_f32.pt: the same reference ReferenceNet at latent 16x16 (seed 11), kept in fp32 so that the port can be
    held to 2e-5: the bank pairing order, the absolute sums of the output and of every bank, and fixed seeded samples
    (flat indices stored next to the values) of 16384 output elements and 2048 elements per bank; the full tensors
    take 19 MB."""
    cfg = UNetConfig()
    unet = ref_host.build_reference_unet2d()
    unet.load_state_dict(synth_state_dict_2d(cfg), strict=True)
    c = dict(h=16, seed=11)
    inp = synth_refnet_inputs(cfg, c["h"], c["h"], seed=c["seed"])
    out, banks, names = ref_host.run_reference_net(unet, inp)
    g = torch.Generator().manual_seed(0)

    def sample(t, n):
        i = torch.randperm(t.numel(), generator=g)[:n].sort().values
        return dict(index=i.int(), values=t.float().reshape(-1)[i], abs_sum=checksum(t))
    fx = dict(case=c, out=sample(out, 16384), bank_order=names, banks={n: sample(b, 2048) for n, b in zip(names, banks)},
              input_checksums=dict(sample=checksum(inp["sample"])), torch_version=torch.__version__)
    path = os.path.join(GOLD, "refnet_h16_f32.pt")
    torch.save(fx, path)
    print("wrote", path, tuple(out.shape))


def make_process_audio_emb():
    """process_audio_emb.pt: process_audio_emb of the reference's scripts/inference.py (the function alone, executed
    without importing the script's dependencies) on a seeded (37, 12, 8) embedding."""
    import ast
    src = open(os.path.join(ref_host.REFERENCE_ROOT, "scripts", "inference.py")).read()
    fn = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "process_audio_emb")
    ns = {"torch": torch}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "inference.py", "exec"), ns)
    emb = torch.randn(37, 12, 8, generator=torch.Generator().manual_seed(0))
    fx = dict(case=dict(shape=(37, 12, 8), seed=0), input_checksum=checksum(emb), out=ns["process_audio_emb"](emb))
    path = os.path.join(GOLD, "process_audio_emb.pt")
    torch.save(fx, path)
    print("wrote", path, tuple(fx["out"].shape))


def make_audio_proj():
    """audio_proj_f4.pt: the UNMODIFIED reference AudioProjModel (hallo/models/audio_proj.py) on synth weights, 4 frames."""
    from hallo_b200.synth import synth_audio_proj_state_dict
    ref_host._activate()
    from hallo.models.audio_proj import AudioProjModel          # unmodified reference class
    m = AudioProjModel(seq_len=5, blocks=12, channels=768, intermediate_dim=512, output_dim=768, context_tokens=32)
    sd = synth_audio_proj_state_dict()
    m.load_state_dict(sd, strict=True)
    x = torch.randn(1, 4, 5, 12, 768, generator=torch.Generator().manual_seed(13))
    with torch.no_grad():
        out = m(x)
    fx = dict(case=dict(frames=4, seed=13), out=out.half(), input_checksum=checksum(x),
              weight_checksums={k: checksum(v) for k, v in sd.items()}, torch_version=torch.__version__)
    path = os.path.join(GOLD, "audio_proj_f4.pt")
    torch.save(fx, path)
    print("wrote", path, tuple(out.shape), "std", float(out.std()))


def main():
    only = sys.argv[sys.argv.index("--only") + 1:] if "--only" in sys.argv else None
    torch.set_num_threads(host_threads())
    os.makedirs(GOLD, exist_ok=True)
    others = {"refnet": make_refnet, "refnet_h16": make_refnet_h16, "audio_proj": make_audio_proj,
              "process_audio_emb": make_process_audio_emb}
    if only is not None:
        for name in [o for o in only if o in others]:
            others[name]()
        only = [o for o in only if o not in others]
        if not only:
            return
    cfg = UNetConfig()
    unet = ref_host.build_reference_unet()
    keys = {k: list(v.shape) for k, v in unet.state_dict().items()}
    with open(os.path.join(GOLD, "unet3d_state_dict_keys.json"), "w") as f:
        json.dump(keys, f, indent=0, sort_keys=True)
    sd = synth_state_dict(cfg, seed=0)
    unet.load_state_dict(sd, strict=True)
    wsum = {k: checksum(sd[k]) for k in ("conv_in.weight", "mid_block.attentions.0.transformer_blocks.0.attn1.to_q.weight",
                                          "up_blocks.3.motion_modules.2.temporal_transformer.proj_out.weight")}
    for c in CASES:
        if only is not None and f"h{c['h']}_f{c['f']}" not in only:
            continue
        inp = synth_inputs(cfg, c["h"], c["h"], c["f"], seed=c["seed"], timestep=c["t"], motion_scale=c["ms"])
        ref_host.attach_reader(unet, inp["banks"])
        taps = {}
        hooks = []
        for name in ["down_blocks.0", "down_blocks.1", "down_blocks.2", "down_blocks.3", "mid_block",
                     "up_blocks.0", "up_blocks.1", "up_blocks.2", "up_blocks.3"]:
            mod = unet.get_submodule(name)

            def mk(n):
                def hook(m, i, o):
                    t = o[0] if isinstance(o, tuple) else o
                    taps[n] = dict(mean=float(t.mean()), std=float(t.std()), abs_sum=checksum(t))
                return hook
            hooks.append(mod.register_forward_hook(mk(name)))
        out = ref_host.run_reference_unet(unet, inp)
        for hk in hooks:
            hk.remove()
        # full-size outputs are stored in fp16 (rounding 5e-4 relative, far below the 1e-2 tolerance) to keep fixtures small
        fx = dict(case=c, out=(out.clone() if out.numel() < (1 << 18) else out.half()), taps=taps, weight_checksums=wsum,
                  input_checksums=dict(sample=checksum(inp["sample"]), audio=checksum(inp["audio_embedding"]),
                                       bank0=checksum(inp["banks"]["mid_block.attentions.0"].float())),
                  torch_version=torch.__version__)
        path = os.path.join(GOLD, f"unet_fwd_h{c['h']}_f{c['f']}.pt")
        torch.save(fx, path)
        print("wrote", path, tuple(out.shape), "std", float(out.std()))
    if only is None:
        for make in others.values():
            make()


if __name__ == "__main__":
    main()
