"""Architecture description of Hallo's denoising UNet3D: configuration, the exact state-dict
key/shape list, and the structural walk the engine compiles into a kernel plan.

Reference:
  hallo/models/unet_3d.py:121-361          UNet3DConditionModel.__init__
  hallo/models/unet_3d_blocks.py:497-640   CrossAttnDownBlock3D.__init__ (audio width quirk :589)
  hallo/models/unet_3d_blocks.py:940-1090  CrossAttnUpBlock3D.__init__   (audio width quirk :1051)
  configs/inference/default.yaml:46-75     unet_additional_kwargs
  SD-1.5 unet/config.json                  the remaining fields (SURVEY.md 8b)
The state-dict contract (1946 entries for the shipped configuration) is what lets the released
``net.pth`` load strictly (scripts/inference.py:244-250).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

# SD-1.5 unet/config.json fields the 3D UNet consumes + the reference's unet_additional_kwargs.
SD15_UNET_CONFIG = dict(
    sample_size=64, in_channels=4, out_channels=4, center_input_sample=False, flip_sin_to_cos=True,
    freq_shift=0, block_out_channels=(320, 640, 1280, 1280), layers_per_block=2, downsample_padding=1,
    mid_block_scale_factor=1, act_fn="silu", norm_num_groups=32, norm_eps=1e-5, cross_attention_dim=768,
    attention_head_dim=8, use_linear_projection=False,
)
HALLO_UNET_KWARGS = dict(
    use_inflated_groupnorm=True, unet_use_cross_frame_attention=False, unet_use_temporal_attention=False,
    use_motion_module=True, use_audio_module=True, motion_module_resolutions=(1, 2, 4, 8),
    motion_module_mid_block=True, motion_module_decoder_only=False, motion_module_type="Vanilla",
    motion_module_kwargs=dict(num_attention_heads=8, num_transformer_block=1,
                              attention_block_types=("Temporal_Self", "Temporal_Self"),
                              temporal_position_encoding=True, temporal_position_encoding_max_len=32,
                              temporal_attention_dim_div=1),
    audio_attention_dim=768, stack_enable_blocks_name=("up", "down", "mid"),
    stack_enable_blocks_depth=(0, 1, 2, 3),
)


@dataclass
class UNetConfig:
    in_channels: int = 4
    out_channels: int = 4
    block_out_channels: Tuple[int, ...] = (320, 640, 1280, 1280)
    layers_per_block: int = 2
    heads: int = 8                      # `attention_head_dim` is used as the HEAD COUNT (unet_3d.py:233)
    cross_attention_dim: int = 768
    audio_attention_dim: int = 768
    norm_num_groups: int = 32
    norm_eps: float = 1e-5
    pe_max_len: int = 32
    n_motion_frames: int = 2

    @property
    def time_embed_dim(self) -> int:
        return self.block_out_channels[0] * 4

    @staticmethod
    def from_dicts(base: dict, extra: Optional[dict] = None) -> "UNetConfig":
        extra = extra or {}
        mm = extra.get("motion_module_kwargs") or HALLO_UNET_KWARGS["motion_module_kwargs"]
        boc = tuple(base.get("block_out_channels", (320, 640, 1280, 1280)))
        ahd = base.get("attention_head_dim", 8)
        if not isinstance(ahd, int):
            assert len(set(ahd)) == 1, "per-block head counts are not supported"
            ahd = ahd[0]
        return UNetConfig(
            in_channels=base.get("in_channels", 4), out_channels=base.get("out_channels", 4),
            block_out_channels=boc, layers_per_block=base.get("layers_per_block", 2), heads=ahd,
            cross_attention_dim=base.get("cross_attention_dim", 768),
            audio_attention_dim=extra.get("audio_attention_dim", 768),
            norm_num_groups=base.get("norm_num_groups", 32), norm_eps=base.get("norm_eps", 1e-5),
            pe_max_len=mm.get("temporal_position_encoding_max_len", 32))


# ---------------------------------------------------------------------------------------------
# structural walk
# ---------------------------------------------------------------------------------------------
@dataclass
class ResnetSpec:
    name: str
    cin: int
    cout: int

    @property
    def has_shortcut(self) -> bool:
        return self.cin != self.cout


@dataclass
class LayerSpec:
    """One `resnet -> spatial transformer -> audio transformer -> motion module` layer."""
    resnet: ResnetSpec
    attn: Optional[str] = None        # name of the spatial Transformer3DModel
    audio: Optional[str] = None       # name of the audio Transformer3DModel
    audio_inner: int = 0              # Ci (irregular, SURVEY.md Q5)
    motion: Optional[str] = None      # name of the motion module (None or skipped when not executed)
    motion_executed: bool = False     # Q1b: DownBlock3D / UpBlock3D never run theirs on the shipped branch


@dataclass
class BlockSpec:
    name: str
    kind: str                          # "down_x", "down", "mid", "up", "up_x"
    channels: int                      # C of the block's output
    depth: int                         # mask level used by the audio module (unet_3d.py:250,279,338)
    layers: List[LayerSpec] = field(default_factory=list)
    extra_resnet: Optional[ResnetSpec] = None   # mid block: resnets[0] runs before the layer loop
    downsampler: Optional[str] = None
    upsampler: Optional[str] = None
    skip_channels: List[int] = field(default_factory=list)  # per layer, for up blocks


def build_blocks(cfg: UNetConfig) -> List[BlockSpec]:
    boc = cfg.block_out_channels
    nb = len(boc)
    H = cfg.heads
    blocks: List[BlockSpec] = []
    out_ch = boc[0]
    for i in range(nb):
        in_ch, out_ch = out_ch, boc[i]
        final = i == nb - 1
        cross = not final
        b = BlockSpec(name=f"down_blocks.{i}", kind="down_x" if cross else "down", channels=out_ch, depth=i)
        for j in range(cfg.layers_per_block):
            lin = in_ch if j == 0 else out_ch
            rs = ResnetSpec(f"{b.name}.resnets.{j}", lin, out_ch)
            if cross:
                b.layers.append(LayerSpec(rs, attn=f"{b.name}.attentions.{j}", audio=f"{b.name}.audio_modules.{j}",
                                          audio_inner=H * (lin // H), motion=f"{b.name}.motion_modules.{j}",
                                          motion_executed=True))
            else:
                b.layers.append(LayerSpec(rs, motion=f"{b.name}.motion_modules.{j}", motion_executed=False))
        if not final:
            b.downsampler = f"{b.name}.downsamplers.0"
        blocks.append(b)
    C = boc[-1]
    mid = BlockSpec(name="mid_block", kind="mid", channels=C, depth=3)
    mid.extra_resnet = ResnetSpec("mid_block.resnets.0", C, C)
    mid.layers.append(LayerSpec(ResnetSpec("mid_block.resnets.1", C, C), attn="mid_block.attentions.0",
                                audio="mid_block.audio_modules.0", audio_inner=H * (C // H),
                                motion="mid_block.motion_modules.0", motion_executed=True))
    blocks.append(mid)
    rev = list(reversed(boc))
    out_ch = rev[0]
    for i in range(nb):
        prev_out = out_ch
        out_ch = rev[i]
        in_ch = rev[min(i + 1, nb - 1)]
        final = i == nb - 1
        cross = i != 0
        b = BlockSpec(name=f"up_blocks.{i}", kind="up_x" if cross else "up", channels=out_ch, depth=3 - i)
        nl = cfg.layers_per_block + 1
        for j in range(nl):
            skip = in_ch if j == nl - 1 else out_ch
            rin = prev_out if j == 0 else out_ch
            b.skip_channels.append(skip)
            rs = ResnetSpec(f"{b.name}.resnets.{j}", rin + skip, out_ch)
            if cross:
                b.layers.append(LayerSpec(rs, attn=f"{b.name}.attentions.{j}", audio=f"{b.name}.audio_modules.{j}",
                                          audio_inner=H * (in_ch // H), motion=f"{b.name}.motion_modules.{j}",
                                          motion_executed=True))
            else:
                b.layers.append(LayerSpec(rs, motion=f"{b.name}.motion_modules.{j}", motion_executed=False))
        if not final:
            b.upsampler = f"{b.name}.upsamplers.0"
        blocks.append(b)
    return blocks


# ---------------------------------------------------------------------------------------------
# state-dict key / shape list
# ---------------------------------------------------------------------------------------------
def _norm(keys, name, c):
    keys.append((f"{name}.weight", (c,), "norm_w"))
    keys.append((f"{name}.bias", (c,), "norm_b"))


def _lin(keys, name, cout, cin, bias=True, kind="w"):
    keys.append((f"{name}.weight", (cout, cin), kind))
    if bias:
        keys.append((f"{name}.bias", (cout,), "b"))


def _conv(keys, name, cout, cin, k, kind="w"):
    keys.append((f"{name}.weight", (cout, cin, k, k), kind))
    keys.append((f"{name}.bias", (cout,), "b"))


def _resnet(keys, rs: ResnetSpec, temb):
    _norm(keys, f"{rs.name}.norm1", rs.cin)
    _conv(keys, f"{rs.name}.conv1", rs.cout, rs.cin, 3)
    _lin(keys, f"{rs.name}.time_emb_proj", rs.cout, temb)
    _norm(keys, f"{rs.name}.norm2", rs.cout)
    _conv(keys, f"{rs.name}.conv2", rs.cout, rs.cout, 3)
    if rs.has_shortcut:
        _conv(keys, f"{rs.name}.conv_shortcut", rs.cout, rs.cin, 1)


def _attn(keys, name, dim, kv_dim):
    _lin(keys, f"{name}.to_q", dim, dim, bias=False)
    _lin(keys, f"{name}.to_k", dim, kv_dim, bias=False)
    _lin(keys, f"{name}.to_v", dim, kv_dim, bias=False)
    _lin(keys, f"{name}.to_out.0", dim, dim)


def _ff(keys, name, dim):
    _lin(keys, f"{name}.net.0.proj", 8 * dim, dim)
    _lin(keys, f"{name}.net.2", dim, 4 * dim)


def _spatial_tf(keys, name, C, cross_dim):
    _norm(keys, f"{name}.norm", C)
    _conv(keys, f"{name}.proj_in", C, C, 1)
    tb = f"{name}.transformer_blocks.0"
    _attn(keys, f"{tb}.attn1", C, C)
    _norm(keys, f"{tb}.norm1", C)
    _attn(keys, f"{tb}.attn2", C, cross_dim)
    _norm(keys, f"{tb}.norm2", C)
    _ff(keys, f"{tb}.ff", C)
    _norm(keys, f"{tb}.norm3", C)
    _conv(keys, f"{name}.proj_out", C, C, 1)


def _audio_tf(keys, name, C, Ci, audio_dim):
    _norm(keys, f"{name}.norm", C)
    _conv(keys, f"{name}.proj_in", Ci, C, 1)
    tb = f"{name}.transformer_blocks.0"
    for r in ("full", "face", "lip"):
        _conv(keys, f"{tb}.zero_conv_{r}", Ci, Ci, 1, kind="zero_w")
    _attn(keys, f"{tb}.attn1", Ci, Ci)
    _norm(keys, f"{tb}.norm1", Ci)
    for r in range(3):
        _attn(keys, f"{tb}.attn2_{r}", Ci, audio_dim)
    _norm(keys, f"{tb}.norm2", Ci)
    _ff(keys, f"{tb}.ff", Ci)
    _norm(keys, f"{tb}.norm3", Ci)
    _conv(keys, f"{name}.proj_out", C, Ci, 1)


def _motion(keys, name, C, pe_len):
    tt = f"{name}.temporal_transformer"
    _norm(keys, f"{tt}.norm", C)
    _lin(keys, f"{tt}.proj_in", C, C)
    tb = f"{tt}.transformer_blocks.0"
    for a in range(2):
        _attn(keys, f"{tb}.attention_blocks.{a}", C, C)
        keys.append((f"{tb}.attention_blocks.{a}.pos_encoder.pe", (1, pe_len, C), "pe"))
    for a in range(2):
        _norm(keys, f"{tb}.norms.{a}", C)
    _ff(keys, f"{tb}.ff", C)
    _norm(keys, f"{tb}.ff_norm", C)
    _lin(keys, f"{tt}.proj_out", C, C, kind="zero_w")


def param_spec(cfg: UNetConfig) -> List[Tuple[str, Tuple[int, ...], str]]:
    """[(state-dict key, shape, kind)] in the reference's registration order.  kind in
    {w, zero_w, b, norm_w, norm_b, pe}; zero_w marks tensors the reference zero-initialises
    (attention.py:691-701, motion_module.py:169-172)."""
    keys = _stem_and_blocks(cfg, build_blocks(cfg))
    c0 = cfg.block_out_channels[0]
    _norm(keys, "conv_norm_out", c0)
    _conv(keys, "conv_out", cfg.out_channels, c0, 3)
    return keys


def _stem_and_blocks(cfg: UNetConfig, blocks: List[BlockSpec]) -> List[Tuple[str, Tuple[int, ...], str]]:
    keys: List[Tuple[str, Tuple[int, ...], str]] = []
    temb = cfg.time_embed_dim
    c0 = cfg.block_out_channels[0]
    _conv(keys, "conv_in", c0, cfg.in_channels, 3)
    _lin(keys, "time_embedding.linear_1", temb, c0)
    _lin(keys, "time_embedding.linear_2", temb, temb)
    for b in blocks:
        # registration order in the reference: attentions, resnets, audio_modules, motion_modules, samplers
        # (key ORDER is irrelevant for strict loading; we keep a readable order).
        if b.extra_resnet is not None:
            _resnet(keys, b.extra_resnet, temb)
        for l in b.layers:
            _resnet(keys, l.resnet, temb)
            if l.attn:
                _spatial_tf(keys, l.attn, b.channels, cfg.cross_attention_dim)
            if l.audio:
                _audio_tf(keys, l.audio, b.channels, l.audio_inner, cfg.audio_attention_dim)
            if l.motion:
                _motion(keys, l.motion, b.channels, cfg.pe_max_len)
        if b.downsampler:
            _conv(keys, f"{b.downsampler}.conv", b.channels, b.channels, 3)
        if b.upsampler:
            _conv(keys, f"{b.upsampler}.conv", b.channels, b.channels, 3)
    return keys


def reader_bank_order(cfg: UNetConfig) -> List[Tuple[str, int]]:
    """Spatial transformer blocks in the order ReferenceAttentionControl pairs readers with writers:
    module DFS order (down_blocks, up_blocks, mid_block -- mid is assigned last, unet_3d.py:203-205,258)
    stably sorted by -norm1 width (mutual_self_attention.py:371-385, 404-453).  -> [(attn name, C)]"""
    blocks = build_blocks(cfg)
    downs = [b for b in blocks if b.name.startswith("down_blocks")]
    ups = [b for b in blocks if b.name.startswith("up_blocks")]
    mids = [b for b in blocks if b.name == "mid_block"]
    order = []
    for b in downs + ups + mids:
        for l in b.layers:
            if l.attn:
                order.append((l.attn, b.channels))
    return sorted(order, key=lambda x: -x[1])


def sinusoid_pe(max_len: int, d_model: int):
    """PositionalEncoding buffer (hallo/models/motion_module.py:435-445)."""
    import torch
    position = torch.arange(max_len).unsqueeze(1)
    div_term = torch.exp(torch.arange(0, d_model, 2) * (-math.log(10000.0) / d_model))
    pe = torch.zeros(1, max_len, d_model)
    pe[0, :, 0::2] = torch.sin(position * div_term)
    pe[0, :, 1::2] = torch.cos(position * div_term)
    return pe


# ---------------------------------------------------------------------------------------------
# ReferenceNet (hallo/models/unet_2d_condition.py: the SD-1.5 UNet2D that produces the K/V banks)
# ---------------------------------------------------------------------------------------------
def build_blocks_2d(cfg: UNetConfig) -> List[BlockSpec]:
    """The UNet2D's structural walk: the 3D walk with the audio and motion modules removed (same names)."""
    blocks = build_blocks(cfg)
    for b in blocks:
        b.layers = [LayerSpec(l.resnet, attn=l.attn) for l in b.layers]
    return blocks


def param_spec_2d(cfg: UNetConfig) -> List[Tuple[str, Tuple[int, ...], str]]:
    """State-dict keys of the reference's UNet2DConditionModel built from the SD-1.5 config: the resnet / spatial
    transformer / sampler subset of the 3D walk (same names).  The reference deletes conv_norm_out / conv_act / conv_out
    (the ReferenceNet returns after the up blocks), so they are not part of the contract: 682 entries, verified against
    the instantiated reference class (tests/golden/unet2d_state_dict_keys.json)."""
    return _stem_and_blocks(cfg, build_blocks_2d(cfg))
