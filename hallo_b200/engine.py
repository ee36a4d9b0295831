"""Kernel-plan executor for the denoising UNet3D (the device hot path).

The reference walks an nn.Module tree and issues ~2.3k library kernels per forward
(hallo/models/unet_3d.py:510-715 and everything below it).  Here the same arithmetic is a flat,
pre-planned sequence of hand-written sm_100a kernels (hallo_b200/csrc) over channels-last token
matrices, with all weights pre-packed once and all step-invariant work hoisted out of the 40-step loop:

  per model load : weight packing (fused QKV, interleaved GEGLU, [Cout][tap][Cin] convs, ...)
  per window     : ReferenceNet-bank K/V, image-token K/V, audio-token K/V, motion-frame GroupNorm
                   inputs, masks, mask_cond_fea, motion_scale-folded zero-conv weights
  per step       : the kernels in `_forward()` -- captured once into a CUDA graph and replayed.

`_forward()` is `_walk()` (time embedding, conv_in, down / mid / up blocks) plus the conv_out head.  The ReferenceNet
(refnet.py) runs the same `_walk()`: its block list has no audio / motion modules and its window no reference K/V.

Layout: every activation is a token matrix [rows, C]; rows are ordered (cfg_half, frame, pixel) --
i.e. the reference's `(b f) (h w) c` -- so NCHW<->NLC permutes, `rearrange`s and `torch.cat`s of the
reference disappear (channel concats become two-source reads, frame concats become row offsets).

Multi-GPU (SURVEY.md 8e): a rank owns a contiguous FRAME group of BOTH CFG halves, so everything except the motion
modules -- and the CFG combine + DDIM update -- is rank-local and perfectly balanced.  The temporal attention mixes
all frames of a pixel; around each motion module the ranks swap frame <-> pixel ownership (`_motion_px`): the
GroupNorm that feeds the module stores its rows straight into the pixel owner's buffer over NVLink, the module runs
on (all frames x L/R pixels) with a purely local temporal attention and no replicated motion-frame rows, and the
proj_out GEMM's epilogue stores every row back into the frame owner's buffer.  Two flag barriers per module replace
the collectives (hallo_b200/peer.py); an NCCL all-to-all variant of the same exchange is kept for A/B runs.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
import os
from typing import Dict, Optional, Sequence, Tuple

import torch

from . import ops
from .spec import BlockSpec, LayerSpec, ResnetSpec, UNetConfig, build_blocks, reader_bank_order


@dataclass
class Shard:
    """Which (cfg half, frame) rows this rank owns.  halves: subset of (0, 1); frames: global frame ids."""
    halves: Tuple[int, ...] = (0, 1)
    frames: Tuple[int, ...] = tuple(range(16))
    group: Optional[object] = None          # torch.distributed group of the ranks sharing the window
    group_size: int = 1
    rank_in_group: int = 0
    exchange: str = "peer"                  # "peer": kernels store into peer-mapped buffers; "nccl": all_to_all_single
    emulate_group: int = 1                  # PROFILING AID ONLY (bench.py --emulate-shard): single GPU running ONE rank's
                                            # kernel shapes of an R-rank job; the peers' rows are stand-in copies of the
                                            # local ones, so the numbers it produces are not a valid denoising result


class PackedWeights:
    """Device-resident, kernel-ready copies of the state dict (packed once per model load)."""
    build_blocks = staticmethod(build_blocks)     # the layers to pack and run; refnet.ReferenceNetWeights: the UNet2D's

    def __init__(self, sd: Dict[str, torch.Tensor], cfg: UNetConfig, device, dtype):
        self.cfg = cfg
        self.dtype = dtype
        self.device = device
        self.t: Dict[str, torch.Tensor] = {}
        blocks = self.build_blocks(cfg)
        self.blocks = blocks

        def dev(x):
            return x.detach().to(device=device, dtype=dtype).contiguous()

        def put(name, x):
            self.t[name] = dev(x)

        def lin(name, bias=True):
            put(f"{name}.w", sd[f"{name}.weight"].reshape(sd[f"{name}.weight"].shape[0], -1))
            if bias and f"{name}.bias" in sd:
                put(f"{name}.b", sd[f"{name}.bias"])

        def norm(name):
            put(f"{name}.w", sd[f"{name}.weight"])
            put(f"{name}.b", sd[f"{name}.bias"])

        def conv3(name):
            put(f"{name}.w", ops.pack_conv3x3_weight(sd[f"{name}.weight"]))
            put(f"{name}.b", sd[f"{name}.bias"])

        def transformer(name, norms, self_attns):
            """The part the spatial, audio and motion transformers share: GroupNorm, proj_in / proj_out, the block's
            LayerNorms, each self-attention's fused QKV and to_out, the GEGLU feed-forward."""
            tb = f"{name}.transformer_blocks.0"
            norm(f"{name}.norm"); lin(f"{name}.proj_in"); lin(f"{name}.proj_out")
            for k in norms:
                norm(f"{tb}.{k}")
            for a in self_attns:
                put(f"{tb}.{a}.qkv", torch.cat([sd[f"{tb}.{a}.to_{p}.weight"] for p in "qkv"], 0))
                lin(f"{tb}.{a}.to_out.0")
            wi, bi = ops.pack_geglu_weight(sd[f"{tb}.ff.net.0.proj.weight"], sd[f"{tb}.ff.net.0.proj.bias"])
            put(f"{tb}.ff.w1", wi)
            put(f"{tb}.ff.b1", bi)
            lin(f"{tb}.ff.net.2")
            return tb

        # stem / head
        w_in = sd["conv_in.weight"]                                  # [C0, Cl, 3, 3] -> [C0, 64], k = tap*Cl + c
        c0, cl = w_in.shape[0], w_in.shape[1]
        if 9 * cl > 64:
            raise NotImplementedError(f"conv_in with {cl} input channels (use_landmark=True variant) is not implemented: "
                                      "the im2col stem packs 9*in_channels <= 64 columns (Hallo ships in_channels=4)")
        wi = torch.zeros(c0, 64, dtype=w_in.dtype, device=w_in.device)
        wi[:, :9 * cl] = w_in.permute(0, 2, 3, 1).reshape(c0, 9 * cl)
        put("conv_in.w", wi)
        put("conv_in.b", sd["conv_in.bias"])
        lin("time_embedding.linear_1")
        lin("time_embedding.linear_2")
        if "conv_out.weight" in sd:                                    # the UNet2D ends at the last up block
            norm("conv_norm_out")
            w_out = ops.pack_conv3x3_weight(sd["conv_out.weight"])       # [Cl, 9*C0] -> padded to 8 rows
            wo = torch.zeros(8, w_out.shape[1], dtype=w_out.dtype, device=w_out.device)
            wo[:w_out.shape[0]] = w_out
            bo = torch.zeros(8, dtype=w_out.dtype, device=w_out.device)
            bo[:w_out.shape[0]] = sd["conv_out.bias"]
            put("conv_out.w", wo)
            put("conv_out.b", bo)

        temb_w, temb_b = [], []
        self.temb_off: Dict[str, int] = {}
        off = 0

        def resnet(rs: ResnetSpec):
            nonlocal off
            norm(f"{rs.name}.norm1")
            conv3(f"{rs.name}.conv1")
            norm(f"{rs.name}.norm2")
            conv3(f"{rs.name}.conv2")
            if rs.has_shortcut:
                lin(f"{rs.name}.conv_shortcut")
            temb_w.append(sd[f"{rs.name}.time_emb_proj.weight"])
            temb_b.append(sd[f"{rs.name}.time_emb_proj.bias"])
            self.temb_off[rs.name] = off
            off += rs.cout

        for b in blocks:
            if b.extra_resnet is not None:
                resnet(b.extra_resnet)
            for l in b.layers:
                resnet(l.resnet)
                if l.attn:
                    tb = transformer(l.attn, ("norm1", "norm2", "norm3"), ("attn1",))
                    put(f"{tb}.attn1.kv", torch.cat([sd[f"{tb}.attn1.to_k.weight"], sd[f"{tb}.attn1.to_v.weight"]], 0))
                    put(f"{tb}.attn2.q", sd[f"{tb}.attn2.to_q.weight"])
                    put(f"{tb}.attn2.kv", torch.cat([sd[f"{tb}.attn2.to_k.weight"], sd[f"{tb}.attn2.to_v.weight"]], 0))
                    lin(f"{tb}.attn2.to_out.0")
                if l.audio:
                    tb = transformer(l.audio, ("norm1", "norm2", "norm3"), ("attn1",))
                    put(f"{tb}.attn2.q3", torch.cat([sd[f"{tb}.attn2_{r}.to_q.weight"] for r in range(3)], 0))
                    put(f"{tb}.attn2.kv6", torch.cat([torch.cat([sd[f"{tb}.attn2_{r}.to_k.weight"],
                                                                 sd[f"{tb}.attn2_{r}.to_v.weight"]], 0)
                                                      for r in range(3)], 0))
                    for r in range(3):
                        lin(f"{tb}.attn2_{r}.to_out.0")
                    # zero convs stay in fp32 on the host side of the pack: folded with motion_scale per window
                    self.t[f"{tb}.zero.w"] = torch.stack(
                        [sd[f"{tb}.zero_conv_{r}.weight"].reshape(l.audio_inner, l.audio_inner).float()
                         for r in ("full", "face", "lip")], 0).to(device)
                    self.t[f"{tb}.zero.b"] = torch.stack([sd[f"{tb}.zero_conv_{r}.bias"].float()
                                                          for r in ("full", "face", "lip")], 0).to(device)
                if l.motion_executed:
                    tb = transformer(f"{l.motion}.temporal_transformer", ("norms.0", "norms.1", "ff_norm"),
                                     ("attention_blocks.0", "attention_blocks.1"))
                    for a in range(2):
                        self.t[f"{tb}.attention_blocks.{a}.pe"] = \
                            sd[f"{tb}.attention_blocks.{a}.pos_encoder.pe"][0].float().to(device).contiguous()
            if b.downsampler:
                conv3(f"{b.downsampler}.conv")
            if b.upsampler:
                conv3(f"{b.upsampler}.conv")
        put("temb_all.w", torch.cat(temb_w, 0))
        put("temb_all.b", torch.cat(temb_b, 0))
        self.temb_total = off

    def __getitem__(self, k):
        return self.t[k]

    def get(self, k):
        return self.t.get(k)


class DenoiseEngine:
    """Executes UNet3D forward (+ optional CFG/DDIM step) for one rank's shard of a window."""

    def __init__(self, weights: PackedWeights, h: int, w: int, n_frames: int, shard: Optional[Shard] = None):
        self.W = weights
        self.cfg = weights.cfg
        self.dtype = weights.dtype
        self.dev = weights.device
        self.h, self.w, self.f = h, w, n_frames
        self.shard = shard or Shard(frames=tuple(range(n_frames)))
        self.nb = len(self.shard.halves)
        self.fl = len(self.shard.frames)
        self.nm = self.cfg.n_motion_frames
        self.B = self.nb * self.fl                      # local (cfg half, frame) rows
        self._bufs: Dict[Tuple, torch.Tensor] = {}
        self.window: Dict[str, torch.Tensor] = {}
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        nblk = len(self.cfg.block_out_channels)
        self.level_hw = [(h >> i, w >> i) for i in range(nblk)]
        # scheduler state on the device
        self.step_idx = torch.zeros(1, dtype=torch.int32, device=self.dev)
        # fixed-capacity, fixed-address tables: a captured graph holds these pointers, so schedules are copied IN PLACE
        self.MAX_STEPS = 1024
        self.t_table = torch.zeros(self.MAX_STEPS, dtype=torch.float32, device=self.dev)
        self.coef = torch.zeros(self.MAX_STEPS, 4, dtype=torch.float32, device=self.dev)
        self.n_steps = 1
        self.guidance = 1.0
        self._captured_with = None                       # (n_steps, guidance) baked into the graph as kernel arguments
        assert self.nm + n_frames <= self.cfg.pe_max_len, "temporal length exceeds the positional-encoding table"
        self.latents = torch.zeros(1, self.cfg.in_channels, self.fl, h, w, dtype=torch.float32, device=self.dev)
        self.model_out: Optional[torch.Tensor] = None
        self.sample: Optional[torch.Tensor] = None      # per-half fp32 sample for the plain forward() API path
        # frame-sharded window: R ranks (or an emulated R on one GPU) swap frame <-> pixel ownership around motion modules
        self.R = max(self.shard.group_size, self.shard.emulate_group)
        self.px = self.R > 1
        self.arena = None
        if self.px:
            assert self.nb == 2, "a frame shard holds both CFG halves (the CFG combine stays rank-local)"
            assert n_frames % self.R == 0 and self.fl == n_frames // self.R
            self._init_px()

    # ------------------------------------------------------------------ frame <-> pixel exchange set-up
    def _motion_modules(self):
        """(module name, attention name, level, channels) of the executed motion modules, in execution order."""
        out = []
        for b in self.W.blocks:
            lv = self._block_level(b.name)
            for l in b.layers:
                if l.motion and l.motion_executed:
                    out.append((l.motion, l.attn, lv, b.channels))
        return out

    def _init_px(self):
        sh, esz = self.shard, torch.empty(0, dtype=self.dtype).element_size()
        nb, nm, fl, f, R = self.nb, self.nm, self.fl, self.f, self.R
        regions = []
        recv = 0
        for name, _, lv, C in self._motion_modules():
            L = self.L(lv)
            if L % R != 0:
                raise ValueError(f"frame-sharded window: {L} tokens of level {lv} do not split over {R} ranks")
            regions.append((f"x18.{name}", nb * (nm + f) * (L // R) * C * esz))
            recv = max(recv, nb * fl * L * C * esz)
        regions.append(("recv", recv))
        self.me = sh.rank_in_group
        if sh.group_size > 1 and sh.exchange == "peer":
            from .peer import PeerArena
            try:
                # PeerArena agrees on success across the ranks: either every rank gets a mapped arena or every rank raises
                self.arena = PeerArena(regions, sh.group, sh.rank_in_group, sh.group_size, self.dev)
            except RuntimeError as e:                    # e.g. CUDA IPC not permitted between these processes
                self.arena = None
                sh.exchange = "nccl"
                import sys
                print(f"# hallo_b200: {e}; every rank uses the NCCL all-to-all exchange instead", file=sys.stderr)
        self._px_regions = dict(regions)

    def _x18(self, name: str, rows: int, C: int) -> torch.Tensor:
        if self.arena is not None:
            return self.arena.local(f"x18.{name}", (rows, C), self.dtype)
        return self.buf(f"x18.{name}", rows, C)

    # ------------------------------------------------------------------ buffers
    def buf(self, tag: str, rows: int, cols: int, dtype=None) -> torch.Tensor:
        key = (tag, rows, cols, dtype or self.dtype)
        t = self._bufs.get(key)
        if t is None:
            t = torch.empty(rows, cols, device=self.dev, dtype=dtype or self.dtype)
            self._bufs[key] = t
        return t

    def _wset(self, key: str, t: torch.Tensor) -> torch.Tensor:
        """Window constants live in persistent buffers (updated in place) so a captured graph stays valid."""
        cur = self.window.get(key)
        if isinstance(cur, torch.Tensor) and cur.shape == t.shape and cur.dtype == t.dtype:
            cur.copy_(t)
            return cur
        self.window[key] = t.clone() if t._base is not None or not t.is_contiguous() else t
        if isinstance(cur, torch.Tensor):
            self.graph = None            # shapes changed: any captured graph is stale
        return self.window[key]

    def _gn_ws(self) -> torch.Tensor:
        """GroupNorm statistics workspace: 2 floats per (frame row, group or channel) -- sized from this engine's row
        count and the widest (concatenated) channel count, not a constant."""
        rows = max(self.nb * (self.nm + self.fl), 2 * (1 + self.nm))
        cmax = 2 * max(self.cfg.block_out_channels)
        return self.buf("gn_ws", 1, ops.gn_workspace_floats(rows, self.h * self.w, self.cfg.norm_num_groups, cmax),
                        torch.float32)

    def L(self, level: int) -> int:
        hh, ww = self.level_hw[level]
        return hh * ww

    # ------------------------------------------------------------------ per-window constants
    def _block_level(self, name: str) -> int:
        nblk = len(self.cfg.block_out_channels)
        if name.startswith("mid_block"):
            return nblk - 1
        i = int(name.split(".")[1])
        return i if name.startswith("down_blocks") else nblk - 1 - i

    @torch.no_grad()
    def begin_window(self, *, encoder_hidden_states, audio_embedding, mask_cond_fea, full_mask, face_mask, lip_mask,
                     motion_scale, banks: Dict[str, torch.Tensor], local_frames: bool = False):
        """Hoists everything that does not depend on (latents, timestep) -- SURVEY.md 8a "step-invariant work".
        Inputs use the reference's shapes (full CFG batch, all frames) and this rank slices its shard; with
        local_frames=True the per-frame tensors (audio, mask_cond_fea, masks) already hold only this rank's frames
        (rows ordered (half, local frame)) -- a sharded caller then moves 1/R of them to the device."""
        W, cfg, sh = self.W, self.cfg, self.shard
        dt, dev = self.dtype, self.dev
        halves, frames = list(sh.halves), list(sh.frames)
        f, fl, nb, nm, H = self.f, self.fl, self.nb, self.nm, cfg.heads
        win = self.window
        trace = os.environ.get("HALLO_B200_TRACE_WINDOW")          # debugging aid: host wall time per section (synchronised)
        if trace:
            import time
            torch.cuda.synchronize()
            _t = [time.perf_counter()]

            def mark(what):
                torch.cuda.synchronize()
                _t.append(time.perf_counter())
                print(f"# begin_window {what}: {(_t[-1] - _t[-2]) * 1e3:.2f} ms", flush=True)
        else:
            def mark(what):
                pass
        fr_idx = torch.tensor(frames, device=dev)
        # global (b f) row ids of the local rows, in local order
        rows = [b * f + g for b in halves for g in frames]
        win["row_ids"] = rows
        # reference tiles CFG halves over the batch (Q9): row n attends to ref[n % 2]; uncond rows: none (Q3)
        ridx = [(-1 if n < f else (n % 2)) for n in rows]
        self._wset("ref_index", torch.tensor(ridx, dtype=torch.int32, device=dev))
        # temporal positions: motion frames 0..nm-1, then nm + global frame id
        self._wset("pe_index", torch.tensor(list(range(nm)) + [nm + g for g in frames], dtype=torch.int32, device=dev))
        self._wset("pe_index_all", torch.arange(nm + f, dtype=torch.int32, device=dev))     # pixel-sharded motion path

        ehs = encoder_hidden_states.to(dev, dt)[halves]                       # [nb, 4, 768]
        if local_frames:
            assert nb == 2 and audio_embedding.shape[1] == fl and mask_cond_fea.shape[2] == fl
            fr_idx = torch.arange(fl, device=dev)
        aud = audio_embedding.to(dev, dt)[halves][:, fr_idx]                  # [nb, fl, 32, 768]
        aud2 = aud.reshape(nb * fl * aud.shape[2], aud.shape[3]).contiguous()
        ehs2 = ehs.reshape(nb * ehs.shape[1], ehs.shape[2]).contiguous()
        win["n_img_tokens"] = ehs.shape[1]
        win["kvimg_frame_div"] = fl                    # the local rows of CFG half b read image K/V rows of batch b
        win["n_aud_tokens"] = aud.shape[2]
        mcf = mask_cond_fea.to(dev, dt)[halves][:, :, fr_idx]                 # [nb, C0, fl, h, w]
        self._wset("mask_cond", mcf.permute(0, 2, 3, 4, 1).reshape(-1, mcf.shape[1]).contiguous())
        rid = torch.arange(nb * fl, device=dev) if local_frames else torch.tensor(rows, device=dev)
        for nme, m in (("full", full_mask), ("face", face_mask), ("lip", lip_mask)):
            for lv, t in enumerate(m):
                self._wset(f"mask.{nme}.{lv}", t.to(dev, dt)[rid].reshape(-1).contiguous())
        ms = [float(x) for x in motion_scale] if motion_scale is not None else [1.0, 1.0, 1.0]
        mark("per-frame tensors (audio, mask_cond_fea, masks)")

        for b in W.blocks:
            lv = self._block_level(b.name)
            L = self.L(lv)
            for l in b.layers:
                if l.attn:
                    tb = f"{l.attn}.transformer_blocks.0"
                    C = b.channels
                    bank = banks[l.attn].to(dev, torch.float16).to(dt)          # update() casts to fp16 (Q4)
                    bank = bank.reshape(2, 1 + nm, L, C)
                    refs = bank[:, 0].reshape(2 * L, C).contiguous()           # both CFG halves' ref tokens
                    kv = self.buf(f"{l.attn}.kvref", 2 * L, 2 * C)
                    ops.gemm(refs, W[f"{tb}.attn1.kv"], kv)
                    win[f"{l.attn}.kvref"] = kv
                    kvi = self.buf(f"{l.attn}.kvimg", ehs2.shape[0], 2 * C)
                    ops.gemm(ehs2, W[f"{tb}.attn2.kv"], kvi)
                    win[f"{l.attn}.kvimg"] = kvi
                    # motion-frame features of the local halves, token layout [nb*nm*L, C]
                    self._wset(f"{l.attn}.motion", bank[halves][:, 1:].reshape(nb * nm * L, C).contiguous())
                if l.audio:
                    tb = f"{l.audio}.transformer_blocks.0"
                    Ci = l.audio_inner
                    kva = self.buf(f"{l.audio}.kvaud", aud2.shape[0], 6 * Ci)
                    ops.gemm(aud2, W[f"{tb}.attn2.kv6"], kva)
                    win[f"{l.audio}.kvaud"] = kva
                    zw, zb = W[f"{tb}.zero.w"], W[f"{tb}.zero.b"]
                    self._wset(f"{l.audio}.zero.w", torch.cat([ms[r] * zw[r] for r in range(3)], 1).to(dt).contiguous())
                    self._wset(f"{l.audio}.zero.b", sum(ms[r] * zb[r] for r in range(3)).to(dt).contiguous())
                if l.motion and l.motion_executed:
                    # GroupNorm of the motion frames is step-invariant: normalise once into frames [0, nm)
                    tt = f"{l.motion}.temporal_transformer"
                    C = b.channels
                    ws = self._gn_ws()
                    if self.px:
                        # pixel-sharded module: this rank keeps its pixel slice of ALL frames; the motion frames'
                        # GroupNorm needs whole frames, so it is computed in full once per window and sliced
                        Lg, F18 = L // self.R, nm + f
                        gnm = self.buf("mm.gnm", nb * nm * L, C)
                        ops.groupnorm(win[f"{l.attn}.motion"], W[f"{tt}.norm.w"], W[f"{tt}.norm.b"], gnm, ws,
                                      n_frames=nb * nm, hw=L, groups=cfg.norm_num_groups, eps=1e-6)
                        x18 = self._x18(l.motion, nb * F18 * Lg, C)
                        x18.view(nb, F18, Lg, C)[:, :nm].copy_(
                            gnm.view(nb, nm, L, C)[:, :, self.me * Lg:(self.me + 1) * Lg])
                    else:
                        gn18 = self.buf(f"{l.motion}.gn18", nb * (nm + fl) * L, C)
                        ops.groupnorm(win[f"{l.attn}.motion"], W[f"{tt}.norm.w"], W[f"{tt}.norm.b"], gn18, ws,
                                      n_frames=nb * nm, hw=L, groups=cfg.norm_num_groups, eps=1e-6,
                                      fpb_in=nm, fpb_out=nm + fl, frame_off=0)
            mark(f"block {b.name}")
        if self.arena is not None:
            # ranks meet once per window on the device (flag barrier, stream-ordered, no host round trip): a peer's first
            # scatter store of the new window cannot overtake this rank's window set-up
            self.arena.barrier()
        torch.cuda.current_stream().synchronize()

    def set_schedule(self, timesteps: Sequence[int], coef: torch.Tensor, guidance: float):
        """Per-window schedule.  The tables keep their device addresses (a captured graph reads them); the step count
        and the guidance scale are kernel ARGUMENTS of the captured launches, so changing them drops the graph."""
        n = len(timesteps)
        if n > self.MAX_STEPS:
            raise ValueError(f"{n} inference steps exceed the engine's schedule capacity ({self.MAX_STEPS})")
        self.n_steps = n
        self.t_table[:n].copy_(torch.tensor([float(t) for t in timesteps], dtype=torch.float32))
        self.coef[:n].copy_(coef.to(torch.float32).reshape(n, 4))
        self.guidance = float(guidance)
        if self.graph is not None and self._captured_with != (self.n_steps, self.guidance):
            self.graph = None
        self.step_idx.zero_()

    def set_timestep(self, t: float):
        """Single-forward API path (UNet3DConditionModel.forward): slot 0 of the table, in place."""
        self.t_table[:1].fill_(float(t))

    # ------------------------------------------------------------------ modules
    def _gn(self, x1, name, out, n_frames, hw, eps, silu, x2=None, **kw):
        ws = self._gn_ws()
        return ops.groupnorm(x1, self.W[f"{name}.w"], self.W[f"{name}.b"], out, ws, n_frames=n_frames, hw=hw,
                             groups=self.cfg.norm_num_groups, eps=eps, silu=silu, x2=x2, **kw)

    def _ln(self, x, name, tag, **kw):
        out = self.buf(tag, x.shape[0], x.shape[1])
        return ops.layernorm(x, self.W[f"{name}.w"], self.W[f"{name}.b"], out, **kw)

    def _resnet(self, rs: ResnetSpec, x1, x2, level: int, out_tag: str):
        W, B = self.W, self.B
        hh, ww = self.level_hw[level]
        L = hh * ww
        M = B * L
        cin, cout = rs.cin, rs.cout
        t1 = self.buf("rs.gn1", M, cin)
        self._gn(x1, f"{rs.name}.norm1", t1, B, L, self.cfg.norm_eps, True, x2=x2)
        t2 = self.buf("rs.c1", M, cout)
        off = W.temb_off[rs.name]
        ops.conv3x3(t1.view(B, hh, ww, cin), W[f"{rs.name}.conv1.w"], t2, bias=W[f"{rs.name}.conv1.b"],
                    group_bias=self.temb_all[:, off:off + cout], rows_per_group=self.fl * L)
        t3 = self.buf("rs.gn2", M, cout)
        self._gn(t2, f"{rs.name}.norm2", t3, B, L, self.cfg.norm_eps, True)
        if rs.has_shortcut:
            sc = self.buf("rs.sc", M, cout)
            ops.gemm(x1, W[f"{rs.name}.conv_shortcut.w"], sc, bias=W[f"{rs.name}.conv_shortcut.b"], a2=x2)
        else:
            assert x2 is None
            sc = x1
        out = self.buf(out_tag, M, cout)
        ops.conv3x3(t3.view(B, hh, ww, cout), W[f"{rs.name}.conv2.w"], out, bias=W[f"{rs.name}.conv2.b"], residual=sc)
        return out

    def _ff(self, x, name, norm_name, tag):
        W = self.W
        n = self._ln(x, norm_name, "ln")
        M, C = x.shape
        g = self.buf("ff.mid", M, 4 * C)
        ops.gemm(n, W[f"{name}.w1"], g, bias=W[f"{name}.b1"], geglu=True)
        out = self.buf(tag, M, C)
        ops.gemm(g, W[f"{name}.net.2.w"], out, bias=W[f"{name}.net.2.b"], residual=x)
        return out

    def _norm1_tag(self, name: str) -> str:
        """Buffer of the spatial transformer's norm1 output (the ReferenceNet banks it)."""
        return "ln"

    def _spatial(self, name: str, x, level: int, C: int, out_tag: str):
        """Transformer3DModel + BasicTransformerBlock: self-attention (+ the window's reference K/V where it has them),
        image cross-attention on the window's image K/V, GEGLU feed-forward."""
        W, B, win, H = self.W, self.B, self.window, self.cfg.heads
        L = self.L(level)
        M = B * L
        tb = f"{name}.transformer_blocks.0"
        t = self.buf("tf.gn", M, C)
        self._gn(x, f"{name}.norm", t, B, L, 1e-6, False)
        h = self.buf("tf.h0", M, C)
        ops.gemm(t, W[f"{name}.proj_in.w"], h, bias=W[f"{name}.proj_in.b"])
        n1 = self._ln(h, f"{tb}.norm1", self._norm1_tag(name))
        qkv = self.buf("tf.qkv", M, 3 * C)
        ops.gemm(n1, W[f"{tb}.attn1.qkv"], qkv)
        a = self.buf("tf.attn", M, C)
        kvref = win.get(f"{name}.kvref")
        ref = {} if kvref is None else dict(kref=kvref[:, :C], vref=kvref[:, C:], ref_index=win["ref_index"])
        ops.attention(qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:], a, heads=H, L=L, **ref)
        h1 = self.buf("tf.h1", M, C)
        ops.gemm(a, W[f"{tb}.attn1.to_out.0.w"], h1, bias=W[f"{tb}.attn1.to_out.0.b"], residual=h)
        n2 = self._ln(h1, f"{tb}.norm2", "ln")
        q2 = self.buf("tf.q2", M, C)
        ops.gemm(n2, W[f"{tb}.attn2.q"], q2)
        kvi = win[f"{name}.kvimg"]
        a2 = self.buf("tf.attn", M, C)
        ops.cross_attention(q2, kvi[:, :C], kvi[:, C:], a2, frames=B, tokens=L, heads=H, head_dim=C // H,
                            n_keys=win["n_img_tokens"], kv_frame_div=win["kvimg_frame_div"])
        h2 = self.buf("tf.h2", M, C)
        ops.gemm(a2, W[f"{tb}.attn2.to_out.0.w"], h2, bias=W[f"{tb}.attn2.to_out.0.b"], residual=h1)
        h3 = self._ff(h2, f"{tb}.ff", f"{tb}.norm3", "tf.h3")
        out = self.buf(out_tag, M, C)
        ops.gemm(h3, W[f"{name}.proj_out.w"], out, bias=W[f"{name}.proj_out.b"], residual=x)
        return out

    def _audio(self, name: str, x, level: int, C: int, Ci: int, depth: int, out_tag: str):
        W, B, win, H = self.W, self.B, self.window, self.cfg.heads
        L = self.L(level)
        M = B * L
        tb = f"{name}.transformer_blocks.0"
        t = self.buf("tf.gn", M, C)
        self._gn(x, f"{name}.norm", t, B, L, 1e-6, False)
        h = self.buf("au.h0", M, Ci)
        ops.gemm(t, W[f"{name}.proj_in.w"], h, bias=W[f"{name}.proj_in.b"])
        n1 = self._ln(h, f"{tb}.norm1", "ln")
        qkv = self.buf("tf.qkv", M, 3 * Ci)
        ops.gemm(n1, W[f"{tb}.attn1.qkv"], qkv)
        a = self.buf("tf.attn", M, Ci)
        ops.attention(qkv[:, :Ci], qkv[:, Ci:2 * Ci], qkv[:, 2 * Ci:], a, heads=H, L=L)
        h1 = self.buf("au.h1", M, Ci)
        ops.gemm(a, W[f"{tb}.attn1.to_out.0.w"], h1, bias=W[f"{tb}.attn1.to_out.0.b"], residual=h)
        n2 = self._ln(h1, f"{tb}.norm2", "ln")
        q3 = self.buf("au.q3", M, 3 * Ci)
        ops.gemm(n2, W[f"{tb}.attn2.q3"], q3)
        kva = win[f"{name}.kvaud"]
        a3 = self.buf("au.a3", M, 3 * Ci)
        ops.cross_attention(q3, kva[:, :Ci], kva[:, Ci:2 * Ci], a3, frames=B, tokens=L, heads=H, head_dim=Ci // H,
                            n_keys=win["n_aud_tokens"], kv_frame_div=1, regions=3, q_region_stride=Ci,
                            kv_region_stride=2 * Ci, o_region_stride=Ci)
        m3 = self.buf("au.m3", M, 3 * Ci)
        for r, rn in enumerate(("full", "face", "lip")):
            ops.gemm(a3[:, r * Ci:(r + 1) * Ci], W[f"{tb}.attn2_{r}.to_out.0.w"], m3[:, r * Ci:(r + 1) * Ci],
                     bias=W[f"{tb}.attn2_{r}.to_out.0.b"], row_scale=win[f"mask.{rn}.{depth}"])
        h2 = self.buf("au.h2", M, Ci)
        ops.gemm(m3, win[f"{name}.zero.w"], h2, bias=win[f"{name}.zero.b"], residual=h1)
        h3 = self._ff(h2, f"{tb}.ff", f"{tb}.norm3", "au.h3")
        out = self.buf(out_tag, M, C)
        ops.gemm(h3, W[f"{name}.proj_out.w"], out, bias=W[f"{name}.proj_out.b"], residual=x)
        return out

    def _motion_px(self, name: str, x, level: int, C: int, out_tag: str):
        """Motion module of a frame-sharded window (motion_module.py:270-316 + :387-423): frame <-> pixel ownership is
        swapped around the module.  Rank `me` owns frames [me*fl, (me+1)*fl) everywhere else; inside the module it owns
        the pixel slice [me*Lg, (me+1)*Lg) of ALL nm + f frames (x18 rows: (half, frame, pixel)).

          in : GroupNorm of the local frames; its apply pass stores each row into the pixel owner's x18 over NVLink
               (ops.groupnorm_scatter) -> flag barrier
          mid: `_motion_body` over the nm + f frames of Lg pixels -- all rank-local, no replicated motion-frame rows
          out: proj_out GEMM whose epilogue stores every (frame, pixel) row into the frame owner's `recv`
               (hb_row_scatter) -> flag barrier -> out = recv + x (the module's residual)

        exchange == "nccl" performs the same two swaps with all_to_all_single (A/B baseline); emulate_group fills the
        peers' rows with copies of the local ones (single-GPU profile of one rank's shapes)."""
        W = self.W
        nb, nm, fl, f, R, me = self.nb, self.nm, self.fl, self.f, self.R, self.me
        L = self.L(level)
        Lg, F18 = L // R, nm + f
        tt = f"{name}.temporal_transformer"
        x18 = self._x18(name, nb * F18 * Lg, C)
        if self.arena is not None:
            ops.groupnorm_scatter(x, W[f"{tt}.norm.w"], W[f"{tt}.norm.b"], self.arena.addrs(f"x18.{name}"),
                                  self._gn_ws(), n_frames=nb * fl, hw=L, groups=self.cfg.norm_num_groups, eps=1e-6,
                                  fpb_in=fl, fpb_out=F18, frame_off=nm + me * fl)
            with ops.timed_region(f"peer_barrier in C{C} L{L}"):
                self.arena.barrier()
        else:
            gnl = self.buf("mm.gnl", nb * fl * L, C)
            self._gn(x, f"{tt}.norm", gnl, nb * fl, L, 1e-6, False)
            # send chunk d = my frames, pixel slice d; received chunk s = frames of rank s, my pixel slice
            got = self._exchange(gnl.view(nb, fl, R, Lg, C).permute(2, 0, 1, 3, 4),
                                 f"a2a_frames_to_pixels C{C} L{L} R{R}")
            x18.view(nb, F18, Lg, C)[:, nm:].view(nb, R, fl, Lg, C).copy_(got.permute(1, 0, 2, 3, 4))
        h = self._motion_body(name, x18, Lg, F18, self.window["pe_index_all"])
        out = self.buf(out_tag, nb * fl * L, C)
        if self.arena is not None:
            recv = self.arena.local("recv", (nb * fl * L, C), self.dtype)
            bases = self.arena.addrs("recv")
            for b in range(nb):                          # real frames only (the caller drops the motion frames)
                rows_in = h[(b * F18 + nm) * Lg:(b + 1) * F18 * Lg]                    # row r = g * Lg + p, g global frame
                sc = ops.row_scatter(bases, seg=Lg, segs_per_dest=fl, seg_stride=L, row0=b * fl * L + me * Lg)
                ops.gemm(rows_in, W[f"{tt}.proj_out.w"], recv[:f * Lg], bias=W[f"{tt}.proj_out.b"], scatter=sc)
            with ops.timed_region(f"peer_barrier out C{C} L{L}"):
                self.arena.barrier()
            ops.add(recv, x, out)
        else:
            y = self.buf("mm.y", nb * f * Lg, C)
            for b in range(nb):
                ops.gemm(h[(b * F18 + nm) * Lg:(b + 1) * F18 * Lg], W[f"{tt}.proj_out.w"], y[b * f * Lg:(b + 1) * f * Lg],
                         bias=W[f"{tt}.proj_out.b"])
            # send chunk d = frames of rank d, my pixel slice; received chunk s = my frames, pixel slice s
            got = self._exchange(y.view(nb, R, fl, Lg, C).permute(1, 0, 2, 3, 4),
                                 f"a2a_pixels_to_frames C{C} L{L} R{R}")
            torch.add(got.permute(1, 2, 0, 3, 4), x.view(nb, fl, R, Lg, C), out=out.view(nb, fl, R, Lg, C))
        return out

    def _exchange(self, chunks: torch.Tensor, region: str) -> torch.Tensor:
        """All-to-all of an exchange == "nccl" window: chunks[d] goes to rank d; returns chunks' shape with the chunk
        received from rank s at [s].  An emulated group receives copies of the chunk this rank keeps."""
        if self.shard.group_size == 1:
            return chunks[self.me].unsqueeze(0).expand(chunks.shape)
        import torch.distributed as dist
        C = chunks.shape[-1]
        send = self.buf("mm.a2a.s", chunks.numel() // C, C)
        recv = self.buf("mm.a2a.r", chunks.numel() // C, C)
        send.view(chunks.shape).copy_(chunks)
        with ops.timed_region(region):
            dist.all_to_all_single(recv, send, group=self.shard.group)
        return recv.view(chunks.shape)

    def _motion_body(self, name: str, x, tokens: int, frames: int, pe_index: torch.Tensor) -> torch.Tensor:
        """proj_in, 2 x {LayerNorm + PE, QKV, temporal attention over the frames, to_out}, FF of a motion module on the
        rows (cfg half, frame, pixel) of x, `frames` frames of `tokens` pixels each; returns the FF output."""
        W, H = self.W, self.cfg.heads
        M, C = x.shape
        tt = f"{name}.temporal_transformer"
        tb = f"{tt}.transformer_blocks.0"
        h = self.buf("mm.h", M, C)
        ops.gemm(x, W[f"{tt}.proj_in.w"], h, bias=W[f"{tt}.proj_in.b"])
        for a in range(2):
            n = self._ln(h, f"{tb}.norms.{a}", "mm.ln", pe=W[f"{tb}.attention_blocks.{a}.pe"], pe_index=pe_index,
                         tokens_per_frame=tokens, frames=frames)
            qkv = self.buf("mm.qkv", M, 3 * C)
            ops.gemm(n, W[f"{tb}.attention_blocks.{a}.qkv"], qkv)
            o = self.buf("mm.attn", M, C)
            ops.temporal_attention(qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:], o, batch=self.nb, fq=frames, fk=frames,
                                   tokens=tokens, heads=H)
            h2 = self.buf(f"mm.h{a + 1}", M, C)
            ops.gemm(o, W[f"{tb}.attention_blocks.{a}.to_out.0.w"], h2,
                     bias=W[f"{tb}.attention_blocks.{a}.to_out.0.b"], residual=h)
            h = h2
        return self._ff(h, f"{tb}.ff", f"{tb}.ff_norm", "mm.h3")

    def _motion(self, name: str, x, level: int, C: int, out_tag: str):
        if self.px:
            return self._motion_px(name, x, level, C, out_tag)
        W, nb, nm, fl = self.W, self.nb, self.nm, self.fl
        Fl = nm + fl
        L = self.L(level)
        tt = f"{name}.temporal_transformer"
        gn18 = self.buf(f"{name}.gn18", nb * Fl * L, C)          # frames [0, nm) were filled in begin_window
        self._gn(x, f"{tt}.norm", gn18, nb * fl, L, 1e-6, False, fpb_in=fl, fpb_out=Fl, frame_off=nm)
        h = self._motion_body(name, gn18, L, Fl, self.window["pe_index"])
        out = self.buf(out_tag, nb * fl * L, C)
        for b in range(nb):                              # proj_out only on the real frames (drops motion frames)
            rows_in = slice((b * Fl + nm) * L, (b + 1) * Fl * L)
            rows_out = slice(b * fl * L, (b + 1) * fl * L)
            ops.gemm(h[rows_in], W[f"{tt}.proj_out.w"], out[rows_out], bias=W[f"{tt}.proj_out.b"], residual=x[rows_out])
        return out

    def _cross_layer(self, b: BlockSpec, l: LayerSpec, x, level: int, out_tag: str):
        """The layer's spatial transformer, then its audio and motion modules where it has them: the last module writes
        out_tag, the others the shared lyr.* buffers."""
        C = b.channels
        x = self._spatial(l.attn, x, level, C, "lyr.sp" if l.audio or l.motion_executed else out_tag)
        if l.audio:
            x = self._audio(l.audio, x, level, C, l.audio_inner, b.depth, "lyr.au" if l.motion_executed else out_tag)
        if l.motion_executed:
            x = self._motion(l.motion, x, level, C, out_tag)
        return x

    # ------------------------------------------------------------------ forward
    def _walk(self):
        """Time embedding -> conv_in -> down / mid / up blocks over the local rows; reads self.latents (or self.sample)
        and the window, returns the last up block's features [B*L0, C0]."""
        W, cfg, B = self.W, self.cfg, self.B
        L0 = self.h * self.w
        c0 = cfg.block_out_channels[0]
        # time embedding (unet_3d.py:565-588) -> SiLU(emb) -> all 22 time_emb_proj at once
        emb = self.buf("temb.sin", self.nb, c0)
        ops.timestep_embed(self.t_table, self.step_idx, emb)
        e1 = self.buf("temb.e1", self.nb, cfg.time_embed_dim)
        ops.gemm(emb, W["time_embedding.linear_1.w"], e1, bias=W["time_embedding.linear_1.b"], silu=True)
        e2 = self.buf("temb.e2", self.nb, cfg.time_embed_dim)
        ops.gemm(e1, W["time_embedding.linear_2.w"], e2, bias=W["time_embedding.linear_2.b"], silu=True)
        self.temb_all = self.buf("temb.all", self.nb, W.temb_total)
        ops.gemm(e2, W["temb_all.w"], self.temb_all, bias=W["temb_all.b"])
        # conv_in (+ mask_cond_fea, unet_3d.py:603-605)
        cols = self.buf("im2col", B * L0, 64)
        ops.im2col_latent(self.sample if self.sample is not None else self.latents, cols, batch=self.nb)
        x = self.buf("x.conv_in", B * L0, c0)
        ops.gemm(cols, W["conv_in.w"], x, bias=W["conv_in.b"], residual=self.window.get("mask_cond"))
        skips = [x]
        level = 0
        for b in W.blocks:
            C = b.channels
            if b.kind in ("down_x", "down"):
                for j, l in enumerate(b.layers):
                    tag = f"skip.{b.name}.{j}"
                    x = self._resnet(l.resnet, x, None, level, "lyr.rs" if l.attn else tag)    # Q1b: resnet only
                    if l.attn:
                        x = self._cross_layer(b, l, x, level, tag)
                    skips.append(x)
                if b.downsampler:
                    hh, ww = self.level_hw[level]
                    planes = self.buf("ds.planes", B * hh * ww, C)
                    ops.phase_split(x.view(B, hh, ww, C), planes.view(4 * B, hh // 2, ww // 2, C))
                    level += 1
                    x = self.buf(f"skip.{b.name}.ds", B * self.L(level), C)
                    ops.conv3x3_stride2(planes.view(4 * B, hh // 2, ww // 2, C), W[f"{b.downsampler}.conv.w"], x,
                                        n=B, ho=hh // 2, wo=ww // 2, bias=W[f"{b.downsampler}.conv.b"])
                    skips.append(x)
            elif b.kind == "mid":
                # UNetMidBlock3D/2DCrossAttn: resnets[0] -> the layer's transformer modules -> resnets[1]
                x = self._resnet(b.extra_resnet, x, None, level, "mid.rs0")
                x = self._cross_layer(b, b.layers[0], x, level, "mid.mm")
                x = self._resnet(b.layers[0].resnet, x, None, level, "mid.out")
            else:
                for j, l in enumerate(b.layers):
                    tag = f"up.{b.name}.{j % 2}"
                    x = self._resnet(l.resnet, x, skips.pop(), level, "lyr.rs" if l.attn else tag)    # Q1b
                    if l.attn:
                        x = self._cross_layer(b, l, x, level, tag)
                if b.upsampler:
                    hh, ww = self.level_hw[level]
                    up = self.buf("us.up", B * 4 * hh * ww, C)
                    ops.upsample2x(x.view(B, hh, ww, C), up.view(B, 2 * hh, 2 * ww, C))
                    level -= 1
                    x = self.buf(f"up.{b.name}.us", B * self.L(level), C)
                    ops.conv3x3(up.view(B, 2 * hh, 2 * ww, C), W[f"{b.upsampler}.conv.w"], x,
                                bias=W[f"{b.upsampler}.conv.b"])
        return x

    @torch.no_grad()
    def _forward(self):
        """One UNet3D forward over the local shard; reads self.latents, writes self.model_out [B*L0, 8]."""
        x = self._walk()
        B, h, w, c0 = self.B, self.h, self.w, self.cfg.block_out_channels[0]
        t = self.buf("out.gn", B * h * w, c0)
        self._gn(x, "conv_norm_out", t, B, h * w, self.cfg.norm_eps, True)
        self.model_out = self.buf("out.conv", B * h * w, 8)
        ops.conv3x3(t.view(B, h, w, c0), self.W["conv_out.w"], self.model_out, bias=self.W["conv_out.b"])
        return self.model_out

    @torch.no_grad()
    def _step_tail(self):
        """CFG combine + DDIM update + step counter (face_animate.py:415-420)."""
        mo = self.model_out                    # both CFG halves of the local frames: the combine is rank-local
        ops.cfg_ddim_step(mo, self.latents, self.coef, self.step_idx, guidance=self.guidance)
        ops.advance_step(self.step_idx, self.n_steps)

    # ------------------------------------------------------------------ public
    @torch.no_grad()
    def forward_only(self, latents: torch.Tensor, step: int = 0) -> torch.Tensor:
        """UNet forward for fp32 latents [1, Cl, fl, h, w] (shared by the CFG halves) or a full per-half sample
        [nb, Cl, fl, h, w]; returns fp32 [nb, Cl, fl, h, w]."""
        latents = latents.to(self.dev, torch.float32).contiguous()
        if latents.shape[0] == 1:
            self.latents.copy_(latents)
            self.sample = None
        else:
            assert latents.shape[0] == self.nb
            self.sample = latents
        self.step_idx.fill_(step)
        mo = self._forward()
        self.sample = None
        out = torch.empty(self.nb, self.cfg.out_channels, self.fl, self.h, self.w, device=self.dev, dtype=torch.float32)
        ops.tokens_to_bcfhw(mo, out)
        return out

    @torch.no_grad()
    def capture(self):
        """Warm up (allocates every buffer) and capture forward + CFG/DDIM step into one CUDA graph."""
        lat0 = self.latents.clone()
        st0 = self.step_idx.clone()
        s = torch.cuda.Stream(device=self.dev)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self._forward()
            self._step_tail()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        self.latents.copy_(lat0)
        self.step_idx.copy_(st0)
        g = torch.cuda.CUDAGraph()
        # thread_local: the NCCL watchdog thread may touch CUDA while this thread captures (multi-GPU shards)
        with torch.cuda.graph(g, capture_error_mode="thread_local"):
            self._forward()
            self._step_tail()
        self.graph = g
        self._captured_with = (self.n_steps, self.guidance)
        self.latents.copy_(lat0)
        self.step_idx.copy_(st0)

    @torch.no_grad()
    def step(self):
        if self.graph is not None:
            self.graph.replay()
        else:
            self._forward()
            self._step_tail()
