"""ReferenceNet on the sm_100a kernels (SURVEY.md 8f row 1): the SD-1.5 UNet2D the reference runs once per window at
t = 0 on the reference image + motion frames (hallo/models/unet_2d_condition.py forward :905-1356, blocks
unet_2d_blocks.py, transformer_2d.py:245-420, BasicTransformerBlock attention.py:79-407) whose per-block
`norm1(hidden_states)` are the K/V banks of the denoising UNet's spatial attention (write mode,
mutual_self_attention.py:223-232, 333-366).

It is the denoising engine's kernel plan, `DenoiseEngine._walk`, over a block list without audio / motion modules
(spec.build_blocks_2d) and a window without reference K/V; norm1 writes into the bank buffers.  There is no conv_out:
the reference returns the last up block's features (post_process=False, :1344-1349).
The six samples (2 CFG copies x (reference + nm motion frames)) ride the token layout as six "frames" of one batch.
Reproduced quirk (Q10): the image tokens are tiled over the batch -- `encoder_hidden_states.repeat(tmp, 1, 1)`
(mutual_self_attention.py:340-346) -- so sample n cross-attends to the tokens of CFG half n % 2, not n // 3.
"""
from __future__ import annotations

from typing import List, Tuple

import torch

from . import ops
from .engine import DenoiseEngine, PackedWeights, Shard
from .spec import build_blocks_2d, reader_bank_order


class ReferenceNetWeights(PackedWeights):
    """Kernel-ready copies of the 682-entry UNet2D state dict (same packing as the 3D model's resnets / spatial blocks)."""
    build_blocks = staticmethod(build_blocks_2d)


class ReferenceNetEngine(DenoiseEngine):
    def __init__(self, weights: ReferenceNetWeights, h: int, w: int, n_samples: int):
        super().__init__(weights, h, w, n_samples, Shard(halves=(0,), frames=tuple(range(n_samples))))
        self.n = n_samples
        self.bank_names: List[Tuple[str, int]] = reader_bank_order(self.cfg)

    def _norm1_tag(self, name: str) -> str:
        return f"bank.{name}"

    @torch.no_grad()
    def run(self, sample: torch.Tensor, timestep, encoder_hidden_states: torch.Tensor):
        """sample (n, 4, h, w), timestep scalar, encoder_hidden_states (n_ehs, tokens, 768) with n % n_ehs == 0.
        Returns (features of the last up block as fp32 (n, C0, h, w), {attn name: bank (n, L, C) in model dtype})."""
        W, win = self.W, self.window
        n = sample.shape[0]
        assert n == self.n and n % encoder_hidden_states.shape[0] == 0
        ehs = encoder_hidden_states.to(self.dev, self.dtype)
        tiled = ehs.repeat(n // ehs.shape[0], 1, 1).reshape(n * ehs.shape[1], ehs.shape[2])    # Q10: not interleaved
        win["n_img_tokens"] = ehs.shape[1]
        win["kvimg_frame_div"] = 1                                      # sample n reads image K/V rows of batch n
        for b in W.blocks:
            for l in b.layers:
                if l.attn:
                    kv = win[f"{l.attn}.kvimg"] = self.buf(f"{l.attn}.kvimg", tiled.shape[0], 2 * b.channels)
                    ops.gemm(tiled, W[f"{l.attn}.transformer_blocks.0.attn2.kv"], kv)
        self.set_timestep(float(timestep) if not torch.is_tensor(timestep) else float(timestep.reshape(-1)[0]))
        self.step_idx.zero_()
        # the n samples become n frames of one batch entry: latents [1, Cl, n, h, w]
        self.latents.copy_(sample.to(self.dev, torch.float32).permute(1, 0, 2, 3).unsqueeze(0))
        x = self._walk()
        out = torch.empty(1, self.cfg.block_out_channels[0], n, self.h, self.w, device=self.dev, dtype=torch.float32)
        ops.tokens_to_bcfhw(x, out)
        banks = {}
        for name, C in self.bank_names:
            L = self.L(self._block_level(name))
            banks[name] = self.buf(self._norm1_tag(name), n * L, C).view(n, L, C)
        return out[0].permute(1, 0, 2, 3).contiguous(), banks
