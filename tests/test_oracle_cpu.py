"""CPU tests of the oracle: the restatement (oracle/port.py) against the committed golden vectors made from
the UNMODIFIED reference (oracle/make_golden.py), including fp32 ones held to 2e-5, and against independent formulas."""
import json
import os

import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2
from hallo_b200.spec import UNetConfig, build_blocks, param_spec, reader_bank_order
from hallo_b200.synth import host_threads, synth_inputs, synth_state_dict

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def cfg():
    return UNetConfig()


@pytest.fixture(scope="module")
def sd(cfg):
    torch.set_num_threads(host_threads())
    return synth_state_dict(cfg, seed=0)


def test_state_dict_contract_matches_reference_keys(cfg):
    """The 1946-entry key/shape list of the reference UNet3D (fixture dumped from the reference itself)."""
    ref = json.load(open(os.path.join(GOLD, "unet3d_state_dict_keys.json")))
    mine = {k: list(s) for k, s, _ in param_spec(cfg)}
    assert len(ref) == 1946
    assert mine == ref


def test_structure_quirks(cfg):
    blocks = {b.name: b for b in build_blocks(cfg)}
    # Q5: irregular audio widths
    assert [l.audio_inner for l in blocks["down_blocks.1"].layers] == [320, 640]
    assert [l.audio_inner for l in blocks["down_blocks.2"].layers] == [640, 1280]
    assert [l.audio_inner for l in blocks["up_blocks.1"].layers] == [640, 640, 640]
    assert [l.audio_inner for l in blocks["up_blocks.2"].layers] == [320, 320, 320]
    # Q1b: plain down/up blocks never execute their motion modules
    assert not any(l.motion_executed for l in blocks["down_blocks.3"].layers + blocks["up_blocks.0"].layers)
    assert sum(l.motion_executed for b in blocks.values() for l in b.layers) == 16
    # resnet channel plan (SURVEY 8a-note)
    assert [(l.resnet.cin, l.resnet.cout) for l in blocks["up_blocks.2"].layers] == [(1920, 640), (1280, 640), (960, 640)]
    order = [n for n, _ in reader_bank_order(cfg)]
    assert order[:6] == ["down_blocks.2.attentions.0", "down_blocks.2.attentions.1", "up_blocks.1.attentions.0",
                         "up_blocks.1.attentions.1", "up_blocks.1.attentions.2", "mid_block.attentions.0"]


@pytest.mark.parametrize("name", ["unet_fwd_h8_f2.pt", "unet_fwd_h16_f3.pt", "unet_fwd_h16_f16.pt"])
def test_port_matches_golden(cfg, sd, name):
    from oracle import port
    fx = torch.load(os.path.join(GOLD, name), weights_only=False)
    c = fx["case"]
    inp = synth_inputs(cfg, c["h"], c["h"], c["f"], seed=c["seed"], timestep=c["t"], motion_scale=c["ms"])
    # generator drift guards
    assert abs(float(inp["sample"].double().abs().sum()) - fx["input_checksums"]["sample"]) < 1e-6 * fx["input_checksums"]["sample"]
    for k, v in fx["weight_checksums"].items():
        assert abs(float(sd[k].double().abs().sum()) - v) < 1e-6 * v
    taps = {}
    out = port.unet_forward(sd, cfg, inp, taps=taps)
    assert rel_l2(out, fx["out"]) < 2e-5
    for bname, st in fx["taps"].items():
        t = taps[bname]
        assert abs(float(t.std()) - st["std"]) < 1e-3 * st["std"] + 1e-6, bname


def test_port_matches_reference_host(cfg, sd):
    """fp32 cross-check against the unmodified reference UNet3D (read-mode reader, synthetic banks) on the same synth
    weights and inputs: latent 8x8, 3 frames, t=123, uneven motion scales (fixture unet_fwd_h8_f3.pt)."""
    from oracle import port
    fx = torch.load(os.path.join(GOLD, "unet_fwd_h8_f3.pt"), weights_only=False)
    c = fx["case"]
    assert c == dict(h=8, f=3, seed=7, t=123, ms=(0.7, 1.3, 1.0))
    inp = synth_inputs(cfg, c["h"], c["h"], c["f"], seed=c["seed"], timestep=c["t"], motion_scale=c["ms"])
    out = port.unet_forward(sd, cfg, inp)
    assert fx["out"].dtype == torch.float32 and rel_l2(out, fx["out"]) < 2e-5


def test_attention_restatement_vs_sdpa():
    from oracle import port
    g = torch.Generator().manual_seed(0)
    C, H = 64, 8
    sdx = {f"a.{n}.weight": torch.randn(C, C, generator=g) / 8 for n in ("to_q", "to_k", "to_v", "to_out.0")}
    sdx["a.to_out.0.bias"] = torch.randn(C, generator=g)
    x = torch.randn(3, 10, C, generator=g)
    ctx = torch.randn(3, 7, C, generator=g)
    out = port.attention(sdx, "a", x, ctx, H)
    q = F.linear(x, sdx["a.to_q.weight"]).view(3, 10, H, 8).transpose(1, 2)
    k = F.linear(ctx, sdx["a.to_k.weight"]).view(3, 7, H, 8).transpose(1, 2)
    v = F.linear(ctx, sdx["a.to_v.weight"]).view(3, 7, H, 8).transpose(1, 2)
    o = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(3, 10, C)
    ref = F.linear(o, sdx["a.to_out.0.weight"], sdx["a.to_out.0.bias"])
    assert rel_l2(out, ref) < 1e-5


def test_ddim_schedule_known_answers():
    """Q7: trailing spacing 999..24, zero terminal SNR, v-prediction update."""
    from oracle import port
    s = port.DDIM()
    ts = s.timesteps(40)
    assert ts[0] == 999 and ts[1] == 974 and ts[-1] == 24 and len(ts) == 40
    assert float(s.alphas_cumprod[999]) < 1e-10                      # zero terminal SNR
    assert abs(float(s.alphas_cumprod[0]) - (1 - 0.00085)) < 1e-6    # first alpha_bar is preserved by the rescale
    x = torch.randn(2, 3)
    v = torch.randn(2, 3)
    # at t=999 (alpha_bar=0): x0 = -v, eps = x  ->  x' = sqrt(a') * (-v) + sqrt(1-a') * x
    ap = s.alphas_cumprod[974]
    assert torch.allclose(s.step(v, 999, x, 40), ap.sqrt() * (-v) + (1 - ap).sqrt() * x, atol=1e-6)
    # last step lands on x0 exactly (final_alpha_cumprod = 1)
    a = s.alphas_cumprod[24]
    assert torch.allclose(s.step(v, 24, x, 40), a.sqrt() * x - (1 - a).sqrt() * v, atol=1e-6)


# ------------------------------------------------------------------------------------------------ ReferenceNet (8f row 1)
def test_refnet_state_dict_contract_matches_reference_keys(cfg):
    """The 682-entry key/shape list of the reference's UNet2DConditionModel (dumped from the reference class itself)."""
    from hallo_b200.spec import param_spec_2d
    ref = json.load(open(os.path.join(GOLD, "unet2d_state_dict_keys.json")))
    mine = {k: list(s) for k, s, _ in param_spec_2d(cfg)}
    assert len(ref) == 682 and mine == ref
    from hallo_b200.models.unet_2d_condition import UNet2DConditionModel
    from hallo_b200.spec import SD15_UNET_CONFIG
    m = UNet2DConditionModel.from_config(SD15_UNET_CONFIG)
    assert {k: list(v.shape) for k, v in m.state_dict().items()} == ref


def test_refnet_port_matches_golden(cfg):
    """oracle/port.reference_net_forward against the fixture produced by the UNMODIFIED reference UNet2D with the
    reference's own write-mode ReferenceAttentionControl: output features, bank pairing order, every bank's statistics,
    three banks element-wise."""
    from hallo_b200.synth import synth_refnet_inputs, synth_state_dict_2d
    from oracle import port
    fx = torch.load(os.path.join(GOLD, "refnet_h8.pt"), weights_only=False)
    torch.set_num_threads(host_threads())
    sd2 = synth_state_dict_2d(cfg)
    inp = synth_refnet_inputs(cfg, fx["case"]["h"], fx["case"]["h"], seed=fx["case"]["seed"])
    assert abs(float(inp["sample"].double().abs().sum()) - fx["input_checksums"]["sample"]) < 1e-6 * fx["input_checksums"]["sample"]
    out, banks = port.reference_net_forward(sd2, cfg, inp)
    assert rel_l2(out, fx["out"].float()) < 1e-3                        # fixture stored in fp16
    assert fx["bank_order"] == [n for n, _ in reader_bank_order(cfg)]   # A11: the reference control's own pairing order
    for n, st in fx["bank_stats"].items():
        b = banks[n]
        assert list(b.shape) == st["shape"]
        assert abs(float(b.double().abs().sum()) - st["abs_sum"]) < 1e-4 * st["abs_sum"], n
    for n, b in fx["banks"].items():
        assert rel_l2(banks[n], b.float()) < 1e-3, n


def test_refnet_port_matches_reference_host(cfg):
    """fp32 cross-check against the unmodified reference UNet2D + reference writer at latent 16x16 (fixture
    refnet_h16_f32.pt: seeded samples of the output and of every bank, and the absolute sums of the full tensors)."""
    from oracle import port
    from hallo_b200.synth import synth_refnet_inputs, synth_state_dict_2d
    fx = torch.load(os.path.join(GOLD, "refnet_h16_f32.pt"), weights_only=False)
    torch.set_num_threads(host_threads())
    sd2 = synth_state_dict_2d(cfg)
    inp = synth_refnet_inputs(cfg, fx["case"]["h"], fx["case"]["h"], seed=fx["case"]["seed"])

    def err(t, ref):
        """relative L2 over the stored sample, or the relative error of the full tensor's absolute sum if larger"""
        return max(rel_l2(t.reshape(-1)[ref["index"].long()], ref["values"]),
                   abs(float(t.double().abs().sum()) - ref["abs_sum"]) / ref["abs_sum"])
    o2, b2 = port.reference_net_forward(sd2, cfg, inp)
    assert fx["bank_order"] == [n for n, _ in reader_bank_order(cfg)]
    assert err(o2, fx["out"]) < 2e-5
    assert set(b2) == set(fx["banks"]) and max(err(b2[n], b) for n, b in fx["banks"].items()) < 2e-5
    # Q10: the image tokens are tiled over the 6 samples (n % 2), not interleaved (n // 3): a restatement with
    # repeat_interleave must NOT match
    inp_sw = dict(inp)
    wrong = inp["encoder_hidden_states"].repeat_interleave(3, dim=0)
    inp_sw["encoder_hidden_states"] = wrong
    o3, _ = port.reference_net_forward(sd2, cfg, inp_sw)
    assert rel_l2(o3.reshape(-1)[fx["out"]["index"].long()], fx["out"]["values"]) > 1e-3
