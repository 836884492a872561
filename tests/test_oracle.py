"""CPU tests of the oracle (oracle/unet_ref.py): structure against the reference's module dump, LoRA semantics against
vectors produced by the REAL reference classes (tests/golden/ref_lora_linear.pt, ref_lora_wrap_layer.pt,
tests/golden/make_golden.py)."""
import json
import os

import torch

from oracle import unet_ref as U


def test_param_count_and_shapes_match_reference_dump(golden_dir):
    shapes = U.param_shapes(U.SD15)
    assert sum(torch.Size(s).numel() for s in shapes.values()) == 859_520_964      # SD1.5 UNet
    leaves = json.load(open(os.path.join(golden_dir, "unet_struct_sd15.json")))
    expected = {}
    for name, m in leaves.items():
        if m["type"] == "Linear":
            expected[name + ".weight"] = (m["out"], m["in"])
            if m["bias"]:
                expected[name + ".bias"] = (m["out"],)
        elif m["type"] == "Conv2d":
            expected[name + ".weight"] = (m["out"], m["in"], m["k"], m["k"])
            expected[name + ".bias"] = (m["out"],)
        elif m["type"] in ("GroupNorm", "LayerNorm"):
            expected[name + ".weight"] = (m["ch"],)
            expected[name + ".bias"] = (m["ch"],)
    assert set(expected) == set(shapes)
    for k, s in expected.items():
        assert tuple(shapes[k]) == tuple(s), k
    # eps / stride pins the oracle hard-codes
    assert leaves["down_blocks.0.attentions.0.norm"]["eps"] == U.SD15.transformer_norm_eps
    assert leaves["down_blocks.0.resnets.0.norm1"]["eps"] == U.SD15.resnet_eps
    assert leaves["down_blocks.0.attentions.0.transformer_blocks.0.norm1"]["eps"] == U.SD15.layernorm_eps
    assert leaves["down_blocks.0.downsamplers.0.conv"]["stride"] == 2 and leaves["up_blocks.0.upsamplers.0.conv"]["stride"] == 1


def test_lora_targets_match_survey():
    layers = U.lora_target_layers(U.SD15, r".*\.attn.?$")
    assert len(layers) == 128
    shapes = U.param_shapes()
    assert sum(8 * (shapes[l + ".weight"][0] + shapes[l + ".weight"][1]) for l in layers) == 1_594_368
    assert len(U.lora_target_layers(U.SD15, r".*\.attn.?$|.*\.ff$")) == 160


def _oracle_from_golden(fx):
    sd, lora = {}, {}
    for k, v in fx["host"].items():
        sd[k.replace("._host", "")] = v
    for k, v in fx["ckpt"].items():
        layer, key = k.split(".___.")
        e = lora.setdefault(layer, {})
        e[key] = v
    out = {}
    for layer, e in lora.items():
        out[layer] = [U.LoraEntry(e["layer.W_down"].clone(), e["layer.W_up"].clone(), float(e["alpha"]))]
    sb = fx["second_block"]
    out["attn1.to_q"].append(U.LoraEntry(sb["layer.W_down"].clone(), sb["layer.W_up"].clone(), float(sb["alpha"])))
    return sd, out


def test_oracle_lora_matches_reference_golden(golden_dir):
    fx = torch.load(os.path.join(golden_dir, "ref_lora_linear.pt"))
    sd, lora = _oracle_from_golden(fx)
    x = fx["x"].clone().requires_grad_(True)
    for entries in lora.values():
        for e in entries:
            e.W_down.requires_grad_(True)
            e.W_up.requires_grad_(True)
    outs = {
        "attn1.to_q": U._linear(sd, lora, "attn1.to_q", x), "attn1.to_k": U._linear(sd, lora, "attn1.to_k", x),
        "attn1.to_out.0": U._linear(sd, lora, "attn1.to_out.0", x), "attn2.to_k": U._linear(sd, lora, "attn2.to_k", fx["ctx"]),
        "attn2.to_q": U._linear(sd, lora, "attn2.to_q", x),
    }
    for k, v in outs.items():
        torch.testing.assert_close(v, fx["outs"][k], rtol=1e-5, atol=1e-6)
    sum((o ** 2).sum() for o in outs.values()).backward()
    torch.testing.assert_close(x.grad, fx["grad_x"], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(lora["attn1.to_q"][0].W_down.grad, fx["grads"]["attn1.to_q.lora_block_0.layer.W_down"], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(lora["attn1.to_q"][1].W_up.grad, fx["grads"]["attn1.to_q.lora_block_1.layer.W_up"], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(lora["attn2.to_k"][0].W_up.grad, fx["grads"]["attn2.to_k.lora_block_0.layer.W_up"], rtol=1e-4, atol=1e-5)
    # alpha = alpha/rank (auto scale): block 0 rank 4 alpha 1.0, block 1 rank 2 alpha 0.5
    assert abs(float(fx["ckpt"]["attn1.to_q.___.alpha"]) - 0.25) < 1e-7 and abs(float(fx["second_block"]["alpha"]) - 0.25) < 1e-7


def test_oracle_lora_matches_live_reference_classes(golden_dir):
    """The reference's LoraLayer.wrap_layer on a biased Linear (rank 8, alpha 2.0 -> 0.25 after auto scale): its output, stored in
    tests/golden/ref_lora_wrap_layer.pt by tests/golden/make_golden.py, vs the oracle's `_linear` on the same weights and input."""
    fx = torch.load(os.path.join(golden_dir, "ref_lora_wrap_layer.pt"))
    sd = {"lin.weight": fx["weight"], "lin.bias": fx["bias"]}
    lora = {"lin": [U.LoraEntry(fx["W_down"], fx["W_up"], fx["alpha"])]}
    assert fx["W_down"].shape == (8, 40) and fx["alpha"] == 0.25
    torch.testing.assert_close(U._linear(sd, lora, "lin", fx["x"]), fx["out"], rtol=1e-5, atol=1e-6)


def test_tiny_unet_forward_backward_runs_and_is_deterministic():
    sd = U.init_params(U.TINY)
    lat, noise, t, ehs = U.synthetic_batch(2, U.TINY, ctx_len=9)
    lora = U.init_lora(U.TINY, rank=4)
    loss1, pred1, grads1 = U.lora_step_loss_and_grads(sd, lora, lat, noise, t, ehs, U.TINY)
    loss2, pred2, _ = U.lora_step_loss_and_grads(sd, U.init_lora(U.TINY, rank=4), lat, noise, t, ehs, U.TINY)
    assert pred1.shape == (2, 4, 16, 16) and torch.isfinite(pred1).all()
    torch.testing.assert_close(pred1, pred2)
    assert float(loss1) == float(loss2)
    assert all(torch.isfinite(g).all() for bl in grads1.values() for pair in bl for g in pair)
    # an all-ones attention mask is the identity; masking a token changes the result
    m = torch.ones(2, 9)
    p_mask = U.unet_forward(sd, lat, t, ehs, encoder_attention_mask=m, spec=U.TINY)
    torch.testing.assert_close(p_mask, U.unet_forward(sd, lat, t, ehs, spec=U.TINY), rtol=1e-4, atol=1e-5)
    m[:, -1] = 0
    assert not torch.allclose(U.unet_forward(sd, lat, t, ehs, encoder_attention_mask=m, spec=U.TINY), p_mask)


def test_timestep_embedding_layout():
    e = U.timestep_embedding(torch.tensor([0, 10]), 320)
    assert e.shape == (2, 320)
    torch.testing.assert_close(e[0, :160], torch.ones(160))      # cos(0) first (flip_sin_to_cos)
    torch.testing.assert_close(e[0, 160:], torch.zeros(160))


def _dapp_conv_oracle(fx):
    """(state dict of the host layers, LoraDict) of the DAPP / Conv2d-LoRA golden fixture."""
    sd, lora = {}, {}
    st = fx["state"]
    for k, v in st.items():
        if "._host." in k:
            sd[k.replace("._host", "")] = v
    for k in st:
        if k.endswith(".layer.W_down"):
            base = k[: -len(".layer.W_down")]                       # '<layer>.lora_block_<id>'
            layer = base.rsplit(".", 1)[0]
            branch = None
            if fx["container_types"][layer] == "DAPPPatchContainer":
                branch = "p" if base.endswith("lora_block_0") else "n"     # make_golden.py wraps ('p', rank 4) then ('n', rank 2)
            lora.setdefault(layer, []).append(U.LoraEntry(st[k].clone(), st[base + ".layer.W_up"].clone(), float(st[base + ".alpha"]), branch))
    return sd, lora


def test_oracle_dapp_and_conv_lora_match_reference_golden(golden_dir):
    """DAPPPatchContainer / DAPPLayer and LoraLayer.Conv2dLayer of the REAL reference (tests/golden/ref_lora_dapp_conv.pt) vs the
    oracle's `_linear` (batch = [negative | positive]) and `_conv`: outputs, input gradients, parameter gradients."""
    fx = torch.load(os.path.join(golden_dir, "ref_lora_dapp_conv.pt"))
    assert fx["container_types"]["to_k"] == "DAPPPatchContainer" and fx["container_types"]["conv"] == "LoraPatchContainer"
    sd, lora = _dapp_conv_oracle(fx)
    for blocks in lora.values():
        for e in blocks:
            e.W_down.requires_grad_(True)
            e.W_up.requires_grad_(True)
    xk, xf, xc = (fx[k].clone().requires_grad_(True) for k in ("xk", "xf", "xc"))
    outs = {"to_k": U._linear(sd, lora, "to_k", xk), "ff": U._linear(sd, lora, "ff", xf),
            "conv": U._conv(sd, lora, "conv", xc, padding=1), "conv_s2": U._conv(sd, lora, "conv_s2", xc, stride=2, padding=1),
            "proj": U._conv(sd, lora, "proj", xc)}
    for k, v in outs.items():
        torch.testing.assert_close(v, fx["outs"][k], rtol=1e-5, atol=1e-5)
    sum((o ** 2).sum() for o in outs.values()).backward()
    for k, x in (("xk", xk), ("xf", xf), ("xc", xc)):
        torch.testing.assert_close(x.grad, fx["grad_in"][k], rtol=1e-4, atol=1e-4)
    n = 0
    for layer, blocks in lora.items():
        for e in blocks:
            bid = 0 if e.branch in (None, "p") else 1
            torch.testing.assert_close(e.W_down.grad, fx["grads"][f"{layer}.lora_block_{bid}.layer.W_down"], rtol=1e-4, atol=1e-4)
            torch.testing.assert_close(e.W_up.grad, fx["grads"][f"{layer}.lora_block_{bid}.layer.W_up"], rtol=1e-4, atol=1e-4)
            n += 2
    assert n == len(fx["grads"])
    # the two halves of a DAPP batch really see different weights
    assert not torch.allclose(outs["to_k"][:2], U._mm(fx["xk"][:2], sd["to_k.weight"] + U.lora_delta(lora["to_k"], "p"), None))
