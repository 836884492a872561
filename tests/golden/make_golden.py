"""Generate the golden fixtures under tests/golden/ from the UNMODIFIED reference tree (/root/reference).

Run in the build container only (the GPU box has no /root/reference):  python tests/golden/make_golden.py

Outputs (small, committed):
  unet_struct_sd15.json   leaf modules of cfgs/unet_struct.txt -> parameter names/shapes/eps/stride (structure pin)
  ref_lora_linear.pt      vectors produced by the REAL reference classes hcpdiff.models.lora_layers_patch.LoraLayer /
                          lora_base_patch.LoraPatchContainer / plugin.PluginGroup: inputs, outputs, gradients and the
                          checkpoint key names (the operator the CUDA kernels sit behind)
  ref_lora_dapp_conv.pt   the same for the DreamArtist++ pair (DAPPLayer / DAPPPatchContainer: batch = [negative | positive]) and
                          for LoraLayer on Conv2d hosts (3x3 stride 1 / stride 2 and 1x1)
  ref_lora_wrap_layer.pt  LoraLayer.wrap_layer on a biased Linear (rank 8, alpha 2.0): weights, input and the reference output
  ref_step.pt             the step either side of the UNet, from the REAL reference code: MinSNRLoss / SoftMinSNRLoss / KDiffMinSNRLoss /
                          EDMLoss (hcpdiff/loss/min_snr_loss.py), a ModelEMA trajectory (hcpdiff/utils/ema.py), DreamArtistPTContext
                          pre/post (hcpdiff/models/cfg_context.py), get_cfg_range (hcpdiff/utils/utils.py), and DAPPLayer on a 3x3
                          Conv2d host (batch = [negative | positive])
  lora_webui_keys.json    hcpdiff <-> webui key maps of the REAL reference LoraConverter for the 160 SD1.5 attention/ff LoRA layers
"""
import importlib
import json
import os
import re
import sys
import types

import torch
from torch import nn

REF = os.environ.get("HCP_REFERENCE", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))


def import_reference_lora():
    """Import hcpdiff.models.{plugin,lora_base_patch,lora_layers_patch} without diffusers/accelerate/hydra:
    pre-register empty packages and stub the two helper modules they need (SURVEY.md App. D)."""
    sys.dont_write_bytecode = True
    for name, path in (("hcpdiff", "hcpdiff"), ("hcpdiff.utils", "hcpdiff/utils"), ("hcpdiff.models", "hcpdiff/models")):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__path__ = [os.path.join(REF, path)]
            sys.modules[name] = m
    u = types.ModuleType("hcpdiff.utils.utils")
    u.low_rank_approximate = lambda w, rank: (_ for _ in ()).throw(NotImplementedError())
    u.make_mask = lambda *a, **k: None
    u.isinstance_list = lambda obj, cls_list: any(isinstance(obj, c) for c in cls_list)
    sys.modules["hcpdiff.utils.utils"] = u
    nu = types.ModuleType("hcpdiff.utils.net_utils")

    def split_module_name(layer_name):
        name_split = layer_name.rsplit(".", 1)
        if len(name_split) == 1:
            return "", name_split[0]
        return name_split[0], name_split[1]

    nu.split_module_name = split_module_name
    sys.modules["hcpdiff.utils.net_utils"] = nu
    lay = types.ModuleType("hcpdiff.models.layers")
    lay.GroupLinear = type("GroupLinear", (nn.Module,), {})
    sys.modules["hcpdiff.models.layers"] = lay
    plugin = importlib.import_module("hcpdiff.models.plugin")
    base = importlib.import_module("hcpdiff.models.lora_base_patch")
    layers = importlib.import_module("hcpdiff.models.lora_layers_patch")
    return plugin, base, layers


def parse_struct(path):
    """cfgs/unet_struct.txt -> {module_path: {'type':..., ...}} for leaf modules with parameters."""
    stack = []   # (indent, name)
    leaves = {}
    line_re = re.compile(r"^(\s*)\((\w+)\): (\w+)\((.*)$")
    for raw in open(path):
        m = line_re.match(raw.rstrip("\n"))
        if not m:
            continue
        indent, name, typ, rest = len(m.group(1)), m.group(2), m.group(3), m.group(4)
        while stack and stack[-1][0] >= indent:
            stack.pop()
        full = ".".join([s[1] for s in stack] + [name])
        stack.append((indent, name))
        rest = rest[:-1] if rest.endswith(")") else rest
        if typ == "Linear":
            a = dict(re.findall(r"(\w+)=([\w\.]+)", rest))
            leaves[full] = {"type": "Linear", "in": int(a["in_features"]), "out": int(a["out_features"]),
                            "bias": a["bias"] == "True"}
        elif typ == "Conv2d":
            mm = re.match(r"(\d+), (\d+), kernel_size=\((\d+), (\d+)\), stride=\((\d+), (\d+)\)(?:, padding=\((\d+), (\d+)\))?", rest)
            leaves[full] = {"type": "Conv2d", "in": int(mm.group(1)), "out": int(mm.group(2)), "k": int(mm.group(3)),
                            "stride": int(mm.group(5)), "padding": int(mm.group(7) or 0)}
        elif typ == "GroupNorm":
            mm = re.match(r"(\d+), (\d+), eps=([\de\-\.]+)", rest)
            leaves[full] = {"type": "GroupNorm", "groups": int(mm.group(1)), "ch": int(mm.group(2)), "eps": float(mm.group(3))}
        elif typ == "LayerNorm":
            mm = re.match(r"\((\d+),\), eps=([\de\-\.]+)", rest)
            leaves[full] = {"type": "LayerNorm", "ch": int(mm.group(1)), "eps": float(mm.group(2))}
    return leaves


def make_struct():
    leaves = parse_struct(os.path.join(REF, "cfgs/unet_struct.txt"))
    with open(os.path.join(HERE, "unet_struct_sd15.json"), "w") as f:
        json.dump(leaves, f, indent=0, sort_keys=True)
    print("unet_struct_sd15.json:", len(leaves), "leaf modules")


class _Attn(nn.Module):
    def __init__(self, c, ctx):
        super().__init__()
        self.to_q = nn.Linear(c, c, bias=False)
        self.to_k = nn.Linear(ctx, c, bias=False)
        self.to_out = nn.ModuleList([nn.Linear(c, c, bias=True), nn.Dropout(0.0)])


class _Blk(nn.Module):
    def __init__(self):
        super().__init__()
        self.attn1 = _Attn(48, 48)
        self.attn2 = _Attn(48, 24)


def make_lora():
    plugin, base, layers = import_reference_lora()
    torch.manual_seed(0)
    model = _Blk().float()
    fx = {}
    named = dict(model.named_modules())
    # what reference make_hcpdiff does for one `lora_unet` item (cfg_net_tools.py:108-121): wrap_model on each match
    blocks = {}
    for lname in ("attn1", "attn2"):
        d = layers.LoraLayer.wrap_model(0, named[lname], parent_block=None, host_name=None, rank=4, dropout=0.0, alpha=1.0,
                                        exclude_key=None)
        blocks.update({f"{lname}.{k}": v for k, v in d.items()})
    # second stacked block on attn1.to_q (two `lora_unet` items hitting one layer)
    d = layers.LoraLayer.wrap_model(1, named["attn1"].to_q, parent_block=named["attn1"], host_name="to_q", rank=2,
                                    dropout=0.0, alpha=0.5)
    second = d[""]
    g = torch.Generator().manual_seed(5)
    for blk in list(blocks.values()) + [second]:
        blk.init_weights()
        with torch.no_grad():
            blk.layer.W_up.copy_(torch.randn(blk.layer.W_up.shape, generator=g) * 0.1)
    group = plugin.PluginGroup(blocks)
    fx["state_keys_model"] = sorted(model.state_dict().keys())
    fx["ckpt_keys"] = sorted(group.state_dict().keys())
    fx["ckpt"] = {k: v.clone() for k, v in group.state_dict().items()}
    fx["second_block"] = {k: v.clone() for k, v in second.state_dict().items()}
    fx["host"] = {k: v.clone() for k, v in model.state_dict().items() if "._host." in k}
    x = torch.randn(3, 7, 48, generator=g)
    ctx = torch.randn(3, 5, 24, generator=g)
    x.requires_grad_(True)
    outs = {"attn1.to_q": model.attn1.to_q(x), "attn1.to_k": model.attn1.to_k(x), "attn1.to_out.0": model.attn1.to_out[0](x),
            "attn2.to_k": model.attn2.to_k(ctx), "attn2.to_q": model.attn2.to_q(x)}
    loss = sum((o ** 2).sum() for o in outs.values())
    loss.backward()
    fx["x"], fx["ctx"] = x.detach().clone(), ctx.clone()
    fx["outs"] = {k: v.detach().clone() for k, v in outs.items()}
    fx["grad_x"] = x.grad.clone()
    fx["grads"] = {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None and "lora_block" in n}
    torch.save(fx, os.path.join(HERE, "ref_lora_linear.pt"))
    print("ref_lora_linear.pt: ckpt keys", fx["ckpt_keys"][:4], "...", len(fx["ckpt_keys"]))
    print("  model keys sample:", [k for k in fx["state_keys_model"] if "to_q" in k][:6])


class _DappConvNet(nn.Module):
    def __init__(self):
        super().__init__()
        self.to_k = nn.Linear(24, 32, bias=False)
        self.ff = nn.Linear(32, 32, bias=True)
        self.conv = nn.Conv2d(8, 16, 3, padding=1)
        self.conv_s2 = nn.Conv2d(8, 16, 3, stride=2, padding=1)
        self.proj = nn.Conv2d(8, 16, 1)


def make_dapp_conv():
    """DreamArtist++ (DAPPLayer / DAPPPatchContainer) and Conv2d LoRA (LoraLayer.Conv2dLayer) vectors from the real reference."""
    plugin, base, layers = import_reference_lora()
    torch.manual_seed(1)
    model = _DappConvNet().float()
    g = torch.Generator().manual_seed(7)
    blocks = {}
    for lname in ("to_k", "ff"):
        for lora_id, (branch, rank) in enumerate((("p", 4), ("n", 2))):
            host = getattr(model, lname)
            blk = layers.DAPPLayer.wrap_layer(lora_id, host, rank=rank, dropout=0.0, alpha=1.0, branch=branch, parent_block=model,
                                              host_name=lname)
            blocks[f"{lname}.{branch}"] = blk
    for lname in ("conv", "conv_s2", "proj"):
        blk = layers.LoraLayer.wrap_layer(0, getattr(model, lname), rank=4, dropout=0.0, alpha=2.0, parent_block=model, host_name=lname)
        blocks[lname] = blk
    for blk in blocks.values():
        with torch.no_grad():
            blk.layer.W_up.copy_(torch.randn(blk.layer.W_up.shape, generator=g) * 0.2)
    fx = {"state_keys_model": sorted(model.state_dict().keys())}
    fx["state"] = {k: v.clone() for k, v in model.state_dict().items()}
    fx["container_types"] = {n: type(m).__name__ for n, m in model.named_children()}
    xk = torch.randn(4, 5, 24, generator=g, requires_grad=True)          # batch 4 = [2 negative | 2 positive]
    xf = torch.randn(4, 5, 32, generator=g, requires_grad=True)
    xc = torch.randn(2, 8, 8, 8, generator=g, requires_grad=True)
    outs = {"to_k": model.to_k(xk), "ff": model.ff(xf), "conv": model.conv(xc), "conv_s2": model.conv_s2(xc), "proj": model.proj(xc)}
    loss = sum((o ** 2).sum() for o in outs.values())
    loss.backward()
    fx["xk"], fx["xf"], fx["xc"] = xk.detach().clone(), xf.detach().clone(), xc.detach().clone()
    fx["outs"] = {k: v.detach().clone() for k, v in outs.items()}
    fx["grad_in"] = {"xk": xk.grad.clone(), "xf": xf.grad.clone(), "xc": xc.grad.clone()}
    fx["grads"] = {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None and "lora_block" in n}
    torch.save(fx, os.path.join(HERE, "ref_lora_dapp_conv.pt"))
    print("ref_lora_dapp_conv.pt:", fx["container_types"], len(fx["grads"]), "lora grads")


def make_wrap_layer():
    """LoraLayer.wrap_layer on a biased Linear (rank 8, alpha 2.0, random W_up): host weights, adapter weights, input and the
    output of the REAL reference layer."""
    plugin, base, layers = import_reference_lora()
    torch.manual_seed(3)
    holder = nn.Module()
    holder.lin = nn.Linear(40, 24, bias=True)
    blk = layers.LoraLayer.wrap_layer(0, holder.lin, rank=8, alpha=2.0, parent_block=holder, host_name="lin")
    with torch.no_grad():
        blk.layer.W_up.normal_(0, 0.1)
    x = torch.randn(5, 40)
    with torch.no_grad():
        out = holder.lin(x)
    fx = {"weight": holder.lin._host.weight.detach().clone(), "bias": holder.lin._host.bias.detach().clone(),
          "W_down": blk.layer.W_down.detach().clone(), "W_up": blk.layer.W_up.detach().clone(), "alpha": float(blk.alpha),
          "x": x, "out": out.clone()}
    torch.save(fx, os.path.join(HERE, "ref_lora_wrap_layer.pt"))
    print("ref_lora_wrap_layer.pt: alpha", fx["alpha"], "out", tuple(out.shape))


def make_webui_keys():
    """Key maps of the REAL reference LoraConverter (hcpdiff/tools/lora_convert.py) for the SD1.5 attention + ff LoRA layers."""
    import_reference_lora()
    ck = types.ModuleType("hcpdiff.ckpt_manager")
    ck.auto_manager = lambda path: None
    sys.modules["hcpdiff.ckpt_manager"] = ck
    for name, path in (("hcpdiff.tools", "hcpdiff/tools"), ("hcpdiff.deprecated", "hcpdiff/deprecated")):
        m = types.ModuleType(name)
        m.__path__ = [os.path.join(REF, path)]
        sys.modules[name] = m
    dep = importlib.import_module("hcpdiff.deprecated.lora_convert")
    sys.modules["hcpdiff.deprecated"].convert_to_webui_maybe_old = dep.convert_to_webui_maybe_old
    sys.modules["hcpdiff.deprecated"].convert_to_webui_xl_maybe_old = dep.convert_to_webui_xl_maybe_old
    conv = importlib.import_module("hcpdiff.tools.lora_convert").LoraConverter()
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from oracle import unet_ref as U
    layers = U.lora_target_layers(U.SD15, r".*\.attn.?$|.*\.ff$")
    shapes = U.param_shapes(U.SD15)
    sd = {}
    for i, layer in enumerate(layers):
        o, k = shapes[layer + ".weight"]
        sd[f"{layer}.___.layer.W_down"] = torch.full((4, 2), float(i))         # tiny stand-ins: only names and the scale rule matter
        sd[f"{layer}.___.layer.W_up"] = torch.full((2, 4), float(i) + 0.5)
        sd[f"{layer}.___.alpha"] = torch.tensor(0.25)
    te = {"text_model.encoder.layers.0.self_attn.q_proj.___.layer.W_down": torch.ones(4, 2),
          "text_model.encoder.layers.0.self_attn.q_proj.___.layer.W_up": torch.ones(2, 4),
          "text_model.encoder.layers.0.self_attn.q_proj.___.alpha": torch.tensor(0.5),
          "text_model.encoder.layers.11.mlp.fc1.___.layer.W_down": torch.ones(4, 2),
          "text_model.encoder.layers.11.mlp.fc1.___.layer.W_up": torch.ones(2, 4),
          "text_model.encoder.layers.11.mlp.fc1.___.alpha": torch.tensor(0.5)}
    web = conv.convert_to_webui(dict(sd), dict(te), auto_scale_alpha=False)
    web_scaled = conv.convert_to_webui(dict(sd), dict(te), auto_scale_alpha=True)
    back_te, back_unet = conv.convert_from_webui(dict(web), auto_scale_alpha=False)
    fx = {"to_webui": {k: wk for k, wk in zip(list(sd) + list(te), web.keys())},
          "from_webui_unet": sorted(back_unet["lora"].keys()), "from_webui_te": sorted(back_te["lora"].keys()),
          "scaled_sample": {k: [float(x) for x in web_scaled[k].flatten()[:2]] for k in list(web_scaled)[:6]},
          "hcp_keys": list(sd) + list(te)}
    assert sorted(back_unet["lora"].keys()) == sorted(sd.keys())
    with open(os.path.join(HERE, "lora_webui_keys.json"), "w") as f:
        json.dump(fx, f, indent=0)
    print("lora_webui_keys.json:", len(fx["to_webui"]), "keys; sample", list(fx["to_webui"].items())[0])


def _load_by_path(name, rel):
    import importlib.util
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def make_step():
    """Loss / EMA / CFG-context / cfg-range vectors of the real reference, plus DAPP on a 3x3 convolution."""
    sys.dont_write_bytecode = True
    if "diffusers" not in sys.modules:                       # min_snr_loss.py only needs the name for a type annotation
        d = types.ModuleType("diffusers")
        d.SchedulerMixin = type("SchedulerMixin", (), {})
        sys.modules["diffusers"] = d
    if "omegaconf" not in sys.modules:                       # utils.py imports the names at module level; get_cfg_range does not use them
        o = types.ModuleType("omegaconf")
        o.OmegaConf = type("OmegaConf", (), {})
        o.ListConfig = type("ListConfig", (), {})
        sys.modules["omegaconf"] = o
    loss_mod = _load_by_path("_ref_min_snr_loss", "hcpdiff/loss/min_snr_loss.py")
    ema_mod = _load_by_path("_ref_ema", "hcpdiff/utils/ema.py")
    ctx_mod = _load_by_path("_ref_cfg_context", "hcpdiff/models/cfg_context.py")
    utils_mod = _load_by_path("_ref_utils", "hcpdiff/utils/utils.py")
    g = torch.Generator().manual_seed(11)
    fx = {}
    # --- losses: scheduler stand-in carrying the SD1.5 scaled-linear alphas_cumprod (what DDPMScheduler holds)
    betas = torch.linspace(0.00085 ** 0.5, 0.012 ** 0.5, 1000, dtype=torch.float32) ** 2
    sched = types.SimpleNamespace(alphas_cumprod=torch.cumprod(1.0 - betas, dim=0))
    pred = torch.randn(6, 4, 8, 8, generator=g)
    target = torch.randn(6, 4, 8, 8, generator=g)
    t = torch.tensor([0, 17, 250, 499, 873, 999])
    fx["loss"] = {"pred": pred, "target": target, "t": t, "out": {}}
    for cls, gamma in (("MinSNRLoss", 5.0), ("MinSNRLoss", 1.0), ("SoftMinSNRLoss", 2.0), ("KDiffMinSNRLoss", 1.0), ("EDMLoss", 1.0)):
        crit = getattr(loss_mod, cls)(gamma=gamma, noise_scheduler=sched, device="cpu")
        p = pred.clone().requires_grad_(True)
        per_elem = crit(p.float(), target.float(), t)           # reduction 'none' (train_base.yaml:29), then .mean() in get_loss
        loss = per_elem.mean()
        loss.backward()
        fx["loss"]["out"][f"{cls}:{gamma}"] = {"loss": loss.detach().clone(), "dpred": p.grad.clone()}
    # --- ModelEMA: 6 updates of a 2-parameter module (+ a buffer) with the ema.yaml hyper-parameters and the defaults
    class M(nn.Module):
        def __init__(self):
            super().__init__()
            self.a = nn.Parameter(torch.randn(5, 3, generator=g))
            self.b = nn.Parameter(torch.randn(7, generator=g))
            self.frozen = nn.Parameter(torch.randn(2, generator=g), requires_grad=False)
            self.register_buffer("alpha", torch.tensor(0.125))
    fx["ema"] = []
    for kw in ({"decay_max": 0.9997, "power": 0.85}, {}, {"decay_max": 0.5, "inv_gamma": 2.0, "power": 0.75}):
        m = M()
        ema = ema_mod.ModelEMA(m, **kw)
        # ModelEMA keeps `p.data.to(device)`: with model and EMA on the same device that is an ALIAS of the live parameter (in
        # training the model is on the GPU and the EMA on the CPU, a real copy) -- give the EMA its own storage like there
        ema.train_params = {k: v.clone() for k, v in ema.train_params.items()}
        traj = {"kw": kw, "init": {k: v.detach().clone() for k, v in m.named_parameters()}, "params": [], "ema": []}
        for _ in range(6):
            with torch.no_grad():
                m.a.add_(torch.randn(m.a.shape, generator=g) * 0.1)
                m.b.add_(torch.randn(m.b.shape, generator=g) * 0.1)
            ema.update(m)
            traj["params"].append({"a": m.a.detach().clone(), "b": m.b.detach().clone()})
            traj["ema"].append({k: v.clone() for k, v in ema.state_dict().items()})
        fx["ema"].append(traj)
    # --- DreamArtistPTContext
    fx["cfg"] = []
    for text in ("3.0", "1.0-3.0:cos", "1.5-4.0:cos2", "2.0-5.0:ln", "1.0-3.0"):
        rng = utils_mod.get_cfg_range(text)
        ctx = ctx_mod.DreamArtistPTContext(rng, 1000)
        lat = torch.randn(3, 4, 8, 8, generator=g)
        ts = torch.tensor([5, 500, 999])
        lat2, ts2 = ctx.pre(lat, ts)
        eps2 = torch.randn(6, 4, 8, 8, generator=g, requires_grad=True)
        out = ctx.post(eps2)
        dout = torch.randn(out.shape, generator=g)
        out.backward(dout)
        fx["cfg"].append({"text": text, "range": rng, "lat": lat, "t": ts, "lat2": lat2.clone(), "t2": ts2.clone(), "eps2": eps2.detach().clone(),
                          "out": out.detach().clone(), "dout": dout, "deps2": eps2.grad.clone()})
    # --- DAPP on a 3x3 convolution
    plugin, base, layers = import_reference_lora()
    class Net(nn.Module):
        def __init__(self):
            super().__init__()
            self.conv = nn.Conv2d(8, 16, 3, padding=1)
            self.conv_s2 = nn.Conv2d(8, 8, 3, stride=2, padding=1)
    torch.manual_seed(3)
    net = Net().float()
    blocks = {}
    for lname in ("conv", "conv_s2"):
        for lora_id, (branch, rank) in enumerate((("p", 4), ("n", 2))):
            blk = layers.DAPPLayer.wrap_layer(lora_id, getattr(net, lname), rank=rank, dropout=0.0, alpha=1.0, branch=branch, parent_block=net,
                                              host_name=lname)
            with torch.no_grad():
                blk.layer.W_up.copy_(torch.randn(blk.layer.W_up.shape, generator=g) * 0.2)
            blocks[f"{lname}.{branch}"] = blk
    x = torch.randn(4, 8, 8, 8, generator=g, requires_grad=True)             # [2 negative | 2 positive]
    outs = {"conv": net.conv(x), "conv_s2": net.conv_s2(x)}
    sum((o ** 2).sum() for o in outs.values()).backward()
    fx["dapp_conv"] = {"state": {k: v.detach().clone() for k, v in net.state_dict().items()}, "x": x.detach().clone(),
                       "outs": {k: v.detach().clone() for k, v in outs.items()}, "dx": x.grad.clone(),
                       "grads": {n: p.grad.clone() for n, p in net.named_parameters() if p.grad is not None and "lora_block" in n},
                       "container_types": {n: type(m).__name__ for n, m in net.named_children()}}
    torch.save(fx, os.path.join(HERE, "ref_step.pt"))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "step":
        make_step()
        sys.exit(0)
    make_struct()
    make_lora()
    make_dapp_conv()
    make_wrap_layer()
    make_step()
    make_webui_keys()
