"""CPU oracle for the UNet denoising hot path -- TEST INFRASTRUCTURE, not product code.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu-baseline / ``--impl reference`` legs may import
this module; the product package (``hcp_diffusion_b200``) never does.

What it restates
----------------
The arithmetic of HCP-Diffusion's hot path ``noise_pred = unet(noisy_latents, t, encoder_hidden_states).sample``
(call site: reference ``hcpdiff/models/wrapper.py:29`` reached from ``hcpdiff/train_ac.py:454``) lives in the third-party
package ``diffusers`` (pinned ``diffusers<=0.26.1``, reference ``requirements.txt:4``), which is NOT vendored in the
reference tree and NOT installable here (no network).  This file is a from-scratch, functional, fp32 restatement of
``diffusers.UNet2DConditionModel.forward`` for the SD1.5 topology, driven by a flat ``{name: tensor}`` state dict whose
keys are the diffusers parameter names.  Structure follows the reference's module dump ``cfgs/unet_struct.txt:1-932``
(every module, shape, eps, bias flag, kernel/stride/padding) and the diffusers<->LDM index map
``hcpdiff/tools/diffusers2sd.py:17-110``; data flow follows the published diffusers 0.26 algorithm (SURVEY.md App. A).

LoRA semantics follow the reference operator exactly (``hcpdiff/models/lora_base_patch.py:21-35,61-74`` and
``hcpdiff/models/lora_layers_patch.py:44-57``): for every patched Linear, ``W' = W_host + sum_blocks alpha_b *
(W_up_b @ W_down_b)`` is MATERIALISED and ``y = x @ W'^T + b``.  ``tests/test_oracle.py`` checks this against the
committed golden vectors generated from the real reference classes (``tests/golden/make_golden.py``).

PARITY PINNING: the LoRA operator is pinned to the reference's own code; the UNet data flow is **parity unpinned** by the
reference (it ships no tests, no golden vectors and not the diffusers code) -- it is defended structurally only
(parameter names/shapes == ``cfgs/unet_struct.txt``, 859,520,964 parameters).
"""
from __future__ import annotations

import math
import re
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple, Union

import torch
import torch.nn.functional as F

Tensor = torch.Tensor


@dataclass(frozen=True)
class UNetSpec:
    """Architecture hyper-parameters (defaults = SD1.5, reference cfgs/unet_struct.txt).  The SDXL fields follow the diffusers
    config of stable-diffusion-xl-base-1.0 (the reference only ever sees it through `UNet2DConditionModel.from_pretrained` and
    the `added_cond_kwargs` of hcpdiff/models/wrapper.py:57-75): restated from knowledge, parity unpinned like the SD1.5 flow."""
    in_channels: int = 4
    out_channels: int = 4
    block_out_channels: Tuple[int, ...] = (320, 640, 1280, 1280)
    layers_per_block: int = 2
    num_heads: Union[int, Tuple[int, ...]] = 8   # diffusers' `attention_head_dim` is the HEAD COUNT (per level for SDXL)
    cross_attention_dim: int = 768
    norm_groups: int = 32
    # which down blocks carry transformers (SD1.5: first three)
    down_has_attn: Tuple[bool, ...] = (True, True, True, False)
    resnet_eps: float = 1e-5                # unet_struct.txt:93
    transformer_norm_eps: float = 1e-6      # unet_struct.txt:13
    layernorm_eps: float = 1e-5             # unet_struct.txt:44
    sample_size: int = 64
    transformer_depth: Union[int, Tuple[int, ...]] = 1     # BasicTransformerBlocks per Transformer2DModel, per level
    use_linear_projection: bool = False     # proj_in / proj_out are nn.Linear on the token matrix (SDXL) instead of 1x1 convs
    addition_time_embed_dim: Optional[int] = None          # SDXL 'text_time' additional embedding: sinusoid width per time id
    projection_class_embeddings_input_dim: Optional[int] = None   # text_embeds dim + 6 * addition_time_embed_dim

    @property
    def time_embed_dim(self) -> int:
        return self.block_out_channels[0] * 4

    @property
    def up_has_attn(self) -> Tuple[bool, ...]:
        return tuple(reversed(self.down_has_attn))

    def heads(self, level: int) -> int:
        return self.num_heads if isinstance(self.num_heads, int) else self.num_heads[level]

    def depth(self, level: int) -> int:
        return self.transformer_depth if isinstance(self.transformer_depth, int) else self.transformer_depth[level]


SD15 = UNetSpec()
# a small topology with the same block structure, for tests that must finish in seconds
TINY = UNetSpec(block_out_channels=(64, 128, 128, 128), num_heads=2, cross_attention_dim=64, sample_size=16)
# stable-diffusion-xl-base-1.0: three levels, no attention at the top one, transformer depth 2 / 10, head dim 64 everywhere,
# linear projections, 2048-wide text context, (pooled text | 6 sinusoidal time ids) additional embedding
SDXL = UNetSpec(block_out_channels=(320, 640, 1280), num_heads=(5, 10, 20), cross_attention_dim=2048,
                down_has_attn=(False, True, True), sample_size=128, transformer_depth=(1, 2, 10), use_linear_projection=True,
                addition_time_embed_dim=256, projection_class_embeddings_input_dim=2816)
TINY_XL = UNetSpec(block_out_channels=(64, 128, 128), num_heads=(1, 2, 2), cross_attention_dim=64, down_has_attn=(False, True, True),
                   sample_size=16, transformer_depth=(1, 2, 3), use_linear_projection=True, addition_time_embed_dim=32,
                   projection_class_embeddings_input_dim=256)


# ----------------------------------------------------------------------------------------------------------------------
# parameter inventory (names + shapes), in diffusers naming
# ----------------------------------------------------------------------------------------------------------------------
def _resnet_params(prefix: str, cin: int, cout: int, temb: int) -> List[Tuple[str, Tuple[int, ...]]]:
    p = [
        (f"{prefix}.norm1.weight", (cin,)), (f"{prefix}.norm1.bias", (cin,)),
        (f"{prefix}.conv1.weight", (cout, cin, 3, 3)), (f"{prefix}.conv1.bias", (cout,)),
        (f"{prefix}.time_emb_proj.weight", (cout, temb)), (f"{prefix}.time_emb_proj.bias", (cout,)),
        (f"{prefix}.norm2.weight", (cout,)), (f"{prefix}.norm2.bias", (cout,)),
        (f"{prefix}.conv2.weight", (cout, cout, 3, 3)), (f"{prefix}.conv2.bias", (cout,)),
    ]
    if cin != cout:
        p += [(f"{prefix}.conv_shortcut.weight", (cout, cin, 1, 1)), (f"{prefix}.conv_shortcut.bias", (cout,))]
    return p


def _transformer_params(prefix: str, c: int, ctx: int, depth: int = 1, linear_proj: bool = False) -> List[Tuple[str, Tuple[int, ...]]]:
    proj = (c, c) if linear_proj else (c, c, 1, 1)
    p = [
        (f"{prefix}.norm.weight", (c,)), (f"{prefix}.norm.bias", (c,)),
        (f"{prefix}.proj_in.weight", proj), (f"{prefix}.proj_in.bias", (c,)),
    ]
    for k in range(depth):
        tb = f"{prefix}.transformer_blocks.{k}"
        for attn, kdim in (("attn1", c), ("attn2", ctx)):
            p += [
                (f"{tb}.{attn}.to_q.weight", (c, c)),
                (f"{tb}.{attn}.to_k.weight", (c, kdim)),
                (f"{tb}.{attn}.to_v.weight", (c, kdim)),
                (f"{tb}.{attn}.to_out.0.weight", (c, c)), (f"{tb}.{attn}.to_out.0.bias", (c,)),
            ]
        p += [
            (f"{tb}.ff.net.0.proj.weight", (8 * c, c)), (f"{tb}.ff.net.0.proj.bias", (8 * c,)),
            (f"{tb}.ff.net.2.weight", (c, 4 * c)), (f"{tb}.ff.net.2.bias", (c,)),
        ]
        for n in ("norm1", "norm2", "norm3"):
            p += [(f"{tb}.{n}.weight", (c,)), (f"{tb}.{n}.bias", (c,))]
    p += [(f"{prefix}.proj_out.weight", proj), (f"{prefix}.proj_out.bias", (c,))]
    return p


def param_shapes(spec: UNetSpec = SD15) -> Dict[str, Tuple[int, ...]]:
    """Every parameter of the UNet, diffusers names -> shape (follows cfgs/unet_struct.txt)."""
    ch = spec.block_out_channels
    temb = spec.time_embed_dim
    out: List[Tuple[str, Tuple[int, ...]]] = [
        ("conv_in.weight", (ch[0], spec.in_channels, 3, 3)), ("conv_in.bias", (ch[0],)),
        ("time_embedding.linear_1.weight", (temb, ch[0])), ("time_embedding.linear_1.bias", (temb,)),
        ("time_embedding.linear_2.weight", (temb, temb)), ("time_embedding.linear_2.bias", (temb,)),
    ]
    if spec.addition_time_embed_dim:
        out += [("add_embedding.linear_1.weight", (temb, spec.projection_class_embeddings_input_dim)), ("add_embedding.linear_1.bias", (temb,)),
                ("add_embedding.linear_2.weight", (temb, temb)), ("add_embedding.linear_2.bias", (temb,))]
    lin = spec.use_linear_projection
    skip_ch = [ch[0]]
    cprev = ch[0]
    nblk = len(ch)
    for i, c in enumerate(ch):
        for j in range(spec.layers_per_block):
            out += _resnet_params(f"down_blocks.{i}.resnets.{j}", cprev, c, temb)
            if spec.down_has_attn[i]:
                out += _transformer_params(f"down_blocks.{i}.attentions.{j}", c, spec.cross_attention_dim, spec.depth(i), lin)
            cprev = c
            skip_ch.append(c)
        if i < nblk - 1:
            out += [(f"down_blocks.{i}.downsamplers.0.conv.weight", (c, c, 3, 3)),
                    (f"down_blocks.{i}.downsamplers.0.conv.bias", (c,))]
            skip_ch.append(c)
    cm = ch[-1]
    out += _resnet_params("mid_block.resnets.0", cm, cm, temb)
    out += _transformer_params("mid_block.attentions.0", cm, spec.cross_attention_dim, spec.depth(nblk - 1), lin)
    out += _resnet_params("mid_block.resnets.1", cm, cm, temb)
    rev = list(reversed(ch))
    cprev = cm
    for i, c in enumerate(rev):
        for j in range(spec.layers_per_block + 1):
            cskip = skip_ch.pop()
            out += _resnet_params(f"up_blocks.{i}.resnets.{j}", cprev + cskip, c, temb)
            if spec.up_has_attn[i]:
                out += _transformer_params(f"up_blocks.{i}.attentions.{j}", c, spec.cross_attention_dim, spec.depth(nblk - 1 - i), lin)
            cprev = c
        if i < nblk - 1:
            out += [(f"up_blocks.{i}.upsamplers.0.conv.weight", (c, c, 3, 3)),
                    (f"up_blocks.{i}.upsamplers.0.conv.bias", (c,))]
    out += [("conv_norm_out.weight", (ch[0],)), ("conv_norm_out.bias", (ch[0],)),
            ("conv_out.weight", (spec.out_channels, ch[0], 3, 3)), ("conv_out.bias", (spec.out_channels,))]
    return dict(out)


def init_params(spec: UNetSpec = SD15, seed: int = 0, dtype=torch.float32) -> Dict[str, Tensor]:
    """Deterministic synthetic weights (SURVEY.md 8d): conv/linear ~ N(0, 1/fan_in); norm gamma = 1 + 0.02 N(0,1),
    beta = 0.02 N(0,1); biases 0.02 N(0,1).  Independent of parameter order (each tensor has its own seed)."""
    sd: Dict[str, Tensor] = {}
    for idx, (name, shape) in enumerate(param_shapes(spec).items()):
        g = torch.Generator().manual_seed(seed * 1_000_003 + idx)
        is_norm = re.search(r"(^|\.)(norm\d?|conv_norm_out)\.(weight|bias)$", name) is not None
        if name.endswith(".weight") and not is_norm:
            fan_in = 1
            for s in shape[1:]:
                fan_in *= s
            t = torch.randn(shape, generator=g) * (1.0 / math.sqrt(fan_in))
        elif name.endswith(".weight"):
            t = 1.0 + 0.02 * torch.randn(shape, generator=g)
        else:
            t = 0.02 * torch.randn(shape, generator=g)
        sd[name] = t.to(dtype)
    return sd


# ----------------------------------------------------------------------------------------------------------------------
# LoRA (reference semantics: materialise W' = W + sum alpha * up @ down)
# ----------------------------------------------------------------------------------------------------------------------
@dataclass
class LoraEntry:
    """One LoRA block on one layer.  Linear: W_down [r,in], W_up [out,r]; Conv2d (lora_layers_patch.py:64-100): W_down
    [r,in,kh,kw], W_up [out,r,1,1].  alpha = alpha/rank (a scalar).  branch: None, or 'p' / 'n' for DreamArtist++ blocks."""
    W_down: Tensor
    W_up: Tensor
    alpha: float
    branch: Optional[str] = None


LoraDict = Dict[str, List[LoraEntry]]   # layer path (e.g. '...attn1.to_q') -> stacked blocks


def lora_target_layers(spec: UNetSpec = SD15, pattern: str = r".*\.attn.?$", include_conv: bool = False) -> List[str]:
    """Layers hit by a reference `layers: ['re:<pattern>']` item: every nn.Linear (and, with `include_conv`, nn.Conv2d --
    LoraBlock.wrapable_classes, lora_base_patch.py:39) below a module whose name matches (reference
    hcpdiff/utils/cfg_net_tools.py:30-75 + plugin.py:297-315)."""
    rx = re.compile(pattern)
    names = []
    for k, shp in param_shapes(spec).items():
        if not k.endswith(".weight") or not (len(shp) == 2 or (include_conv and len(shp) == 4)):
            continue
        layer = k[: -len(".weight")]
        parts = layer.split(".")
        # any proper-or-equal prefix of the layer path that matches the pattern makes the layer a target
        if any(rx.match(".".join(parts[:n])) for n in range(1, len(parts) + 1)):
            names.append(layer)
    return names


def init_lora(spec: UNetSpec = SD15, rank: int = 8, alpha: float = 1.0, seed: int = 1, up_std: float = 0.02,
              pattern: str = r".*\.attn.?$", include_conv: bool = False, branch: Optional[str] = None) -> LoraDict:
    """W_down: kaiming-uniform(a=sqrt5) like the reference init (lora_layers_patch.py:38-42); W_up ~ N(0, up_std) so the
    delta does not vanish in parity tests (up_std=0 reproduces the reference's zero init)."""
    shapes = param_shapes(spec)
    out: LoraDict = {}
    for idx, layer in enumerate(lora_target_layers(spec, pattern, include_conv)):
        shp = shapes[layer + ".weight"]
        o, i = shp[0], shp[1]
        g = torch.Generator().manual_seed(seed * 7_000_003 + idx)
        fan_in = i * (shp[2] * shp[3] if len(shp) == 4 else 1)
        bound = 1.0 / math.sqrt(fan_in)     # kaiming_uniform(a=sqrt(5)) on [r, in(, kh, kw)]
        down = (torch.rand((rank, *shp[1:]), generator=g) * 2 - 1) * bound
        up = torch.randn((o, rank) if len(shp) == 2 else (o, rank, 1, 1), generator=g) * up_std
        out[layer] = [LoraEntry(down, up, alpha / rank, branch)]
    return out


def lora_delta(entries: List[LoraEntry], branch: Optional[str] = None) -> Optional[Tensor]:
    """sum of alpha * W_up . W_down over the blocks of one layer (of one DAPP branch when `branch` is given)."""
    dw = None
    for e in entries:
        if branch is not None and e.branch != branch:
            continue
        if e.W_down.dim() == 2:
            d = torch.mm(e.W_up, e.W_down) * e.alpha       # lora_layers_patch.py:44-45, lora_base_patch.py:61-62
        else:                                              # einsum('o r ..., r i ... -> o i ...'), lora_layers_patch.py:91-92
            d = torch.einsum("or,rikl->oikl", e.W_up[:, :, 0, 0], e.W_down) * e.alpha
        dw = d if dw is None else dw + d                   # lora_base_patch.py:24-28
    return dw


def _mm(x: Tensor, w: Tensor, b: Optional[Tensor]) -> Tensor:
    shp = x.shape
    y = torch.mm(x.reshape(-1, shp[-1]), w.transpose(0, 1)).view(*shp[:-1], -1)   # lora_layers_patch.py:50-57
    return y if b is None else y + b


def _linear(sd: Dict[str, Tensor], lora: Optional[LoraDict], name: str, x: Tensor) -> Tensor:
    w = sd[name + ".weight"]
    b = sd.get(name + ".bias")
    entries = lora.get(name) if lora is not None else None
    if entries and any(e.branch is not None for e in entries):
        # DAPPPatchContainer.forward (lora_layers_patch.py:102-133): x = [negative half | positive half]
        B = x.shape[0] // 2
        y_p = _mm(x[B:], w + lora_delta(entries, "p"), b)
        y_n = _mm(x[:B], w + lora_delta(entries, "n"), b)
        return torch.cat([y_n, y_p], dim=0)
    if entries:
        w = w + lora_delta(entries)                        # lora_base_patch.py:74 (host_weight + weight)
    return _mm(x, w, b)


def _conv(sd: Dict[str, Tensor], lora: Optional[LoraDict], name: str, x: Tensor, stride: int = 1, padding: int = 0) -> Tensor:
    """F.conv2d(x, W_host + delta, b) -- LoraLayer.Conv2dLayer.forward (lora_layers_patch.py:97-98) for patched convolutions."""
    w = sd[name + ".weight"]
    b = sd.get(name + ".bias")
    entries = lora.get(name) if lora is not None else None
    if entries and any(e.branch is not None for e in entries):
        # DAPPPatchContainer.forward on a Conv2d host (lora_layers_patch.py:102-133): x = [negative half | positive half]
        B = x.shape[0] // 2
        y_p = F.conv2d(x[B:], w + lora_delta(entries, "p"), b, stride=stride, padding=padding)
        y_n = F.conv2d(x[:B], w + lora_delta(entries, "n"), b, stride=stride, padding=padding)
        return torch.cat([y_n, y_p], dim=0)
    if entries:
        w = w + lora_delta(entries)
    return F.conv2d(x, w, b, stride=stride, padding=padding)


# ----------------------------------------------------------------------------------------------------------------------
# forward
# ----------------------------------------------------------------------------------------------------------------------
def timestep_embedding(t: Tensor, dim: int) -> Tensor:
    """diffusers get_timestep_embedding(flip_sin_to_cos=True, downscale_freq_shift=0): [cos | sin]."""
    half = dim // 2
    freqs = torch.exp(-math.log(10000.0) * torch.arange(half, dtype=torch.float32) / half)
    a = t.float()[:, None] * freqs[None]
    return torch.cat([torch.cos(a), torch.sin(a)], dim=-1)


def _resnet(sd, p: str, x: Tensor, emb: Tensor, spec: UNetSpec, lora=None) -> Tensor:
    h = F.group_norm(x, spec.norm_groups, sd[p + ".norm1.weight"], sd[p + ".norm1.bias"], spec.resnet_eps)
    h = _conv(sd, lora, p + ".conv1", F.silu(h), padding=1)
    t = _linear(sd, lora, p + ".time_emb_proj", F.silu(emb))
    h = h + t[:, :, None, None]
    h = F.group_norm(h, spec.norm_groups, sd[p + ".norm2.weight"], sd[p + ".norm2.bias"], spec.resnet_eps)
    h = _conv(sd, lora, p + ".conv2", F.silu(h), padding=1)
    if (p + ".conv_shortcut.weight") in sd:
        x = _conv(sd, lora, p + ".conv_shortcut", x)
    return x + h


def _attention(sd, lora, p: str, x: Tensor, ctx: Tensor, bias: Optional[Tensor], heads: int) -> Tensor:
    q = _linear(sd, lora, p + ".to_q", x)
    k = _linear(sd, lora, p + ".to_k", ctx)
    v = _linear(sd, lora, p + ".to_v", ctx)
    B, L, C = q.shape
    d = C // heads
    q = q.view(B, L, heads, d).transpose(1, 2)
    k = k.view(B, -1, heads, d).transpose(1, 2)
    v = v.view(B, -1, heads, d).transpose(1, 2)
    s = torch.matmul(q, k.transpose(-1, -2)) / math.sqrt(d)
    if bias is not None:
        s = s + bias[:, None, :, :]
    o = torch.matmul(torch.softmax(s, dim=-1), v)
    o = o.transpose(1, 2).reshape(B, L, C)
    return _linear(sd, lora, p + ".to_out.0", o)


def _transformer(sd, lora, p: str, x: Tensor, ehs: Tensor, bias: Optional[Tensor], spec: UNetSpec, level: int = 0) -> Tensor:
    """Transformer2DModel: GroupNorm, proj_in, `depth` BasicTransformerBlocks, proj_out, residual.  With
    `use_linear_projection` (SDXL) proj_in / proj_out are Linear layers on the token matrix, applied after / before the
    NCHW <-> token reshape; otherwise 1x1 convolutions applied before / after it."""
    B, C, H, W = x.shape
    heads = spec.heads(level)
    res = x
    h = F.group_norm(x, spec.norm_groups, sd[p + ".norm.weight"], sd[p + ".norm.bias"], spec.transformer_norm_eps)
    if spec.use_linear_projection:
        h = h.permute(0, 2, 3, 1).reshape(B, H * W, C)
        h = _linear(sd, lora, p + ".proj_in", h)
    else:
        h = _conv(sd, lora, p + ".proj_in", h)
        h = h.permute(0, 2, 3, 1).reshape(B, H * W, C)
    for k in range(spec.depth(level)):
        tb = f"{p}.transformer_blocks.{k}"
        n = F.layer_norm(h, (C,), sd[tb + ".norm1.weight"], sd[tb + ".norm1.bias"], spec.layernorm_eps)
        h = _attention(sd, lora, tb + ".attn1", n, n, None, heads) + h
        n = F.layer_norm(h, (C,), sd[tb + ".norm2.weight"], sd[tb + ".norm2.bias"], spec.layernorm_eps)
        h = _attention(sd, lora, tb + ".attn2", n, ehs, bias, heads) + h
        n = F.layer_norm(h, (C,), sd[tb + ".norm3.weight"], sd[tb + ".norm3.bias"], spec.layernorm_eps)
        u = _linear(sd, lora, tb + ".ff.net.0.proj", n)
        a, g = u.chunk(2, dim=-1)
        h = _linear(sd, lora, tb + ".ff.net.2", a * F.gelu(g)) + h
    if spec.use_linear_projection:
        h = _linear(sd, lora, p + ".proj_out", h)
        h = h.reshape(B, H, W, C).permute(0, 3, 1, 2)
        return h + res
    h = h.reshape(B, H, W, C).permute(0, 3, 1, 2)
    return _conv(sd, lora, p + ".proj_out", h) + res


def unet_forward(sd: Dict[str, Tensor], sample: Tensor, timestep: Tensor, encoder_hidden_states: Tensor,
                 encoder_attention_mask: Optional[Tensor] = None, lora: Optional[LoraDict] = None,
                 spec: UNetSpec = SD15, added_cond_kwargs: Optional[Dict[str, Tensor]] = None) -> Tensor:
    """noise_pred [B, out_ch, H, W] for sample [B,4,H,W], timestep [B] (or scalar), ehs [B,Lc,ctx]."""
    B = sample.shape[0]
    bias = None
    if encoder_attention_mask is not None:
        # diffusers convention, restated in the reference at hcpdiff/models/controlnet.py:99-103
        bias = ((1 - encoder_attention_mask.to(sample.dtype)) * -10000.0)[:, None, :]
    t = torch.as_tensor(timestep)
    if t.dim() == 0:
        t = t[None]
    t = t.expand(B)
    emb = timestep_embedding(t, spec.block_out_channels[0]).to(sample.dtype)
    emb = F.linear(emb, sd["time_embedding.linear_1.weight"], sd["time_embedding.linear_1.bias"])
    emb = F.linear(F.silu(emb), sd["time_embedding.linear_2.weight"], sd["time_embedding.linear_2.bias"])
    if spec.addition_time_embed_dim:
        # SDXL 'text_time' (reference wrapper.py:66: added_cond_kwargs = {text_embeds: pooled CLIP-bigG output, time_ids: crop_info}):
        # aug = add_embedding(cat[text_embeds, sinusoid(time_ids).flatten]), emb = emb + aug
        te, ids = added_cond_kwargs["text_embeds"], added_cond_kwargs["time_ids"]
        tid = timestep_embedding(ids.flatten(), spec.addition_time_embed_dim).reshape(B, -1)
        add = torch.cat([te, tid.to(te.dtype)], dim=-1)
        aug = F.linear(add, sd["add_embedding.linear_1.weight"], sd["add_embedding.linear_1.bias"])
        aug = F.linear(F.silu(aug), sd["add_embedding.linear_2.weight"], sd["add_embedding.linear_2.bias"])
        emb = emb + aug

    h = _conv(sd, lora, "conv_in", sample, padding=1)
    skips = [h]
    nblk = len(spec.block_out_channels)
    for i in range(nblk):
        for j in range(spec.layers_per_block):
            h = _resnet(sd, f"down_blocks.{i}.resnets.{j}", h, emb, spec, lora)
            if spec.down_has_attn[i]:
                h = _transformer(sd, lora, f"down_blocks.{i}.attentions.{j}", h, encoder_hidden_states, bias, spec, i)
            skips.append(h)
        if i < nblk - 1:
            p = f"down_blocks.{i}.downsamplers.0.conv"
            h = _conv(sd, lora, p, h, stride=2, padding=1)
            skips.append(h)
    h = _resnet(sd, "mid_block.resnets.0", h, emb, spec, lora)
    h = _transformer(sd, lora, "mid_block.attentions.0", h, encoder_hidden_states, bias, spec, nblk - 1)
    h = _resnet(sd, "mid_block.resnets.1", h, emb, spec, lora)
    for i in range(nblk):
        for j in range(spec.layers_per_block + 1):
            h = torch.cat([h, skips.pop()], dim=1)
            h = _resnet(sd, f"up_blocks.{i}.resnets.{j}", h, emb, spec, lora)
            if spec.up_has_attn[i]:
                h = _transformer(sd, lora, f"up_blocks.{i}.attentions.{j}", h, encoder_hidden_states, bias, spec, nblk - 1 - i)
        if i < nblk - 1:
            p = f"up_blocks.{i}.upsamplers.0.conv"
            h = F.interpolate(h, scale_factor=2.0, mode="nearest")
            h = _conv(sd, lora, p, h, padding=1)
    h = F.group_norm(h, spec.norm_groups, sd["conv_norm_out.weight"], sd["conv_norm_out.bias"], spec.resnet_eps)
    return _conv(sd, lora, "conv_out", F.silu(h), padding=1)


# ----------------------------------------------------------------------------------------------------------------------
# the training step either side of the UNet call (reference train_ac.py:437-447, 449-465, 506-515)
# ----------------------------------------------------------------------------------------------------------------------
def ddpm_alphas_cumprod(num_steps: int = 1000, beta_start: float = 0.00085, beta_end: float = 0.012) -> Tensor:
    """SD1.5 'scaled_linear' schedule (reference tools/gen_from_ptlist.py:14-16 uses the same constants)."""
    betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_steps, dtype=torch.float32) ** 2
    return torch.cumprod(1.0 - betas, dim=0)


def add_noise(x0: Tensor, noise: Tensor, t: Tensor, acp: Tensor) -> Tensor:
    a = acp[t].sqrt()[:, None, None, None]
    s = (1 - acp[t]).sqrt()[:, None, None, None]
    return a * x0 + s * noise


def synthetic_batch(batch: int, spec: UNetSpec = SD15, seed: int = 1234, ctx_len: int = 77):
    """SURVEY.md 8d inputs: latents ~ N(0,1), noise ~ N(0,1), t ~ U{0..999}, ehs ~ N(0,1)."""
    g = torch.Generator().manual_seed(seed)
    s = spec.sample_size
    latents = torch.randn((batch, spec.in_channels, s, s), generator=g)
    noise = torch.randn((batch, spec.in_channels, s, s), generator=g)
    t = torch.randint(0, 1000, (batch,), generator=g, dtype=torch.int64)
    ehs = torch.randn((batch, ctx_len, spec.cross_attention_dim), generator=g)
    return latents, noise, t, ehs


def synthetic_added_cond(batch: int, spec: UNetSpec, seed: int = 4321) -> Optional[Dict[str, Tensor]]:
    """SDXL `added_cond_kwargs` with the statistics of the real inputs: pooled text embedding ~ N(0,1), time ids =
    (orig_h, orig_w, crop_top, crop_left, target_h, target_w) in pixels (reference data/pair_dataset crop_info)."""
    if not spec.addition_time_embed_dim:
        return None
    g = torch.Generator().manual_seed(seed)
    te_dim = spec.projection_class_embeddings_input_dim - 6 * spec.addition_time_embed_dim
    px = spec.sample_size * 8
    ids = torch.tensor([[px, px, 0, 0, px, px]], dtype=torch.float32).repeat(batch, 1)
    ids[:, 2:4] = torch.randint(0, 64, (batch, 2), generator=g).float()
    return {"text_embeds": torch.randn((batch, te_dim), generator=g), "time_ids": ids}


def lora_step_loss_and_grads(sd, lora: LoraDict, latents, noise, t, ehs, spec: UNetSpec = SD15, added_cond_kwargs=None):
    """One reference training forward/backward: eps-prediction MSE (train_ac.py:506-515, reduction mean) and the
    gradients of every LoRA parameter.  Returns (loss, noise_pred, {layer: [(dW_down, dW_up), ...]})."""
    leaves = []
    for layer, blocks in lora.items():
        for e in blocks:
            e.W_down.requires_grad_(True)
            e.W_up.requires_grad_(True)
            e.W_down.grad = None
            e.W_up.grad = None
            leaves += [e.W_down, e.W_up]
    x_t = add_noise(latents, noise, t, ddpm_alphas_cumprod())
    pred = unet_forward(sd, x_t, t, ehs, lora=lora, spec=spec, added_cond_kwargs=added_cond_kwargs)
    loss = F.mse_loss(pred.float(), noise.float(), reduction="none").mean()
    loss.backward()
    grads = {layer: [(e.W_down.grad.clone(), e.W_up.grad.clone()) for e in blocks] for layer, blocks in lora.items()}
    for p in leaves:
        p.requires_grad_(False)
        p.grad = None
    return loss.detach(), pred.detach(), grads


def ddim_cfg_sample(sd, latents: Tensor, prompt_embeds: Tensor, negative_embeds: Tensor, num_inference_steps: int, guidance_scale: float,
                    spec: UNetSpec = SD15, lora: Optional[LoraDict] = None, added_cond_kwargs=None, num_train_timesteps: int = 1000) -> Tensor:
    """The reference text-to-image denoising loop (hcpdiff/utils/pipe_hook.py:115-150) with the DDIM (eta = 0, leading spacing,
    steps_offset 1, set_alpha_to_one False) update, around the oracle UNet: one forward per step on [negative | positive]."""
    acp = ddpm_alphas_cumprod(num_train_timesteps)
    ratio = num_train_timesteps // num_inference_steps
    steps = (torch.arange(0, num_inference_steps) * ratio).flip(0) + 1
    x = latents.clone()
    B = x.shape[0]
    ehs2 = torch.cat([negative_embeds, prompt_embeds], 0)
    with torch.no_grad():
        for t in steps.tolist():
            t = min(t, num_train_timesteps - 1)
            tt = torch.full((2 * B,), t, dtype=torch.int64)
            eps2 = unet_forward(sd, torch.cat([x, x], 0), tt, ehs2, lora=lora, spec=spec, added_cond_kwargs=added_cond_kwargs)
            e_u, e_c = eps2.chunk(2)
            eps = e_u + guidance_scale * (e_c - e_u)
            a_t = acp[t]
            t_prev = t - ratio
            a_prev = acp[t_prev] if t_prev >= 0 else acp[0]
            x0 = (x - (1 - a_t).sqrt() * eps) / a_t.sqrt()
            x = a_prev.sqrt() * x0 + (1 - a_prev).sqrt() * eps
    return x
