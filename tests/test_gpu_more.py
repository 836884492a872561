"""More GPU parity tests (`pytest -m gpu`): UNet-level attention mask, LoRA dropout, DreamArtist++ on 3x3 convolutions, the
`train_ac` entrypoint (incl. resume into the trained blocks), and data-parallel NCCL parity on 2 GPUs."""
import math
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F
from torch import nn

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():          # fp32 torch references must be real fp32
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False

from hcp_diffusion_b200 import ops  # noqa: E402
from hcp_diffusion_b200.models import UNet2DConditionModel  # noqa: E402
from hcp_diffusion_b200.models.lora import DAPPLayer, LoraLayer  # noqa: E402
from hcp_diffusion_b200.utils.cfg_net_tools import make_hcpdiff  # noqa: E402
from oracle import unet_ref as U  # noqa: E402

DEV = "cuda"
BF = torch.bfloat16
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rel_l2(a, b):
    a, b = a.detach().double().flatten().cpu(), b.detach().double().flatten().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def tiny_unet(sd, spec=U.TINY):
    unet = UNet2DConditionModel(sample_size=spec.sample_size, block_out_channels=spec.block_out_channels,
                                attention_head_dim=spec.num_heads, cross_attention_dim=spec.cross_attention_dim)
    unet.load_state_dict(sd)
    return unet.to(DEV).requires_grad_(False).eval()


def test_unet_encoder_attention_mask_matches_oracle():
    """`unet(..., encoder_attention_mask=mask)` (reference wrapper.py:14-30; diffusers turns the mask into a (1 - m) * -10000 bias on
    the text keys of every cross-attention) against the oracle on the TINY topology, plus: masked tokens do not influence the output."""
    spec = U.TINY
    sd = U.init_params(spec)
    unet = tiny_unet(sd)
    lat, noise, t, ehs = U.synthetic_batch(3, spec, ctx_len=77)
    mask = torch.ones(3, 77)
    mask[0, 40:] = 0
    mask[1, 5:] = 0
    with torch.no_grad():
        ref = U.unet_forward(sd, lat, t, ehs, spec=spec, encoder_attention_mask=mask)
        ref_nomask = U.unet_forward(sd, lat, t, ehs, spec=spec)
        got = unet(lat.to(DEV), t.to(DEV), ehs.to(DEV), encoder_attention_mask=mask.to(DEV)).sample
        ehs2 = ehs.clone()
        ehs2[0, 40:] = 7.0                              # garbage in the masked positions must not matter
        got2 = unet(lat.to(DEV), t.to(DEV), ehs2.to(DEV), encoder_attention_mask=mask.to(DEV)).sample
    assert rel_l2(got, ref) < 2e-2
    assert rel_l2(ref, ref_nomask) > 1e-3              # the mask does something in the oracle
    assert rel_l2(got2[0], got[0]) < 1e-3


# ----------------------------------------------------------------------------------------------------------------------
# nn.Dropout on the patched layer output (reference lora_base_patch.py:74)
# ----------------------------------------------------------------------------------------------------------------------
def test_lora_dropout_properties_linear_and_conv():
    """The RNG stream cannot match torch's, so the test is by properties: every output element is either 0 or the p = 0 output
    / (1 - p); the keep rate is 1 - p; the backward applies the SAME mask; eval() turns it off; a new step draws a new mask."""
    torch.manual_seed(0)
    p = 0.25

    class Net(nn.Module):
        def __init__(self):
            super().__init__()
            self.lin = nn.Linear(320, 640)
            self.conv = nn.Conv2d(64, 128, 3, padding=1)
    net = Net().to(DEV).requires_grad_(False)
    blocks = {}
    for name in ("lin", "conv"):
        blk = LoraLayer.wrap_layer(0, getattr(net, name), rank=4, dropout=p, alpha=1.0, parent_block=net, host_name=name)
        nn.init.normal_(blk.layer.W_up, std=0.05)
        blocks[name] = blk
    ops.set_dropout_seed(1234)
    for name, x in (("lin", torch.randn(512, 320, device=DEV)), ("conv", torch.randn(2, 64, 16, 16, device=DEV))):
        layer, blk = getattr(net, name), blocks[name]
        blk.eval()
        y0 = layer(x)
        blk.train()
        xg = x.clone().requires_grad_(True)
        y1 = layer(xg)
        kept = y1 != 0
        rate = float(kept.float().mean())
        assert abs(rate - (1 - p)) < 0.02, (name, rate)
        assert rel_l2(y1[kept], y0[kept] / (1 - p)) < 1e-2
        dy = torch.randn_like(y1)
        y1.backward(dy)
        # reference gradient: d/dx of sum(dy * mask/(1-p) * layer_p0(x)) with the observed mask
        blk.eval()
        xr = x.clone().requires_grad_(True)
        (layer(xr) * dy * kept / (1 - p)).sum().backward()
        assert rel_l2(xg.grad, xr.grad) < 2e-2, name
        blk.train()
        ops.advance_dropout()
        y2 = layer(x)
        assert float(((y2 != 0) != kept).float().mean()) > 0.2      # a fresh mask after the draw counter moved
        ops.advance_dropout()


def test_tiny_unet_trains_with_dropout_under_cuda_graph():
    """DreamArtist++.yaml-style items (float rank, dropout 0.1, to_k / to_v / ff) through the captured step: finite, decreasing loss and
    a different mask on every replay (two replays on the SAME inputs give different losses)."""
    from hcp_diffusion_b200.engine import LoraTrainStep
    spec = U.TINY
    unet = tiny_unet(U.init_params(spec))
    groups, group = make_hcpdiff(unet, None, [{"lr": 1e-3, "rank": 0.0625, "dropout": 0.1,
                                               "layers": [r"re:.*\.to_k$", r"re:.*\.to_v$", r"re:.*\.ff$"]}])
    for blk in group.plugin_dict.values():
        nn.init.normal_(blk.layer.W_up, std=0.02)
    assert {b.rank for b in group.plugin_dict.values()} >= {4, 8}          # round(out_features * 0.0625)
    step = LoraTrainStep(unet, groups, use_cuda_graph=True)
    lat, noise, t, ehs = U.synthetic_batch(4, spec)
    step.set_lr(0.0)
    l0, l1 = float(step.step(lat, noise, t, ehs).cpu()), float(step.step(lat, noise, t, ehs).cpu())
    assert math.isfinite(l0) and l0 != l1                                    # lr 0: only the dropout mask changed
    step.set_lr(1e-3)
    losses = [float(step.step(lat, noise, t, ehs).cpu()) for _ in range(30)]
    assert all(math.isfinite(v) for v in losses) and sum(losses[-5:]) < sum(losses[:5])


# ----------------------------------------------------------------------------------------------------------------------
# DreamArtist++ blocks on 3x3 convolutions
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("stride", [1, 2])
def test_dapp_conv3x3_container_matches_oracle(stride):
    """DAPPPatchContainer on a 3x3 Conv2d host (batch = [negative | positive]) vs the oracle's `_conv` (pinned to the real reference
    DAPPLayer vectors by tests/test_oracle_step.py): output, input gradient and the gradients of both branches' factors."""
    torch.manual_seed(1)
    Cin, Cout, B, H = 64, 128, 4, 16

    class Net(nn.Module):
        def __init__(self):
            super().__init__()
            self.conv = nn.Conv2d(Cin, Cout, 3, stride=stride, padding=1)
    net = Net().to(DEV).requires_grad_(False)
    blocks = {}
    for lora_id, (branch, rank) in enumerate((("p", 4), ("n", 8))):
        blk = DAPPLayer.wrap_layer(lora_id, net.conv, rank=rank, dropout=0.0, alpha=1.0, branch=branch, parent_block=net, host_name="conv")
        nn.init.normal_(blk.layer.W_up, std=0.1)
        blocks[branch] = blk
    assert type(net.conv).__name__ == "DAPPPatchContainer"
    x = torch.randn(B, Cin, H, H, device=DEV)
    xg = x.clone().requires_grad_(True)
    y = net.conv(xg)
    sd = {"conv.weight": net.conv._host.weight.detach().cpu().to(BF).float(), "conv.bias": net.conv._host.bias.detach().cpu()}
    entries = []
    for branch in ("p", "n"):
        b = blocks[branch]
        entries.append(U.LoraEntry(b.layer.W_down.detach().cpu().clone().requires_grad_(True), b.layer.W_up.detach().cpu().clone().requires_grad_(True),
                                   float(b.alpha), branch))
    xr = x.cpu().to(BF).float().requires_grad_(True)
    yr = U._conv(sd, {"conv": entries}, "conv", xr, stride=stride, padding=1)
    assert rel_l2(y, yr) < 1e-2
    dy = torch.randn_like(y)
    y.backward(dy)
    yr.backward(dy.cpu())
    assert rel_l2(xg.grad, xr.grad) < 2e-2
    for e, branch in zip(entries, ("p", "n")):
        assert rel_l2(blocks[branch].layer.W_down.grad, e.W_down.grad) < 2e-2
        assert rel_l2(blocks[branch].layer.W_up.grad, e.W_up.grad) < 2e-2


# ----------------------------------------------------------------------------------------------------------------------
# entrypoint
# ----------------------------------------------------------------------------------------------------------------------
TINY_CFG = """
exp_dir: {exp}
seed: 7
ckpt_type: safetensors
model:
  unet:
    _target_: hcp_diffusion_b200.models.UNet2DConditionModel
    sample_size: 16
    block_out_channels: [64, 128, 128, 128]
    attention_head_dim: 2
    cross_attention_dim: 64
  init: random
  ema: {{decay_max: 0.9997, power: 0.85}}
lora_unet:
  - lr: 1.0e-3
    rank: 4
    layers: ['re:.*\\.attn1$']
  - lr: 2.5e-4
    rank: 2
    layers: ['re:.*\\.attn2$']
train:
  train_steps: 4
  save_step: 2
  log_step: 1
  gradient_accumulation_steps: 2
  scale_lr: false
  max_grad_norm: 1.0
  cuda_graph: true
  optimizer: {{lr: 1.0e-3, weight_decay: 1.0e-2}}
  scheduler: {{name: one_cycle, num_warmup_steps: 2, num_training_steps: 4}}
  loss:
    criterion: {{_target_: hcpdiff.loss.MinSNRLoss, gamma: 2.0}}
data:
  batch_size: 2
  num_samples: 8
  tokens: 77
"""


def test_train_ac_entrypoint_writes_loadable_checkpoint_and_resumes(tmp_path):
    from hcp_diffusion_b200.ckpt_manager import CkptManagerSafe
    from hcp_diffusion_b200.train_ac import Trainer
    from hcp_diffusion_b200.utils.cfg_net_tools import HCPModelLoader
    from hcp_diffusion_b200.utils.config import load_config_with_cli
    cfg_path = os.path.join(tmp_path, "tiny.yaml")
    with open(cfg_path, "w") as f:
        f.write(TINY_CFG.format(exp=os.path.join(tmp_path, "exp")))
    r = subprocess.run([sys.executable, "-m", "hcp_diffusion_b200.train_ac", "--cfg", cfg_path, "train.train_steps=2"], cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "step 2/2" in r.stdout
    ck = os.path.join(tmp_path, "exp", "ckpts", "unet-2.safetensors")
    sd = CkptManagerSafe().load_ckpt(ck)
    assert set(sd) == {"lora", "lora_ema"} and set(sd["lora"]) == set(sd["lora_ema"])
    assert all(".___." in k for k in sd["lora"]) and any(k.endswith(".___.layer.W_down") for k in sd["lora"])
    ups = [v for k, v in sd["lora"].items() if k.endswith("layer.W_up")]
    assert all(float(v.abs().sum()) > 0 for v in ups)                      # W_up starts at zero: training moved it
    # the checkpoint loads into a fresh model through the reference loader interface
    spec = U.TINY
    unet = tiny_unet(U.init_params(spec))
    grp = HCPModelLoader(unet).load_lora([{"path": ck}])
    assert len(grp.plugin_dict) == len(ups)
    # resume: the tensors land in the blocks that are trained and saved (advisor r1: they used to go into orphaned duplicates)
    conf = load_config_with_cli(cfg_path, [f"train.resume.ckpt_path.unet=[{ck}]", "train.resume.start_step=2", "train.train_steps=3"])
    tr = Trainer(conf)
    for c in tr.unet.modules():
        if hasattr(c, "plugin_names"):
            assert len(c.plugin_names) == len(set(c.plugin_names)) == 1
    live = tr.lora.state_dict()
    for k, v in sd["lora"].items():
        torch.testing.assert_close(live[k].cpu(), v, msg=k)
    flat_ptrs = {p.data_ptr() for p in tr.step_fn.flat.params}
    assert all(b.layer.W_down.data_ptr() in flat_ptrs for b in tr.lora.plugin_dict.values())     # the trained tensors ARE the module's
    before = {k: v.clone() for k, v in live.items()}
    tr.train()
    after = tr.lora.state_dict()
    assert any(not torch.equal(after[k], before[k]) for k in before if k.endswith("W_up"))
    assert os.path.exists(os.path.join(tmp_path, "exp", "ckpts", "unet-2.safetensors"))


# ----------------------------------------------------------------------------------------------------------------------
# data parallel: N ranks over NCCL == 1 rank on the concatenated batch
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_nccl_step_equals_single_rank_on_concatenated_batch(tmp_path):
    out = os.path.join(tmp_path, "dp")
    os.makedirs(out)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29611", os.path.join(ROOT, "tests", "dp_worker.py"), out], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    r0, r1 = torch.load(os.path.join(out, "rank0.pt")), torch.load(os.path.join(out, "rank1.pt"))
    single = torch.load(os.path.join(out, "single.pt"))
    # replicas hold bit-identical parameters after every step (same all-reduced gradient, same update)
    assert torch.equal(r0["params"], r1["params"]) and torch.equal(r0["m"], r1["m"])
    # and they match one process stepping on the concatenated batch: the mean over 2B images == the mean of the two rank means
    assert rel_l2(r0["m"], single["m"]) < 2e-2
    du_dp, du_1 = r0["params"] - r0["init"], single["params"] - single["init"]
    cos = float((du_dp.double() @ du_1.double()) / (du_dp.double().norm() * du_1.double().norm()))
    assert cos > 0.98 and torch.equal(r0["init"], r1["init"])
    assert abs(0.5 * (r0["loss"][0] + r1["loss"][0]) - single["loss"][0]) < 1e-3 * abs(single["loss"][0])


# ----------------------------------------------------------------------------------------------------------------------
# the shipped locon.yaml placement, unmodified: attention + ff Linear (item 0) and everything under `resnets` -- conv1, conv2,
# conv_shortcut AND time_emb_proj -- plus proj_in / proj_out / the sampler convs (item 1)
# ----------------------------------------------------------------------------------------------------------------------
def test_tiny_unet_shipped_locon_yaml_items_match_oracle():
    spec = U.TINY
    sd = U.init_params(spec)
    unet = tiny_unet(sd)
    items = [{"lr": 1e-4, "rank": 8, "layers": [r"re:.*\.attn.?$", r"re:.*\.ff$"]},                                       # locon.yaml:3-9
             {"lr": 1e-4, "rank": 8, "layers": [r"re:.*\.resnets$", r"re:.*\.proj_in$", r"re:.*\.proj_out$", r"re:.*\.conv$"]}]  # :10-17
    _, group = make_hcpdiff(unet, None, items)
    pat = r".*\.attn.?$|.*\.ff$|.*\.resnets$|.*\.proj_in$|.*\.proj_out$|.*\.conv$"
    lora = U.init_lora(spec, rank=8, alpha=1.0, seed=9, up_std=0.05, pattern=pat, include_conv=True)
    assert set(lora) == set(group.plugin_dict), set(lora) ^ set(group.plugin_dict)
    assert any(k.endswith("time_emb_proj") for k in lora) and any(k.endswith("conv_shortcut") for k in lora)
    with torch.no_grad():
        for layer, entries in lora.items():
            group[layer].layer.W_down.copy_(entries[0].W_down)
            group[layer].layer.W_up.copy_(entries[0].W_up)
    lat, noise, t, ehs = U.synthetic_batch(2, spec)
    loss_ref, pred_ref, grads_ref = U.lora_step_loss_and_grads(sd, lora, lat, noise, t, ehs, spec)
    x_t = U.add_noise(lat, noise, t, U.ddpm_alphas_cumprod())
    pred = unet(x_t.to(DEV), t.to(DEV), ehs.to(DEV)).sample
    assert rel_l2(pred, pred_ref) < 2e-2
    F.mse_loss(pred, noise.to(DEV), reduction="none").mean().backward()
    num = den = 0.0
    tnum = tden = 0.0
    for layer, blocks in grads_ref.items():
        blk = group[layer]
        for got, ref in ((blk.layer.W_down.grad, blocks[0][0]), (blk.layer.W_up.grad, blocks[0][1])):
            assert got is not None, layer
            e, n = float((got.cpu().double() - ref.double()).pow(2).sum()), float(ref.double().pow(2).sum())
            num, den = num + e, den + n
            if layer.endswith("time_emb_proj"):
                tnum, tden = tnum + e, tden + n
    assert math.sqrt(num / den) < 5e-2
    assert math.sqrt(tnum / tden) < 5e-2          # the time-embedding adapters on their own


# ----------------------------------------------------------------------------------------------------------------------
# round-2 C-ABI additions, called directly: the second GEMM output and the LoRA weight merge
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,K,N,rp", [(300, 320, 320, 8), (1024, 640, 640, 24), (16384, 320, 960, 24), (77, 768, 1280, 16)])
def test_gemm_second_output_matches_torch(M, K, N, rp):
    """hcp_gemm_args.out2 / n_main: columns [N, N + rp) of x . W_ext^T leave raw in a second buffer, the first N get bias + residual
    (M tails, the partly filled last 176-column tile; the main part goes through the TMA-store epilogue)."""
    g = torch.Generator().manual_seed(7)
    x = torch.randn(M, K, generator=g).to(DEV).to(BF)
    w_ext = (torch.randn(N + rp, K, generator=g) / math.sqrt(K)).to(DEV).to(BF)
    bias = (torch.randn(N, generator=g) * 0.1).to(DEV)
    res = torch.randn(M, N, generator=g).to(DEV).to(BF)
    out = torch.empty((M, N), dtype=BF, device=DEV)
    t2 = torch.zeros((M, 64), dtype=BF, device=DEV)
    ops.gemm_raw([(x, K, K)], [(w_ext, K, N + rp, 0)], M, N + rp, out, N, bias=bias, residual=res, ldr=N, out2=t2, ldo2=64, n_main=N)
    ref = x.float() @ w_ext.float().t()
    assert rel_l2(out, ref[:, :N] + bias + res.float()) < 1e-2
    assert rel_l2(t2[:, :rp], ref[:, N:]) < 1e-2
    assert float(t2[:, rp:].float().abs().sum()) == 0.0           # nothing beyond the rank columns is written


def test_lora_merge_kernel_matches_fp32_sum_and_carries_rank_rows():
    """hcp_lora_merge through LinearPack.enable_merge + runtime.pack_lora: W = bf16(W_host + sum alpha W_up W_down) (fp32 sum, one
    rounding), W^T its exact transpose, the extra operand rows = the factors the rank products need."""
    from hcp_diffusion_b200.ops import LinearPack, LoraBlockRef
    from hcp_diffusion_b200.runtime import pack_lora
    g = torch.Generator().manual_seed(11)
    K, n_per = 640, 320
    hosts = [(torch.randn(n_per, K, generator=g) / math.sqrt(K)).to(DEV) for _ in range(2)]        # a fused group of two hosts
    pack = LinearPack(torch.cat(hosts, 0), None)
    refs, per_host = [], []
    for i, (ranks, alpha) in enumerate((((8, 4), 0.125), ((16,), 0.5))):                             # host 0 carries two stacked blocks
        mine = []
        for r in ranks:
            down = (torch.randn(r, K, generator=g) / math.sqrt(K)).to(DEV)
            up = (torch.randn(n_per, r, generator=g) * 0.3).to(DEV)
            ref = LoraBlockRef(down, up, alpha, i * n_per)
            refs.append(ref)
            mine.append(ref)
        per_host.append((hosts[i], i * n_per, n_per, mine))
    pack.attach_lora(refs)
    assert pack.enable_merge(per_host) and pack.ext_rp == 32

    class G:
        pass
    grp = G()
    grp.pack = pack
    pack_lora([grp])
    torch.cuda.synchronize()
    N = 2 * n_per
    want = torch.cat([h + sum(b.alpha * (b.w_up @ b.w_down) for b in blocks) for h, _, _, blocks in per_host], 0)
    got = pack.W[:N].float()
    assert rel_l2(got, want) < 3e-3                                   # bf16 rounding of the fp32 sum
    assert float((got - want.to(BF).float()).abs().max()) <= float(want.abs().max()) * 2 ** -7      # at most one bf16 ulp apart
    assert torch.equal(pack.WT[:K], pack.W[:N].t())
    c0 = 0
    for b in refs:
        assert torch.equal(pack.W[N + c0:N + c0 + b.rank], b.w_down.to(BF))
        assert torch.equal(pack.WT[K + c0:K + c0 + b.rank, b.o0:b.o0 + n_per], (b.alpha * b.w_up).to(BF).t())
        c0 += b.rank
