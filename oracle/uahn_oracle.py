"""ORACLE — test infrastructure only, never the product path.

CPU restatement (torch fp32 functional ops, same ATen operators in the same order) of the
reference UAHN forward, i.e. of `/root/reference/trace_pytorch_model/model_to_trace.py` and
`warp.py`.  Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline /
``--impl reference`` legs may import this module.

Parity pinning: the reference has NO tests or golden vectors for this path (SURVEY §4, §8c), so the
restatement is pinned against outputs of the reference itself: `oracle/make_golden.py` imports the
unmodified reference modules from `/root/reference`, runs them on seeded inputs and commits the
results under `tests/golden/`; `tests/test_oracle.py` requires this restatement to reproduce those
vectors bit-for-bit (same torch version) — see DESIGN.md §Oracle.

Every function cites the reference lines it follows.  The reference model is strictly batch-1
(`warp.py:64`, `model_to_trace.py:25-26,272`), so a "batch" here is a Python loop.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np
import torch
import torch.nn.functional as F

IMG_H, IMG_W = 224, 320
MC = 16
P1 = "model_part1."
P4 = "model_last_block_list.0."


def origin_4pt() -> torch.Tensor:
    """model_to_trace.py:78-83 — UL, BL, BR, UR as (u, v), cornerOffset 0."""
    return torch.tensor([[0.0, 0.0], [0.0, IMG_H - 1.0], [IMG_W - 1.0, IMG_H - 1.0], [IMG_W - 1.0, 0.0]])


def grid_uv1() -> torch.Tensor:
    """warp.py:45-54 — [3, H*W] rows (u, v, 1), flattened row-major v*W+u."""
    u = torch.arange(0, IMG_W).view(1, -1).repeat(IMG_H, 1).unsqueeze(0).float()
    v = torch.arange(0, IMG_H).view(-1, 1).repeat(1, IMG_W).unsqueeze(0).float()
    uv = torch.cat((u, v), dim=0)
    return torch.cat((uv, torch.ones_like(uv[0:1])), dim=0).view(3, IMG_H * IMG_W)


_GRID = None
_FACTOR = torch.FloatTensor([[[2 / (IMG_W - 1), 2 / (IMG_H - 1)]]])  # warp.py:40


def sample_grid(Hm: torch.Tensor) -> torch.Tensor:
    """warp.py:64-70 — normalised sampling grid [H, W, 2] for a 3x3 pixel homography."""
    global _GRID
    if _GRID is None:
        _GRID = grid_uv1()
    uvz = torch.mm(Hm, _GRID)                      # warp.py:65
    uv1 = uvz / uvz[2, :]                          # warp.py:66
    uv = uv1[0:2, :].view(2, IMG_H, IMG_W)         # warp.py:67
    uv = torch.transpose(torch.transpose(uv, 0, 1), 1, 2)  # warp.py:68-69
    return uv * _FACTOR - 1                        # warp.py:70


def sample_indices(Hm: torch.Tensor):
    """Integer NW tap indices grid_sample derives from `sample_grid` (align_corners=True).

    ATen un-normalises with ((g+1)/2)*(size-1) (GridSampler.h:27-31; the vectorised CPU kernel
    uses (g+1)*((size-1)/2), the same real number rounded once) and floors.
    Returns int32 (ix_nw[H,W], iy_nw[H,W]) plus the fp32 (ix, iy).
    """
    g = sample_grid(Hm)
    ix = ((g[..., 0] + 1) / 2) * (IMG_W - 1)
    iy = ((g[..., 1] + 1) / 2) * (IMG_H - 1)
    return torch.floor(ix).to(torch.int32), torch.floor(iy).to(torch.int32), ix, iy


def warp_image(img: torch.Tensor, Hm: torch.Tensor) -> torch.Tensor:
    """warp.py:60-79 — img [1,1,H,W] fp32, Hm [3,3]; bilinear, zeros padding, align_corners=True."""
    g = sample_grid(Hm).unsqueeze(0)
    return F.grid_sample(img, g, mode="bilinear", padding_mode="zeros", align_corners=True)


def dlt_solve(src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    """model_to_trace.py:42-61 — src,dst [bs,4,2] → H [bs,3,3] via explicit inverse(A)·b."""
    bs = src.size(0)
    ones = torch.ones_like(src)[:, :, 0:1]
    xy1 = torch.cat((src, ones), 2)
    zeros = torch.zeros_like(xy1)
    xyu, xyd = torch.cat((xy1, zeros), 2), torch.cat((zeros, xy1), 2)
    M1 = torch.cat((xyu, xyd), 2).reshape(bs, -1, 6)
    M2 = torch.matmul(dst.reshape(-1, 2, 1), src.reshape(-1, 1, 2)).reshape(bs, -1, 2)
    A = torch.cat((M1, -M2), 2)
    b = dst.reshape(bs, -1, 1)
    h8 = torch.matmul(torch.inverse(A), b).reshape(bs, 8)
    return torch.cat((h8, ones[:, 0, :]), 1).reshape(bs, 3, 3)


def conv_lrelu(x, sd, key, stride):
    """model_to_trace.py:7-15 — Conv2d(pad=(k-1)//2, bias) → LeakyReLU(0.1, inplace)."""
    w = sd[key + ".0.weight"]
    return F.leaky_relu(F.conv2d(x, w, sd[key + ".0.bias"], stride=stride, padding=(w.shape[-1] - 1) // 2), 0.1, True)


BLOCK_LAYERS = {
    1: [("block_1_1", 2), ("block_1_2", 2), ("block_1_3", 2)],
    2: [("block_2_1", 2), ("block_2_2", 2), ("block_2_3", 2), ("block_2_4", 2)],
    3: [("block_3_0", 1), ("block_3_1", 2), ("block_3_2", 2), ("block_3_3", 2), ("block_3_4", 2), ("block_3_5", 2)],
    4: [("block_4_0", 1), ("block_4_1", 2), ("block_4_2", 2), ("block_4_3", 2), ("block_4_4", 2), ("block_4_5", 2),
        ("block_4_6", 2)],
}
BLOCK_POOL = {1: 8, 2: 4, 3: 2, 4: 1}


def conv_stack(x, sd, block, taps=None):
    pre = P4 if block == 4 else P1
    for name, s in BLOCK_LAYERS[block]:
        x = conv_lrelu(x, sd, pre + name, s)
        if taps is not None:
            taps[name] = x
    return x


@dataclass
class Taps:
    """Intermediate values of one forward, for stage-level parity tests."""
    H_prior: torch.Tensor | None = None
    H: dict = field(default_factory=dict)        # block -> cumulative H after that block
    d: dict = field(default_factory=dict)        # block -> regressed 4pt offset [8]
    warped: dict = field(default_factory=dict)   # block -> warped img2 [1,1,H,W]
    x_in: dict = field(default_factory=dict)     # block -> pooled 2-channel input
    feat: dict = field(default_factory=dict)     # block -> final [1,256,4,5]
    act: dict = field(default_factory=dict)      # layer name -> activation
    mc_mean: torch.Tensor | None = None          # [16,4,2]
    mc_logvar: torch.Tensor | None = None        # [16,4,2] (already ×1e-3)
    mu: torch.Tensor | None = None
    var: torch.Tensor | None = None
    H_total: torch.Tensor | None = None


def part1(img1, img2, sd, prior=None, blocks_to_run=3, taps: Taps | None = None):
    """model_to_trace.py:124-193 — Down_Net_3blocks.forward; returns cumulative H [1,3,3]."""
    pts0 = origin_4pt().unsqueeze(0)
    if prior is not None:
        Hm = dlt_solve(pts0, pts0 + prior)                                    # :129-130
        if taps is not None:
            taps.H_prior = Hm
        if blocks_to_run == 1:
            return Hm
    run = lambda b, x: conv_stack(x, sd, b, taps.act if taps is not None else None)
    if prior is None:                                                        # block 1  :137-148
        x = F.avg_pool2d(torch.cat((img1, img2), dim=1), 8, 8)
        f = run(1, x)
        d = F.linear(f.view(1, -1), sd[P1 + "fc_block_1.weight"], sd[P1 + "fc_block_1.bias"])
        Hm = dlt_solve(pts0, pts0 + d.view(1, 4, 2))
        if taps is not None:
            taps.x_in[1], taps.feat[1], taps.d[1], taps.H[1] = x, f, d.flatten(), Hm
    if prior is None or blocks_to_run == 3:                                  # block 2  :153-168
        w = warp_image(img2, Hm[0])
        x = F.avg_pool2d(torch.cat((img1, w), dim=1), 4, 4)
        f = run(2, x)
        d = F.linear(f.view(1, -1), sd[P1 + "fc_block_2.weight"], sd[P1 + "fc_block_2.bias"])
        Hb = dlt_solve(pts0, pts0 + d.view(1, 4, 2))
        Hm = torch.bmm(Hm, Hb)
        if taps is not None:
            taps.warped[2], taps.x_in[2], taps.feat[2], taps.d[2], taps.H[2] = w, x, f, d.flatten(), Hm
    if prior is None or blocks_to_run >= 2:                                  # block 3  :171-188
        w = warp_image(img2, Hm[0])
        x = F.avg_pool2d(torch.cat((img1, w), dim=1), 2, 2)
        f = run(3, x)
        d = F.linear(f.view(1, -1), sd[P1 + "fc_block_3.weight"], sd[P1 + "fc_block_3.bias"])
        Hb = dlt_solve(pts0, pts0 + d.view(1, 4, 2))
        Hm = torch.bmm(Hm, Hb)
        if taps is not None:
            taps.warped[3], taps.x_in[3], taps.feat[3], taps.d[3], taps.H[3] = w, x, f, d.flatten(), Hm
    return Hm


def mc_head(f, sd, masks):
    """model_to_trace.py:222-235,252-256,272-281 with explicit dropout masks.

    f [1,256,4,5]; masks = (m1[16,5120], m2[16,256], u1[16,5120], u2[16,256]) with values in
    {0, 1/0.95} — exactly what nn.Dropout(p=0.05) in train mode multiplies by.
    """
    m1, m2, u1, u2 = masks
    x = f.repeat(MC, 1, 1, 1).view(MC, -1)                                   # :272-273

    def head(name, ma, mb):
        h = F.linear(x * ma, sd[P4 + name + ".1.weight"], sd[P4 + name + ".1.bias"])
        h = F.leaky_relu(h, 0.1, True) * mb
        return F.linear(h, sd[P4 + name + ".4.weight"], sd[P4 + name + ".4.bias"]).view(MC, 4, 2)

    mean = head("fc_block_4_mean", m1, m2)
    logvar = head("fc_block_4_uncertainty", u1, u2) * 1e-03                  # :256
    var = torch.exp(logvar)                                                  # :274
    mu = mean.mean(0).unsqueeze(0)                                           # :275
    avg_pred_var = var.mean(0).unsqueeze(0)                                  # :276-277
    emp = torch.square(mu.repeat(MC, 1, 1) - mean).mean(0).unsqueeze(0)      # :278-279
    return mean, logvar, mu, emp + avg_pred_var                              # :280


def transfer_mean_var_single(var, Hm, pts_w):
    """model_to_trace.py:18-38 — var [1,4,2], Hm [1,3,3], pts_w [1,4,2] → pts2 [1,3,4], Cov [1,4,2,2]."""
    uv1 = torch.transpose(torch.cat((pts_w, torch.ones_like(pts_w)[:, :, 0:1]), dim=2), 1, 2)
    p = torch.bmm(Hm, uv1)
    scale = p[:, 2:3, :]
    p = p / scale
    s_i = scale[0, 0, :]
    H0 = Hm[0]
    covs = []
    for i in range(4):
        Hs = H0 / s_i[i]
        V = torch.diag(torch.cat((var[0, i, :], torch.zeros_like(s_i[i]).unsqueeze(0))))
        covs.append(torch.mm(torch.mm(Hs, V), Hs.t())[0:2, 0:2].unsqueeze(0))
    return p, torch.cat(covs, dim=0).unsqueeze(0)


def forward(img1, img2, sd, masks, prior=None, show_error=False, blocks_to_run=3, taps: Taps | None = None):
    """model_to_trace.py:299-330 — combined_stu_model.forward with explicit MC-dropout masks.

    img1 (previous), img2 (current): [1,1,224,320] fp32 in [0,1]; prior: [1,1,4,2] px or None.
    Returns (flow [8,1], Cov [8,8], err [1,1,224,320] or None).
    """
    with torch.no_grad():
        Hp = part1(img1, img2, sd, prior, blocks_to_run, taps)
        w = warp_image(img2, Hp[0])                                          # :261
        x = torch.cat((img1, w), dim=1)
        f = conv_stack(x, sd, 4, taps.act if taps is not None else None)
        mean, logvar, mu, var = mc_head(f, sd, masks)
        pts0 = origin_4pt().unsqueeze(0)
        pts_w = pts0 + mu                                                    # :281
        p2, cov4 = transfer_mean_var_single(var, Hp, pts_w)                  # :309
        flow = (torch.transpose(p2[:, 0:2, :], 1, 2) - pts0).squeeze()       # :311
        cov4 = cov4.squeeze()
        cov = torch.zeros([8, 8])
        for i in range(4):
            cov[2 * i:2 * i + 2, 2 * i:2 * i + 2] = cov4[i]                  # :313-317
        err = None
        Ht = None
        if show_error:                                                       # :319-327
            H4 = dlt_solve(pts0, pts_w)
            Ht = torch.bmm(Hp, H4)
            err = (warp_image(img2, Ht[0]) - img1).abs() * 255.0
        if taps is not None:
            taps.warped[4], taps.x_in[4], taps.feat[4] = w, x, f
            taps.mc_mean, taps.mc_logvar, taps.mu, taps.var, taps.H_total = mean, logvar, mu, var, Ht
            taps.H[4] = Hp
        return flow.reshape(8, 1), cov, err


class TracedModel(torch.nn.Module):
    """`combined_stu_model` (model_to_trace.py:284-330) as far as a TorchScript trace of it shows: the reference's
    parameter tree (the 54 state_dict names, model_to_trace.py:333-350) around `forward` above, with fresh MC-dropout
    masks on every call like the reference's train-mode nn.Dropout."""

    def __init__(self, sd, show_error: bool = False, blocks_to_run: int = 3):
        super().__init__()
        for key, t in sd.items():
            *path, leaf = key.split(".")
            mod = self
            for name in path:
                if name not in mod._modules:
                    mod.add_module(name, torch.nn.Module())
                mod = mod._modules[name]
            mod.register_parameter(leaf, torch.nn.Parameter(t.clone(), requires_grad=False))
        self.show_error, self.blocks_to_run = show_error, blocks_to_run

    def forward(self, img1, img2, prior=None):
        masks = tuple(F.dropout(torch.ones(MC, n), 0.05, True) for n in (5120, 256, 5120, 256))
        flow, cov, err = forward(img1, img2, dict(self.named_parameters()), masks, prior, self.show_error, self.blocks_to_run)
        return (flow, cov) if err is None else (flow, cov, err)


def trace(sd, variant: str = "prior3", show_error: bool = False):
    """TorchScript of one reference graph, traced like trace_model.py:20-22,36-46 (check_trace=False), but of
    `TracedModel`: the reference's `.pt` files without the reference's source.  tests/golden/reference_graphs.json
    records, from the reference's own traces, the op-kind counts and inputs of the full and 3-block graphs (with and
    without the error map) and the state_dict names; tests/test_weights.py holds these traces to that record.  The
    2-block and 1-block graphs were not recorded."""
    import contextlib
    import io
    blocks_to_run = {"full": 3, "prior3": 3, "prior2": 2, "prior1": 1}[variant]
    img1, img2 = torch.ones(1, 1, IMG_H, IMG_W) * 0.2, torch.ones(1, 1, IMG_H, IMG_W) * 0.5
    args = (img1, img2) if variant == "full" else (img1, img2, torch.ones(1, 1, 4, 2) * 0.9)
    with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        return torch.jit.trace(TracedModel(sd, show_error, blocks_to_run), args, check_trace=False)


def u8_to_unit(img_u8) -> torch.Tensor:
    """HomographyNet.cpp:144-146 — u8 HxW → [1,1,H,W] fp32, true division by 255."""
    t = torch.as_tensor(np.ascontiguousarray(img_u8)).to(torch.float32) / 255.0
    return t.view(1, 1, IMG_H, IMG_W)


def forward_batch(prev_u8, curr_u8, sd, masks_list, priors=None, show_error=False, blocks_to_run=3):
    """Loop-of-batch-1 oracle over n pairs (the reference cannot batch, SURVEY §0 fact 3)."""
    n = len(prev_u8)
    means = np.zeros((n, 8), np.float32)
    covs = np.zeros((n, 8, 8), np.float32)
    errs = np.zeros((n, IMG_H, IMG_W), np.float32) if show_error else None
    for i in range(n):
        pr = None if priors is None else torch.as_tensor(priors[i]).float().view(1, 1, 4, 2)
        m, c, e = forward(u8_to_unit(prev_u8[i]), u8_to_unit(curr_u8[i]), sd, masks_list[i], pr, show_error,
                          blocks_to_run)
        means[i], covs[i] = m.flatten().numpy(), c.numpy()
        if show_error:
            errs[i] = e[0, 0].numpy()
    return means, covs, errs
