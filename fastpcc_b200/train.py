"""Training slice of the sparse-convolution path (SURVEY 8a row 19; reference: train.py:139,215,359-404 -- a model wrapped
in DistributedDataParallel, loss.backward(), optimiser step, one process per GPU, NCCL carrying only the gradient
all-reduce).

`OccupancyNet` is the float occupancy predictor of one scale of the lossless coordinate codec
(models/convolutional/lossl_coord/model.py:137-175 in miniature): an embedding conv, residual `Block`s
(model.py:645-660) and a linear head whose 255 logits are trained with the cross entropy of the node's occupancy symbol
-- the codec's bits-per-node objective.  Every convolution is differentiable through `fastpcc_b200/autograd.py`:
forward and dgrad on the fused tcgen05 kernel, wgrad on `fpcc_spconv_wgrad_f16`.

`LossyGeoNet` is the lossy geometry codec (lossy_coord_v2) in miniature on the MinkowskiEngine-shaped layers, trained
with `train_step_lossy`.
"""
from typing import List

import numpy as np
import torch
import torch.nn as nn

from . import lossy_heads, ops, synth
from . import me as ME
from . import minkowski_sparse_conv_layers as L
from .sparse_tensor import SparseTensor
from . import torchsparse_nn as TS


class OccupancyNet(nn.Module):
    def __init__(self, channels: int = 128, n_blocks: int = 2):
        super().__init__()
        self.embed = TS.Conv3d(8, channels, 3, 1, 1, bias=True)
        self.blocks = nn.ModuleList([TS.Block(channels) for _ in range(n_blocks)])
        self.head = nn.Linear(channels, 255)

    def forward(self, x: SparseTensor) -> torch.Tensor:
        y = self.embed(x)
        y.F = torch.nn.functional.leaky_relu(y.F, 0.1)
        for b in self.blocks:
            y = b(y)
        return self.head(y.F.float())


def make_batch(seeds: List[int], level_shift: int, device) -> tuple:
    """Nodes of stride 2^level_shift of synthetic LiDAR scans (one batch index per scan), their occupancy symbol as the
    target and the parent-level occupancy bits as the input feature (what the decoder knows when it predicts the level)."""
    cs = []
    for b, s in enumerate(seeds):
        xyz = np.unique(synth.lidar_frame(s) >> (level_shift - 1), axis=0)  # children of the nodes we predict
        cs.append(synth.with_batch(xyz, b))
    child = torch.from_numpy(np.concatenate(cs)).to(device)
    order = torch.argsort(ops.morton_encode(child, col0=1, msb_axis=0) + (child[:, 0].long() << 52))
    child = ops.gather_rows(child.contiguous(), order)
    node_c, occ, _, _, cnt = ops.downsample(child)
    n = int(cnt.item())
    node_c, occ = node_c[:n].contiguous(), occ[:n].contiguous()
    # input feature: the occupancy bits of the node's PARENT (known context), broadcast to the node
    par_c, par_occ, par_of, _, cnt2 = ops.downsample(node_c)
    bits = ops.occ_to_bits(par_occ[: int(cnt2.item())].contiguous()).float()
    feats = bits[par_of[:n].long()]
    target = occ.long() - 1
    return SparseTensor(feats, node_c, 1), target


def train_step(model: nn.Module, opt: torch.optim.Optimizer, batch) -> torch.Tensor:
    x, target = batch
    opt.zero_grad(set_to_none=True)
    logits = model(SparseTensor(x.F, x.C, x.stride))
    loss = torch.nn.functional.cross_entropy(logits, target) / np.log(2.0)  # bits per node
    loss.backward()
    opt.step()
    return loss.detach()


class LossyGeoNet(nn.Module):
    """The encoder of the lossy geometry codec (config 4, lossy_coord_v2; SURVEY §3.4 and Appendix D give the topology --
    the reference source is not available here) plus one decoder stage, in miniature, built only from the float layer
    API (`minkowski_sparse_conv_layers`), so that every ME layer type trains:

      encoder   ConvBlock(1->16, k3) -> ConvBlock(16->C, k2s2) -> ResBlock(C) -> InceptionResBlock(C)    stride 2
      decoder   ConvBlock(C->C, k3) -> GenConvTransBlock(C->16, k2s2) -> MEMLPBlock(16->8) -> MEMLPBlock(8->1)
                = occupancy logits of the 8 generated children of every stride-2 voxel
      refine    keep = top-N (get_keep, N = input points per sample) | ground truth -> MinkowskiPruning ->
                ConvTransBlock(C->16, k2s2, PReLU) from the stride-2 features onto the kept key -> MEMLPBlock(16->1)

    forward(coords) takes unique, Morton-ordered int32 (batch, x, y, z) rows (`make_lossy_batch`), builds the sparse
    tensor on a fresh coordinate manager (as ME training does per batch) and returns the sum of the two binary cross
    entropies against "the generated child is a voxel of the input"."""

    def __init__(self, channels: int = 64):
        super().__init__()
        c = channels
        self.enc0 = L.ConvBlock(1, 16, 3, 1)
        self.enc1 = L.ConvBlock(16, c, 2, 2)
        self.res = L.ResBlock(c, 'HYPER_CUBE', False, 'relu')
        self.inception = L.InceptionResBlock(c, 'HYPER_CUBE', False, 'relu')
        self.dec0 = L.ConvBlock(c, c, 3, 1)
        self.gen = L.GenConvTransBlock(c, 16, 2, 2)
        self.mlp = L.MEMLPBlock(16, 8)
        self.head = L.MEMLPBlock(8, 1, act=None)
        self.prune = ME.MinkowskiPruning()
        self.tconv = L.ConvTransBlock(c, 16, 2, 2, act='prelu')
        self.head2 = L.MEMLPBlock(16, 1, act=None)

    def forward(self, coords: torch.Tensor) -> torch.Tensor:
        x = ME.SparseTensor(torch.ones((coords.shape[0], 1), device=coords.device), coordinates=coords)
        cm = x.coordinate_manager
        y = self.inception(self.res(self.enc1(self.enc0(x))))
        g = self.gen(self.dec0(y))
        logits = self.head(self.mlp(g)).F.reshape(-1)
        # ground truth: the candidate voxel exists in the input (a 1x1x1 kernel map = one hash probe per candidate)
        gt = cm.kernel_table(x.coordinate_map_key, g.coordinate_map_key, 1, (1, 1, 1))[0] > 0
        bce = torch.nn.functional.binary_cross_entropy_with_logits
        loss = bce(logits.float(), gt.float())
        n_per_sample = torch.bincount(coords[:, 0].long()).tolist()
        keep = lossy_heads.get_keep(logits.detach(), g.C, 1, 2, target_points_num=n_per_sample) | gt
        kept = self.prune(g, keep)
        logits2 = self.head2(self.tconv(y, kept.coordinate_map_key)).F.reshape(-1)
        return loss + bce(logits2.float(), gt[keep].float())


def make_lossy_batch(clouds: List[np.ndarray], device) -> torch.Tensor:
    """unique voxel clouds [n_b, 3] -> int32 (batch, x, y, z) rows, one batch index per cloud, in the shim's Morton order"""
    c = torch.from_numpy(np.concatenate([synth.with_batch(np.unique(xyz, axis=0), b) for b, xyz in enumerate(clouds)])).to(device)
    c = c.to(torch.int32).contiguous()
    return c[ME.morton_order(c)].contiguous()


def train_step_lossy(model: nn.Module, opt: torch.optim.Optimizer, batch: torch.Tensor, scaler=None) -> torch.Tensor:
    """One step of `LossyGeoNet` (or a DistributedDataParallel around it) in the shim's compute dtype
    (`me.set_compute_dtype`).  fp16 wants a `torch.amp.GradScaler`: the BCE means over 10^5 - 10^6 rows give per-row
    gradients below fp16's normal range.  bf16 needs none."""
    opt.zero_grad(set_to_none=True)
    loss = model(batch)
    if scaler is None:
        loss.backward()
        opt.step()
    else:
        scaler.scale(loss).backward()
        scaler.step(opt)
        scaler.update()
    return loss.detach()
