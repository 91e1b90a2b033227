"""Network DERIVED from a searched genotype (SURVEY.md §8f-4, BASELINE config 5).

The reference ends at `Network.genotype()` (darts_vqa/pcdarts/model_search.py:218-263): it never builds the network the
genotype describes, so there is nothing to be bit-compatible with — parity is pinned per operation (every op module against
the reference's own `OPS[name]` layers, tests/test_emu_ops.py) and, for the whole network, against the same modules run as
stock torch layers in float64 (`stock_forward`).  The structure follows the search network it is derived from:

  * same stem, same cell plan (reduction cells at layers//3 and 2*layers//3, model_search.py:118-127), same channel counts,
    same preprocess ops (ReLUConvBN 1x1 / FactorizedReduce when the previous cell reduced, model_search.py:67-71), same
    AdaptiveAvgPool2d(7) + flatten tail (model_search.py:131,176-178), so it drops into `DartsEncoder` in place of the
    search network;
  * a cell keeps, per intermediate node, the two (op, source) pairs the genotype names (`Genotype.normal / .reduce` in node
    order, genotypes.py:3), each op built as `OPS[name](C, stride, True)` on ALL C channels — no partial channels, no
    alpha / beta weighting, BatchNorm with affine parameters; stride 2 on the edges that leave the two cell inputs of a
    reduction cell (model_search.py:79); node = op1(h1) + op2(h2); output = concat of the `*_concat` states.

Execution: every op runs on the library's stand-alone op kernels (pcd_opmods.py), stem / pooling on the kernels the search
network uses.  In eval mode under torch.no_grad() every BatchNorm uses its running statistics: the stem and the preprocess
ops run the eval kernels, each DilConv / SepConv unit depthwise -> pointwise -> running-stat affine.

Drop-path (the regulariser of the DARTS / PC-DARTS evaluation recipes): `net.drop_path_prob = p`.  In training mode every
node is one pcd_droppath_sum launch, which scales each non-Identity op output of the node by (x / keep) * m(b), keep = 1 - p,
with one Bernoulli(keep) mask per sample (DARTS's drop_path), and adds the two.  Identity ops are never dropped; a stride-2
skip_connect is a FactorizedReduce and is.  The masks are a pure function of (seed, global sample index, cell, node input):
the seed is drawn once per forward from torch's generator on the input's device, and under torch.distributed the sample
index is rank * local batch + b, so equally sized shards draw the masks one process would draw on the whole batch.  In eval
mode, and at p = 0, a node is bit-equal to op1(h1) + op2(h2).  The auxiliary head of the CIFAR / ImageNet recipes is not
part of this path.
"""
import torch
import torch.distributed as dist
import torch.nn as nn

import pcd_ops
from .genotypes import Genotype, PRIMITIVES  # noqa: F401  (re-exported: the vocabulary a genotype is written in)
from .operations import OPS, FactorizedReduce, Identity, ReLUConvBN


class Cell(nn.Module):
    """One cell of the derived network: `genotype.normal` (or `.reduce`) = [(op name, source state)] * 2 per node."""

    def __init__(self, genotype, C_prev_prev, C_prev, C, reduction, reduction_prev, index=0):
        super().__init__()
        self.reduction = reduction
        self.index = index            # position in the network: a counter word of the drop-path masks
        if reduction_prev:
            self.preprocess0 = FactorizedReduce(C_prev_prev, C)
        else:
            self.preprocess0 = ReLUConvBN(C_prev_prev, C, 1, 1, 0)
        self.preprocess1 = ReLUConvBN(C_prev, C, 1, 1, 0)
        gene, concat = (genotype.reduce, genotype.reduce_concat) if reduction else (genotype.normal, genotype.normal_concat)
        if len(gene) % 2:
            raise ValueError("a genotype lists two (op, source) pairs per intermediate node")
        self._steps = len(gene) // 2
        self._concat = list(concat)
        self.multiplier = len(self._concat)
        self._ops = nn.ModuleList()
        self._indices = []
        for pos, (name, index) in enumerate(gene):
            if name not in OPS:
                raise ValueError(f"unknown primitive {name!r}")
            if not 0 <= index < 2 + pos // 2:
                raise ValueError(f"gene {pos}: source state {index} does not exist yet")
            stride = 2 if reduction and index < 2 else 1
            self._ops.append(OPS[name](C, stride, True))
            self._indices.append(index)

    def forward(self, s0, s1, stock=False, drop=None):
        """drop: None (no drop-path: eval mode) or, on the native path, (keep tensor, seed tensor, sample offset); on the
        stock path (keep as a float, masks(cell, node, input) -> (B,) tensor of 0 / 1)."""
        run = (lambda m, x: m.stock_forward(x) if hasattr(m, "stock_forward") else m(x)) if stock else (lambda m, x: m(x))
        states = [run(self.preprocess0, s0), run(self.preprocess1, s1)]
        for i in range(self._steps):
            h1 = run(self._ops[2 * i], states[self._indices[2 * i]])
            h2 = run(self._ops[2 * i + 1], states[self._indices[2 * i + 1]])
            flags = [drop is not None and not isinstance(self._ops[2 * i + j], Identity) for j in range(2)]
            if stock:       # the yardstick: DARTS's drop_path in stock torch ops, with masks handed in
                if flags[0]:
                    h1 = h1.div(drop[0]).mul(drop[1](self.index, i, 0).to(h1).view(-1, 1, 1, 1))
                if flags[1]:
                    h2 = h2.div(drop[0]).mul(drop[1](self.index, i, 1).to(h2).view(-1, 1, 1, 1))
                states.append(h1 + h2)
            else:
                keep, seed, offset = drop if drop is not None else (None, None, 0)
                states.append(pcd_ops.droppath_sum(h1, h2, flags[0], flags[1], keep, seed, self.index, i, offset))
        return torch.cat([states[i] for i in self._concat], dim=1)


class NetworkDerived(nn.Module):
    """stem -> `layers` derived cells -> AdaptiveAvgPool2d(7) -> flatten; same interface as the search Network where it makes
    sense (`output_ch`, `output_size`, forward(input) -> (B, output_ch * 7 * 7))."""

    def __init__(self, C, layers, genotype, stem_multiplier=3):
        super().__init__()
        self._C, self._layers, self._genotype = C, layers, genotype
        C_curr = stem_multiplier * C
        self.stem = nn.Sequential(nn.Conv2d(3, C_curr, 3, padding=1, bias=False), nn.BatchNorm2d(C_curr))
        C_prev_prev, C_prev, C_curr = C_curr, C_curr, C
        self.cells = nn.ModuleList()
        reduction_prev = False
        for i in range(layers):
            reduction = i in (layers // 3, 2 * layers // 3)
            if reduction:
                C_curr *= 2
            cell = Cell(genotype, C_prev_prev, C_prev, C_curr, reduction, reduction_prev, index=i)
            reduction_prev = reduction
            self.cells.append(cell)
            C_prev_prev, C_prev = C_prev, cell.multiplier * C_curr
        self.output_ch = C_prev
        self.output_size = 7
        self.global_pooling = nn.AdaptiveAvgPool2d(self.output_size)
        # drop-path: keep = 1 - drop_path_prob lives on the device, read by the node kernels when they run
        self.register_buffer("_drop_keep", torch.ones(1), persistent=False)
        self._drop_path_prob = 0.0
        self.drop_path_seed = None        # None: a fresh seed per forward; a 1-element int64 device tensor fixes the masks
        self.drop_path_offset = None      # None: rank * local batch under torch.distributed, else 0

    @property
    def drop_path_prob(self):
        return self._drop_path_prob

    @drop_path_prob.setter
    def drop_path_prob(self, p):
        p = float(p)
        if not 0.0 <= p < 1.0:
            raise ValueError(f"drop_path_prob must be in [0, 1), got {p}")
        self._drop_path_prob = p
        with torch.no_grad():
            self._drop_keep.fill_(1.0 - p)

    def genotype(self):
        return self._genotype

    def arch_parameters(self):
        return []           # the genotype is fixed: nothing left to search

    def _sample_offset(self, batch):
        if self.drop_path_offset is not None:
            return int(self.drop_path_offset)
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank() * batch       # equally sized shards: sample b of rank r is r * batch + b globally
        return 0

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        pcd_ops.bump_layout_epoch()
        return out

    def forward(self, input, stock=False, drop_masks=None):
        """drop_masks (stock path only): masks(cell, node, input) -> (B,) tensor of 0 / 1, the drop-path masks the yardstick
        applies in training mode when drop_path_prob > 0."""
        n, _, h, w = input.shape
        x = input.expand(n, 3, h, w)
        if stock:       # the same modules as stock torch layers: the yardstick of the parity tests, never the product path
            drop = None
            if self.training and self._drop_path_prob > 0.0:
                if drop_masks is None:
                    raise ValueError("stock forward with drop_path_prob > 0 in training mode needs drop_masks")
                drop = (1.0 - self._drop_path_prob, drop_masks)
            s0 = s1 = self.stem(x)
            for cell in self.cells:
                s0, s1 = s1, cell(s0, s1, stock=True, drop=drop)
            return self.global_pooling(s1).flatten(start_dim=1)
        is_eval = pcd_ops.eval_forward(self, input)
        ar = self.__dict__.get('_stem_arena')
        if ar is None:
            ar = pcd_ops.Arena(self.stem)
            self.__dict__['_stem_arena'] = ar
        ar = ar.ensure()
        if is_eval:
            s0 = s1 = pcd_ops.stem_forward_eval(x, ar.param_ptr, ar.running_ptr, self.stem[0].out_channels)
        else:
            s0 = s1 = pcd_ops.StemFunction.apply(x, (ar.param_ptr, ar.running_ptr, ar.nbt_ptr), *ar.params)
        drop = None
        if not is_eval:     # the flags stay on at p = 0 (keep = 1 is exact), so a captured graph follows a later change of p
            seed = self.drop_path_seed
            if seed is None:
                seed = torch.empty(1, dtype=torch.int64, device=input.device).random_(-2 ** 63, None)
            drop = (self._drop_keep, seed, self._sample_offset(n))
        for cell in self.cells:
            s0, s1 = s1, cell(s0, s1, drop=drop)
        return pcd_ops.AdaptiveAvgPoolFunction.apply(s1, self.output_size).flatten(start_dim=1)


def derive(search_network, layers=None):
    """The network `search_network.genotype()` describes, with the search network's width and depth."""
    return NetworkDerived(search_network._C, layers or search_network._layers, search_network.genotype(),
                          stem_multiplier=search_network._stem_multiplier)
