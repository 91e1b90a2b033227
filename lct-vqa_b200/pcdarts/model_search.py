"""PC-DARTS search network — B200 drop-in for darts_vqa/pcdarts/model_search.py and
basic_vqa/pcdarts/model_search.py.

Public surface kept: channel_shuffle(x, groups); MixedOp(C, stride).forward(x, weights);
Cell(steps, multiplier, C_pp, C_p, C, reduction, reduction_prev).forward(s0, s1, weights, weights2);
Network(C, num_classes, layers[, vqa_model], steps=4, multiplier=4, stem_multiplier=3) with
forward / new / arch_parameters / genotype / save_arch_parameters / load_arch_parameters and the
attributes alphas_*/betas_*, output_ch, output_size.  Sub-module names and registration order match
the reference, so state_dict keys and the architects' flat parameter vector carry over.

Execution is different by design: a Cell is ONE autograd node backed by fused sm_100a kernels
(libpcdarts_sm100.so: partial-channel MixedOps, channel shuffle, beta-weighted node sums and the
preprocess ops), fed from flat parameter arenas; nothing is computed layer by layer and there is no
CPU path.
"""
import weakref

import torch
import torch.nn as nn
import torch.nn.functional as F

import config
import pcd_ops
from pcdarts.genotypes import PRIMITIVES, Genotype
from pcdarts.operations import OPS, FactorizedReduce, ReLUConvBN

K_PARTIAL = 4          # 1/K of the channels go through the candidate ops (model_search.py:36)


def channel_shuffle(x, groups):
    """out[:, j*groups + g] = x[:, g*(C//groups) + j]  (model_search.py:14-28) — one CUDA copy kernel."""
    return pcd_ops.ChannelShuffleFunction.apply(x, groups)


class _ArenaModule(nn.Module):
    """Shared plumbing: modules whose weights the kernels read as one contiguous arena."""

    def _arena(self):
        ar = self.__dict__.get('_pcd_arena')
        if ar is None:
            ar = pcd_ops.Arena(self)
            self.__dict__['_pcd_arena'] = ar
        return ar.ensure()

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        pcd_ops.bump_layout_epoch()       # storages (and buffer objects) were replaced
        return out



class MixedOp(_ArenaModule):
    """Partial-channel mixed operation (model_search.py:30-58)."""

    def __init__(self, C, stride):
        super().__init__()
        self._ops = nn.ModuleList()
        self.mp = nn.MaxPool2d(2, 2)
        self.k = K_PARTIAL
        for primitive in PRIMITIVES:
            op = OPS[primitive](C // self.k, stride, False)
            if 'pool' in primitive:
                op = nn.Sequential(op, nn.BatchNorm2d(C // self.k, affine=False))
            self._ops.append(op)
        self.__dict__['_pcd_handle'] = pcd_ops.MixedHandle(C, stride)

    def forward(self, x, weights):
        is_eval = pcd_ops.eval_forward(self, x, weights)
        ar = self._arena()
        h = self.__dict__['_pcd_handle']
        h.param_ptr, h.running_ptr, h.nbt_ptr = ar.param_ptr, ar.running_ptr, ar.nbt_ptr
        if is_eval:
            return pcd_ops.mixedop_forward_eval(x, weights, h)
        return pcd_ops.MixedOpFunction.apply(x, weights, h, *ar.params)


class Cell(_ArenaModule):
    """Search cell: two preprocess ops, 14 MixedOp edges, 4 beta-weighted nodes (model_search.py:61-94)."""

    def __init__(self, steps, multiplier, C_prev_prev, C_prev, C, reduction, reduction_prev):
        super().__init__()
        if steps != 4 or multiplier != 4:
            raise NotImplementedError("the fused cell kernels implement steps=4, multiplier=4 (the reference default)")
        self.reduction = reduction
        if reduction_prev:
            self.preprocess0 = FactorizedReduce(C_prev_prev, C, affine=False)
        else:
            self.preprocess0 = ReLUConvBN(C_prev_prev, C, 1, 1, 0, affine=False)
        self.preprocess1 = ReLUConvBN(C_prev, C, 1, 1, 0, affine=False)
        self._steps = steps
        self._multiplier = multiplier
        self._ops = nn.ModuleList()
        self._bns = nn.ModuleList()
        for i in range(steps):
            for j in range(2 + i):
                self._ops.append(MixedOp(C, 2 if reduction and j < 2 else 1))
        self.__dict__['_pcd_handle'] = pcd_ops.CellHandle(C_prev_prev, C_prev, C, reduction, reduction_prev)

    def _cell_params(self):
        ps = self.__dict__.get('_pcd_plist')
        if ps is None:
            ps = list(self.parameters())
            self.__dict__['_pcd_plist'] = ps
        return ps

    def forward(self, s0, s1, weights, weights2):
        is_eval = pcd_ops.eval_forward(self, s0, s1, weights, weights2)
        ar = self._arena()
        h = self.__dict__['_pcd_handle']
        h.param_ptr, h.running_ptr, h.nbt_ptr = ar.param_ptr, ar.running_ptr, ar.nbt_ptr
        if is_eval:
            return pcd_ops.cell_forward_eval(s0, s1, weights, weights2, h)
        return pcd_ops.CellFunction.apply(s0, s1, weights, weights2, h, *ar.params)


def _grouped_softmax(betas, steps):
    """softmax over the incoming edges of every node: groups of 2,3,4,5 (model_search.py:157-174)."""
    parts, start = [], 0
    for n in range(2, 2 + steps):
        parts.append(F.softmax(betas[start:start + n], dim=-1))
        start += n
    return torch.cat(parts, dim=0)


class Network(_ArenaModule):
    """Search network: stem, `layers` cells, AdaptiveAvgPool2d(7), flatten (model_search.py:97-263)."""

    def __init__(self, C, num_classes, layers, *args, steps=4, multiplier=4, stem_multiplier=3):
        super().__init__()
        # basic_vqa inserts the owning VqaModel as 4th positional argument (basic_vqa model_search.py:99)
        args = list(args)
        if args and isinstance(args[0], nn.Module):
            self._vqa_model = weakref.ref(args.pop(0))
        if args:
            steps = args.pop(0)
        if args:
            multiplier = args.pop(0)
        if args:
            stem_multiplier = args.pop(0)
        self._C = C
        self._num_classes = num_classes
        self._layers = layers
        self._criterion = nn.CrossEntropyLoss()
        self._steps = steps
        self._multiplier = multiplier
        self._stem_multiplier = stem_multiplier

        C_curr = stem_multiplier * C
        self.stem = nn.Sequential(nn.Conv2d(3, C_curr, 3, padding=1, bias=False), nn.BatchNorm2d(C_curr))
        C_prev_prev, C_prev, C_curr = C_curr, C_curr, C
        self.cells = nn.ModuleList()
        reduction_prev = False
        for i in range(layers):
            reduction = i in (layers // 3, 2 * layers // 3)
            if reduction:
                C_curr *= 2
            self.cells.append(Cell(steps, multiplier, C_prev_prev, C_prev, C_curr, reduction, reduction_prev))
            reduction_prev = reduction
            C_prev_prev, C_prev = C_prev, multiplier * C_curr
        self.global_pooling = nn.AdaptiveAvgPool2d(7)
        self.output_ch = 256
        self.output_size = 7
        self._initialize_alphas()

    # ---- architecture parameters (plain tensors, NOT nn.Parameters: model_search.py:186-202) ----------
    def _initialize_alphas(self):
        k = sum(2 + i for i in range(self._steps))
        n_ops = len(PRIMITIVES)

        def fresh(*shape):
            return (1e-3 * torch.randn(*shape)).to(config.DEVICE).requires_grad_(True)
        self.alphas_normal = fresh(k, n_ops)
        self.alphas_reduce = fresh(k, n_ops)
        self.betas_normal = fresh(k)
        self.betas_reduce = fresh(k)
        self._arch_parameters = [self.alphas_normal, self.alphas_reduce, self.betas_normal, self.betas_reduce]

    def arch_parameters(self):
        return self._arch_parameters

    def save_arch_parameters(self, save_path):
        torch.save({'arch_parameters': self._arch_parameters}, save_path)

    def load_arch_parameters(self, load_path):
        self._arch_parameters = torch.load(load_path)['arch_parameters']
        (self.alphas_normal, self.alphas_reduce, self.betas_normal, self.betas_reduce) = self._arch_parameters

    def new(self):
        # basic_vqa passes the owning VqaModel on to the twin (basic_vqa model_search.py:139-141); darts_vqa has none
        owner = self._vqa_model() if hasattr(self, '_vqa_model') else None
        extra = (owner,) if owner is not None else ()
        twin = Network(self._C, self._num_classes, self._layers, *extra).to(config.DEVICE)
        for mine, theirs in zip(twin.arch_parameters(), self.arch_parameters()):
            mine.data.copy_(theirs.data)
        return twin

    # ---- forward --------------------------------------------------------------------------------------
    def _plan(self, lib, batch, height, width):
        """Byte offsets of the stem / every cell inside the three arenas, for this input geometry."""
        key = (batch, height, width)
        plans = self.__dict__.setdefault('_pcd_plans', {})
        if key not in plans:
            c_stem = self._stem_multiplier * self._C
            p_off, r_off, n_off = c_stem * 29, 2 * c_stem, 1
            cells, h, w = [], height, width
            for cell in self.cells:
                handle = cell.__dict__['_pcd_handle']
                sz = handle.sizes(lib, batch, h, w)
                cells.append((handle, p_off, r_off, n_off, len(cell._cell_params())))
                p_off += sz.param_floats
                r_off += sz.running_floats
                n_off += sz.nbt_int64
                h, w = sz.out_height, sz.out_width
            plans[key] = (cells, p_off)
        return plans[key]

    def forward(self, input):
        is_eval = pcd_ops.eval_forward(self, input, *self._arch_parameters)
        n, _, h, w = input.shape
        x = input.expand(n, 3, h, w)           # 1-channel inputs are broadcast (model_search.py:150)
        ar = self._arena()
        lib = pcd_ops.N.lib_for(x)
        cells, total = self._plan(lib, n, h, w)
        if total != ar.param_floats:
            raise RuntimeError("parameter arena does not match the kernel layout")
        if is_eval:
            return self._forward_eval(x, ar, cells)
        params = ar.params
        wg = pcd_ops.weight_grads_enabled()
        if wg:
            s0 = s1 = pcd_ops.StemFunction.apply(x, (ar.param_ptr, ar.running_ptr, ar.nbt_ptr), *params[:3])
        else:   # activation-only pass: no autograd edges to the weights at all
            with torch.no_grad():
                s0 = s1 = pcd_ops.StemFunction.apply(x, (ar.param_ptr, ar.running_ptr, ar.nbt_ptr), *params[:3])
        w_normal = w_reduce = None
        pos = 3
        for cell, (handle, p_off, r_off, n_off, n_par) in zip(self.cells, cells):
            if cell.reduction:
                if w_reduce is None:
                    w_reduce = (F.softmax(self.alphas_reduce, dim=-1), _grouped_softmax(self.betas_reduce, self._steps))
                weights, weights2 = w_reduce
            else:
                if w_normal is None:
                    w_normal = (F.softmax(self.alphas_normal, dim=-1), _grouped_softmax(self.betas_normal, self._steps))
                weights, weights2 = w_normal
            handle.param_ptr = ar.param_ptr + 4 * p_off
            handle.running_ptr = ar.running_ptr + 4 * r_off
            handle.nbt_ptr = ar.nbt_ptr + 8 * n_off
            cell_params = params[pos:pos + n_par] if wg else ()
            s0, s1 = s1, pcd_ops.CellFunction.apply(s0, s1, weights, weights2, handle, *cell_params)
            pos += n_par
        out = pcd_ops.AdaptiveAvgPoolFunction.apply(s1, self.output_size)
        return out.flatten(start_dim=1)

    def _forward_eval(self, x, ar, cells):
        """Eval mode (running-statistics BatchNorm), forward only: stem, one launch per node, global pooling."""
        s0 = s1 = pcd_ops.stem_forward_eval(x, ar.param_ptr, ar.running_ptr, self._stem_multiplier * self._C)
        w_normal = (F.softmax(self.alphas_normal, dim=-1), _grouped_softmax(self.betas_normal, self._steps))
        w_reduce = (F.softmax(self.alphas_reduce, dim=-1), _grouped_softmax(self.betas_reduce, self._steps))
        for cell, (handle, p_off, r_off, _, _) in zip(self.cells, cells):
            handle.param_ptr = ar.param_ptr + 4 * p_off
            handle.running_ptr = ar.running_ptr + 4 * r_off
            weights, weights2 = w_reduce if cell.reduction else w_normal
            s0, s1 = s1, pcd_ops.cell_forward_eval(s0, s1, weights, weights2, handle)
        with torch.no_grad():
            out = pcd_ops.AdaptiveAvgPoolFunction.apply(s1, self.output_size)
        return out.flatten(start_dim=1)

    def _loss(self, images, questions, labels):
        # basic_vqa/pcdarts/model_search.py:168-171 (dead code in darts_vqa: no owning model there)
        logits, _ = self._vqa_model()(images, questions)
        return self._criterion(logits, labels)

    # ---- discretisation (model_search.py:218-263) -----------------------------------------------------
    def genotype(self):
        none_idx = PRIMITIVES.index('none')

        def parse(alpha_w, beta_w):
            gene, start = [], 0
            for i in range(self._steps):
                n = i + 2
                scaled = alpha_w[start:start + n] * beta_w[start:start + n, None]
                keep = [k for k in range(scaled.shape[1]) if k != none_idx]
                strength = scaled[:, keep].max(axis=1)
                # two strongest incoming edges; sorted() is stable, ties keep the lower edge index
                for j in sorted(range(n), key=lambda e: -strength[e])[:2]:
                    best = keep[0]
                    for k in keep:
                        if scaled[j][k] > scaled[j][best]:
                            best = k
                    gene.append((PRIMITIVES[best], j))
                start += n
            return gene

        with torch.no_grad():
            an = F.softmax(self.alphas_normal, dim=-1).cpu().numpy()
            ar = F.softmax(self.alphas_reduce, dim=-1).cpu().numpy()
            bn = _grouped_softmax(self.betas_normal, self._steps).cpu().numpy()
            br = _grouped_softmax(self.betas_reduce, self._steps).cpu().numpy()
        concat = range(2 + self._steps - self._multiplier, self._steps + 2)
        return Genotype(normal=parse(an, bn), normal_concat=concat, reduce=parse(ar, br), reduce_concat=concat)
