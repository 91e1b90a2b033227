"""One search step of darts_vqa's Experiment.train (experiment.py:169-200): the alpha-step every
`arch_update_freq` batches, then the w-step — without the dataset / logging / metric glue.

    step = SearchStep(model, architect, optimizer, reducer)
    loss = step.step(train_batch, valid_batch, lr, unrolled=True)
"""
import torch
import torch.nn as nn


class SearchStep:
    def __init__(self, model, architect, optimizer, reducer=None, grad_clip=5.0, qst_only=False):
        self.model = model
        self.architect = architect
        self.optimizer = optimizer
        self.reducer = reducer
        self.grad_clip = grad_clip
        self.qst_only = qst_only
        self.criterion = nn.CrossEntropyLoss()
        self._params = list(model.parameters())

    def _verify_arenas(self):
        for m in self.model.modules():
            ar = m.__dict__.get('_pcd_arena')
            if ar is not None and ar.valid:
                ar.verify()

    def w_step(self, image, question, label):
        """experiment.py:187-200."""
        self._verify_arenas()
        self.optimizer.zero_grad()
        if self.reducer is not None and hasattr(self.model, "_loss_staged"):
            # data parallel: the backward is cut at the image embedding so that the all-reduce of the question-encoder / head
            # gradients overlaps the search network's backward (pcd_dist.staged_grads); .grad is set, not accumulated
            from pcd_dist import staged_grads
            loss, grads, _ = staged_grads(self.model, (image, question, label), self._params, self.reducer, self.qst_only)
            for p, g in zip(self._params, grads):
                p.grad = g
        else:
            loss = self.model._loss(image, question, label, self.qst_only)     # = CE(ans) + CE(qst[:, :-1]) of experiment.py:189-194
            loss.backward()
            if self.reducer is not None:
                self.reducer([p.grad for p in self._params if p.grad is not None])
        if hasattr(self.optimizer, "state_tensors"):       # pcd_flat.FlatAdam: norm, clipping and Adam over the flat runs
            import pcd_flat
            self.last_grad_norm = pcd_flat.clip_grad_norm_(self._params, self.grad_clip)
        else:
            self.last_grad_norm = nn.utils.clip_grad_norm_(self._params, self.grad_clip)     # the norm BEFORE clipping
        self.optimizer.step()
        return loss.detach()

    def alpha_step(self, train_batch, valid_batch, lr, unrolled=True):
        """experiment.py:176-185."""
        self.architect.step(*train_batch, *valid_batch, lr, None, unrolled=unrolled)

    def step(self, train_batch, valid_batch, lr, unrolled=True):
        self.alpha_step(train_batch, valid_batch, lr, unrolled)
        return self.w_step(*train_batch)


class _TrainingState:
    """Snapshot of everything a training step mutates (weights, BN buffers, alphas/betas, optimizer moments and step
    counters), restorable IN PLACE — the tensors keep their addresses, so a CUDA graph captured afterwards still points
    at them.  Used to undo the warm-up steps a graph capture needs: construction must not consume training steps."""

    def __init__(self, modules, arch_tensors, optimizers):
        # hold the parameter / buffer OBJECTS, not their .data: the first forward pass re-binds .data to views of one
        # flat arena (pcd_ops.Arena), and the values must go back into whatever storage is live at restore time
        self.holders = []
        for m in modules:
            self.holders += list(m.parameters()) + list(m.buffers())
        self.holders += list(arch_tensors)
        self.saved = [t.detach().clone() for t in self.holders]
        self.optimizers = list(optimizers)
        self.opt_saved = [{id(p): {k: (v.clone() if torch.is_tensor(v) else v) for k, v in st.items()}
                           for p, st in opt.state.items()} for opt in self.optimizers]
        self.flat_state = [t for opt in self.optimizers if hasattr(opt, "state_tensors") for t in opt.state_tensors()]
        self.flat_saved = [t.clone() for t in self.flat_state]

    @property
    def tensors(self):
        return [t.data for t in self.holders]

    def restore(self):
        with torch.no_grad():
            torch._foreach_copy_(self.tensors, self.saved)
            if self.flat_state:
                torch._foreach_copy_(self.flat_state, self.flat_saved)
            for opt, saved in zip(self.optimizers, self.opt_saved):
                for p, st in opt.state.items():
                    old = saved.get(id(p), {})
                    for k, v in st.items():
                        if torch.is_tensor(v):      # state created by the warm-up goes back to its initial zeros
                            v.copy_(old[k]) if k in old else v.zero_()


class GraphedSearchStep:
    """The whole search step (alpha-step + w-step, ~4000 kernel launches and a few thousand torch ops) captured
    once in a CUDA graph and replayed: the step is otherwise host-bound.  Inputs are copied into static device
    buffers; the learning rate is baked in at capture (re-capture when the schedule changes it).

    Requirements: optimizers created with capturable=True (Adam keeps its step counter on the device), shapes
    fixed.  Under data parallelism the NCCL all-reduces of the GradReducer are captured with the rest (bench.py does
    so at N > 1).  The warm-up steps the capture needs run on the first batch and are then UNDONE: weights, BN buffers,
    alphas and both optimizers' state are restored in place, so the first replay is training step 1 exactly as in the
    eager path (dropout draws aside).
    """

    def __init__(self, step, train_batch, valid_batch, lr, unrolled=True, warmup=3):
        self.step_obj = step
        self.lr, self.unrolled = lr, unrolled
        self.train = [t.clone() for t in train_batch]
        self.valid = [t.clone() for t in valid_batch]
        step.architect.device_scalars = True
        # high priority: with weight-grad overlap on, the library's low-priority stream only fills the SMs this one leaves idle
        side = torch.cuda.Stream(priority=-1)
        side.wait_stream(torch.cuda.current_stream())
        modules = [step.model] + ([step.architect._twin] if getattr(step.architect, "_twin", None) is not None else [])
        snap = _TrainingState(modules, step.model.arch_parameters(), [step.optimizer, step.architect.optimizer])
        with torch.cuda.stream(side):                 # warm-up on a side stream (allocator, cuDNN/cuBLAS handles)
            for _ in range(warmup):
                step.step(self.train, self.valid, lr, unrolled)
            snap.restore()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=side):
            self.loss = step.step(self.train, self.valid, lr, unrolled)

    def __call__(self, train_batch=None, valid_batch=None):
        if train_batch is not None:
            for dst, src in zip(self.train, train_batch):
                dst.copy_(src, non_blocking=True)
        if valid_batch is not None:
            for dst, src in zip(self.valid, valid_batch):
                dst.copy_(src, non_blocking=True)
        self.graph.replay()
        return self.loss


def make_capturable(optimizer):
    """Adam keeps `step` on the host unless capturable; flip an existing optimizer (state included) to the device form."""
    for group in optimizer.param_groups:
        group["capturable"] = True
        for p in group["params"]:
            st = optimizer.state.get(p)
            if st and torch.is_tensor(st.get("step")) and st["step"].device != p.device:
                st["step"] = st["step"].to(p.device)


class GraphedLctStep:
    """ArchitectLct.step (basic_vqa/pcdarts/architect_lct.py:32-92: 6 forward / 5 backward search-net passes, 3 greedy decodes,
    the W-model passes and the two finite-difference HVPs) captured once in a CUDA graph and replayed.  The learning rates are
    baked in at capture.  Both question decoders are captured: greedy (argmax) and sampled (ef_model.qst_encoder.deterministic =
    False, inside the decode kernel's envelope), which draws its seed on the device, so every replay samples fresh words."""

    def __init__(self, architect, train_batch, valid_batch, ef_lr, w_lr, warmup=2):
        self.architect = architect
        self.train = [t.clone() for t in train_batch]
        self.valid = [t.clone() for t in valid_batch]
        architect.device_scalars = True
        make_capturable(architect.optimizer)
        side = torch.cuda.Stream(priority=-1)
        side.wait_stream(torch.cuda.current_stream())
        snap = _TrainingState([architect.ef_model, architect.w_model], architect.ef_model.arch_parameters(),
                              [architect.optimizer])      # ArchitectLct.step only steps the architecture optimizer
        with torch.cuda.stream(side):
            for _ in range(warmup):
                architect.step(*self.train, *self.valid, ef_lr, w_lr)
            snap.restore()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=side):
            architect.step(*self.train, *self.valid, ef_lr, w_lr)
        self.loss = architect.last["unrolled_loss"]

    def __call__(self, train_batch=None, valid_batch=None):
        for dst_list, src_list in ((self.train, train_batch), (self.valid, valid_batch)):
            if src_list is not None:
                for dst, src in zip(dst_list, src_list):
                    dst.copy_(src, non_blocking=True)
        self.graph.replay()
        return self.loss
