"""B200-native drop-in for the reference's ``biGRU_model`` module.

``BiGRU`` keeps the class surface of /root/reference/biGRU_model.py:8-286 - constructor
argument order (:32-33), attribute names (:39-47), submodule names ``dropout`` /
``spatial_dropout1d`` / ``gru`` / ``linear`` (so ``model_params.pt`` loads unchanged),
``forward(input_seq, hidden=None)`` (:63), ``add_loss_fn`` / ``add_optimizer`` / ``add_device``
(:141-159), ``train_model`` (:162) and ``evaluate_model`` (:227) with the same return tuples -
but every floating-point operation of forward/backward, the loss, gradient clipping and the
Adam update run in hand-written sm_100a CUDA kernels behind the C ABI of
``libbigru_b200.so`` (include/bigru_b200.h).  PyTorch only owns device memory, streams and the
process group.  There is no CPU path: parameters must live on a CUDA device.
"""
from __future__ import annotations

import math
import os
from typing import Optional

import numpy as np
import torch
import torch.nn as nn

if __package__:
    from . import _lib
    from .parallel import allreduce_flat_
else:
    # drop-in route of the reference's callers (`predict.py:16`, the notebook): this directory itself is on sys.path and
    # the module is imported top-level as `biGRU_model`; bind the sibling modules through the package
    import importlib as _importlib
    import sys as _sys
    _here = os.path.dirname(os.path.abspath(__file__))
    if os.path.dirname(_here) not in _sys.path:
        _sys.path.insert(0, os.path.dirname(_here))
    _lib = _importlib.import_module(os.path.basename(_here) + "._lib")
    allreduce_flat_ = _importlib.import_module(os.path.basename(_here) + ".parallel").allreduce_flat_

_PRECISIONS = {"fp32": _lib.PREC_FP32, "bf16": _lib.PREC_BF16, "bf16x3": _lib.PREC_BF16X3}


def _stream_ptr(device=None):
    """Raw cudaStream_t of torch's current stream ON THE MODEL'S DEVICE (not the process-wide current device)."""
    return torch.cuda.current_stream(device).cuda_stream


class _GRUWeights(nn.Module):
    """Holds the recurrent parameters under torch.nn.GRU's names, shapes, registration order and
    initialisation (U(-1/sqrt(H), 1/sqrt(H)), drawn in registration order), i.e. what
    biGRU_model.py:54-56 constructs.  It has no forward of its own: the recurrence runs inside
    libbigru_b200."""

    def __init__(self, input_size, hidden_size, num_layers, bidirectional, dropout):
        super().__init__()
        self.input_size, self.hidden_size, self.num_layers = input_size, hidden_size, num_layers
        self.bidirectional, self.dropout, self.batch_first, self.bias = bidirectional, float(dropout), True, True
        dirs = 2 if bidirectional else 1
        for layer in range(num_layers):
            fan = input_size if layer == 0 else hidden_size * dirs
            for d in range(dirs):
                sfx = f"l{layer}" + ("_reverse" if d else "")
                self.register_parameter(f"weight_ih_{sfx}", nn.Parameter(torch.empty(3 * hidden_size, fan)))
                self.register_parameter(f"weight_hh_{sfx}", nn.Parameter(torch.empty(3 * hidden_size, hidden_size)))
                self.register_parameter(f"bias_ih_{sfx}", nn.Parameter(torch.empty(3 * hidden_size)))
                self.register_parameter(f"bias_hh_{sfx}", nn.Parameter(torch.empty(3 * hidden_size)))
        bound = 1.0 / math.sqrt(hidden_size) if hidden_size > 0 else 0.0
        with torch.no_grad():
            for p in self.parameters():
                p.uniform_(-bound, bound)

    def forward(self, *args, **kwargs):
        raise RuntimeError("BiGRU.gru only stores parameters; call BiGRU.forward (libbigru_b200 runs the recurrence)")


class _Plan:
    """A C plan plus its device workspaces for one (B, T) shape."""

    def __init__(self, model: "BiGRU", B: int, T: int, device):
        lib = _lib.load()
        _lib.check(lib.bigru_device_check(device.index if device.index is not None else torch.cuda.current_device()),
                   "bigru_device_check")
        h = _lib.C.c_void_p()
        _lib.check(lib.bigru_plan_create(B, T, model.n_features, model.plan_hidden(B), model.n_layers, model.output_size,
                                         int(model.bidirectional), _PRECISIONS[model.resolved_precision(B)], _lib.C.byref(h)),
                   "bigru_plan_create")
        self.handle, self.B, self.T, self.device = h, B, T, device
        a, b = _lib.C.c_size_t(), _lib.C.c_size_t()
        _lib.check(lib.bigru_workspace_bytes(h, _lib.C.byref(a), _lib.C.byref(b)), "bigru_workspace_bytes")
        self.stash_bytes, self.scratch_bytes = a.value, b.value
        self.scratch = torch.empty(max(self.scratch_bytes, 16), dtype=torch.uint8, device=device)
        self._free_stash = []

    def acquire_stash(self):
        if self._free_stash:
            return self._free_stash.pop()
        return torch.empty(max(self.stash_bytes, 16), dtype=torch.uint8, device=self.device)

    def release_stash(self, s):
        if len(self._free_stash) < 2:
            self._free_stash.append(s)

    def __del__(self):
        try:
            if self.handle:
                _lib.load().bigru_plan_destroy(self.handle)
        except Exception:
            pass


class _BiGRUFunction(torch.autograd.Function):
    """autograd boundary: forward/backward are single calls into the C ABI."""

    @staticmethod
    def forward(ctx, model, x, h0, *params):
        lib = _lib.load()
        B = x.shape[0]
        Bp = model._padded_batch(B)
        if Bp != B:                                       # whole batch tiles on the tensor-core paths: zero rows appended
            xp = x.new_zeros((Bp,) + tuple(x.shape[1:]))
            xp[:B] = x
            x = xp
            if h0 is not None:
                hp = h0.new_zeros(h0.shape[0], Bp, h0.shape[2])
                hp[:, :B] = h0
                h0 = hp
        plan = model._plan_for(x)
        ctx.dev_guard = torch.cuda.device(x.device)      # the C ABI launches on the CURRENT device: make it the model's
        ctx.dev_guard.__enter__()
        try:
            out = _BiGRUFunction._forward(ctx, lib, plan, model, x, h0, Bp)
            ctx.real_batch = B
            model._last_batch = B
            if Bp != B:
                model._last_hidden = model._last_hidden[:, :B]
                out = out[:B]
            return out
        finally:
            ctx.dev_guard.__exit__(None, None, None)

    @staticmethod
    def _forward(ctx, lib, plan, model, x, h0, B):
        Hp = model.plan_hidden(B)
        pflat = model._plan_params()                     # zero-padded hidden units scattered in when Hp > hidden_size
        h0 = model._pad_last(h0, Hp)
        logits = torch.empty(B, model.output_size, device=x.device, dtype=torch.float32)
        hn = torch.empty(model.n_layers * model.n_directions, B, Hp, device=x.device, dtype=torch.float32)
        need_grad = any(ctx.needs_input_grad)        # grad mode is off inside Function.forward; ask the ctx
        stash = plan.acquire_stash()
        training = bool(model.training and model.dropout_p > 0)
        seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if training else 0
        model._last_seed = seed                       # the dropout masks are a pure function of (seed, element index)
        _lib.check(lib.bigru_forward(plan.handle, _lib.ptr(pflat), _lib.ptr(x), _lib.ptr(h0),
                                     float(model.dropout_p), int(bool(model.spatial_dropout)), int(training), seed,
                                     _lib.ptr(stash), _lib.ptr(plan.scratch), _lib.ptr(logits), _lib.ptr(hn),
                                     _stream_ptr(x.device)), "bigru_forward")
        model._last_hidden = hn if Hp == model.hidden_size else hn[..., :model.hidden_size]
        ctx.pflat = pflat if need_grad else None
        model._last_plan_stash = (plan, stash)
        if need_grad:
            ctx.model, ctx.plan, ctx.stash, ctx.seed, ctx.training = model, plan, stash, seed, training
            ctx.save_for_backward(x, h0 if h0 is not None else torch.empty(0, device=x.device))
            ctx.has_h0 = h0 is not None
        else:
            plan.release_stash(stash)
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        lib = _lib.load()
        model, plan = ctx.model, ctx.plan
        x, h0 = ctx.saved_tensors
        h0 = h0 if ctx.has_h0 else None
        dlogits = dlogits.contiguous().float()
        B, Bp = ctx.real_batch, x.shape[0]
        if Bp != B:                                       # padded rows: zero upstream gradient
            dl = dlogits.new_zeros(Bp, dlogits.shape[1])
            dl[:B] = dlogits
            dlogits = dl
        grads = torch.empty_like(ctx.pflat)
        dx = torch.empty_like(x) if ctx.needs_input_grad[1] else None
        dh0 = torch.empty_like(h0) if (h0 is not None and ctx.needs_input_grad[2]) else None
        with torch.cuda.device(x.device):
            _lib.check(lib.bigru_backward(plan.handle, _lib.ptr(ctx.pflat), _lib.ptr(x), _lib.ptr(h0),
                                          float(model.dropout_p), int(bool(model.spatial_dropout)), int(ctx.training),
                                          ctx.seed, _lib.ptr(ctx.stash), _lib.ptr(plan.scratch), _lib.ptr(dlogits),
                                          _lib.ptr(grads), _lib.ptr(dx), _lib.ptr(dh0), _stream_ptr(x.device)), "bigru_backward")
        plan.release_stash(ctx.stash)
        ctx.stash = None
        if Bp != B:
            dx = dx[:B] if dx is not None else None
            dh0 = dh0[:, :B] if dh0 is not None else None
        grads = model._plan_grads(grads)                  # drop the padded hidden units' entries
        if dh0 is not None and dh0.shape[-1] != model.hidden_size:
            dh0 = dh0[..., :model.hidden_size]
        ctx.pflat = None
        pg = tuple(grads[o:o + n].view(shape) for (o, n, shape) in model._views)
        return (None, dx, dh0) + pg


class BiGRU(nn.Module):
    """Bidirectional GRU classifier (reference: biGRU_model.py:8).

    Parameters (same order and defaults as the reference, :32-33): hidden_size, n_features,
    output_size, n_layers=1, clip=50, dropout=0.2, spatial_dropout=True, bidirectional=True.
    Extra keyword ``precision``:
      "fp32"    FFMA kernels, exact transcendental functions; any shape (the exact path),
      "bf16x3"  fp32-class on tcgen05 tensor cores (every operand a (hi, lo) bf16 pair, fp32 accumulation / state /
                gradients): meets the reference's 1e-4 logits tolerance; H in {128, 256} (other batch sizes than whole 32-row tiles
                run zero-padded, any feature count),
      "bf16"    single bf16 operands on tcgen05, fp32 accumulation and state (fastest, ~3e-3 on logits); H in {128, 256, 512},
      "auto"    "bf16x3" for hidden sizes up to 256 (smaller models run zero-padded to 128 / 256 hidden units), "fp32" beyond.
    Every precision takes an initial hidden state (``forward(input_seq, hidden)``, ``train_step(x, target, hidden)``) and returns
    its gradient through autograd; on the tensor-core paths W_hh·hidden is formed in fp32 and hidden enters the first step's gate
    math and dW_hh in fp32 (the smaller models' zero padding extends to it).
    A train step with ``hidden`` runs as plain launches (CUDA-graph replay is for steps without it).
    Default: $BIGRU_B200_PRECISION or "auto" (the reference tolerance at tensor-core speed wherever the kernels apply).
    """

    def __init__(self, hidden_size, n_features, output_size, n_layers=1, clip=50, dropout=0.2,
                 spatial_dropout=True, bidirectional=True, precision: Optional[str] = None):
        super().__init__()
        self.hidden_size = hidden_size
        self.n_features = n_features
        self.output_size = output_size
        self.n_layers = n_layers
        self.clip = clip
        self.dropout_p = dropout
        self.spatial_dropout = spatial_dropout
        self.bidirectional = bidirectional
        self.n_directions = 2 if bidirectional else 1
        self.precision = precision or os.environ.get("BIGRU_B200_PRECISION", "auto")
        if self.precision != "auto" and self.precision not in _PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_PRECISIONS) + ['auto']}")

        # same submodule names and construction order as the reference (:50-60) so that a given
        # torch.manual_seed produces the same initial weights and state_dict keys
        self.dropout = nn.Dropout(self.dropout_p)
        if self.spatial_dropout:
            self.spatial_dropout1d = nn.Dropout2d(self.dropout_p)
        self.gru = _GRUWeights(n_features, hidden_size, n_layers, bidirectional, 0 if n_layers == 1 else dropout)
        self.linear = nn.Linear(hidden_size * 3, output_size)

        self.device = torch.device("cpu")
        self.loss_fn = None
        self.optimizer = None
        self._flat = None            # all parameters, one contiguous fp32 vector (C-ABI order)
        self._views = []             # (offset, numel, shape) per parameter in C-ABI order
        self._plans = {}
        self._adam = None            # fused-step optimiser state (flat m, v, step)
        self._dp_group = None
        self._dp_world = 1
        self._last_hidden = None
        self._last_plan_stash = None
        self._last_seed = 0
        self._graphs = {}
        self.use_cuda_graph = os.environ.get("BIGRU_B200_CUDA_GRAPH", "1") != "0"
        self._loss_cache = {}
        self._flatten()

    # ------------------------------------------------------------------ parameter storage
    def _ordered_params(self):
        out = []
        for layer in range(self.n_layers):
            for d in range(self.n_directions):
                sfx = f"l{layer}" + ("_reverse" if d else "")
                for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
                    out.append(getattr(self.gru, f"{n}_{sfx}"))
        out += [self.linear.weight, self.linear.bias]
        return out

    def _flatten(self):
        """(Re)pack every parameter into one contiguous vector and make the nn.Parameters views of it,
        keeping the Parameter objects (optimisers hold references to them)."""
        params = self._ordered_params()
        dev = params[0].device
        total = sum(p.numel() for p in params)
        flat = torch.empty(total, dtype=torch.float32, device=dev)
        views, off = [], 0
        with torch.no_grad():
            for p in params:
                n = p.numel()
                flat[off:off + n].copy_(p.detach().reshape(-1).to(device=dev, dtype=torch.float32))
                p.data = flat[off:off + n].view(p.shape)
                views.append((off, n, tuple(p.shape)))
                off += n
        old = getattr(self, "_adam", None)
        self._flat, self._views = flat, views
        self._plans = {}
        self._graphs = {}
        self._adam = None
        if old is not None and old["m"].numel() == total:        # keep the Adam moments across a re-flatten (.to() / .cuda())
            st = self._fused_state(dev)
            st["m"].copy_(old["m"].to(dev)); st["v"].copy_(old["v"].to(dev))
            st["step"] = old["step"]
            st["dstep"].fill_(old["step"])
            self._mirror_optimizer_state()

    def _is_flat(self):
        f = self._flat
        if f is None:
            return False
        base = f.data_ptr()
        for p, (off, n, _) in zip(self._ordered_params(), self._views):
            if p.device != f.device or p.dtype != torch.float32 or p.data_ptr() != base + 4 * off:
                return False
        return True

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)       # .cuda() / .to() create fresh tensors per parameter
        self._flatten()
        return out

    def flat_parameters(self) -> torch.Tensor:
        if not self._is_flat():
            self._flatten()
        return self._flat

    # ------------------------------------------------------------------ plans
    def resolved_precision(self, batch: int = 0) -> str:
        """The precision a batch runs at ("auto": the fp32-class tensor-core path wherever it applies, i.e. hidden_size <= 256)."""
        if self.precision != "auto":
            return self.precision
        return "bf16x3" if self.hidden_size <= 256 else "fp32"

    def plan_hidden(self, batch: int = 0) -> int:
        """Hidden size of the C plan.  The tensor-core kernels exist for 128 / 256 (/ 512 at "bf16") hidden units; smaller models run
        ZERO-PADDED to the next of these: a padded unit has zero weights and biases, so r = z = 1/2, n = 0 and its state stays 0
        from h0 = 0 on; it feeds zero columns of W_hh / W_ih / the head.  Logits, loss and the gradients of the real parameters are
        exactly those of the unpadded model (up to summation order); the padded gradient entries are dropped."""
        prec, H = self.resolved_precision(batch), self.hidden_size
        sizes = {"bf16x3": (128, 256), "bf16": (128, 256, 512)}.get(prec, ())
        for hp in sizes:
            if H <= hp:
                return hp
        return H

    def _pad_map(self, dev):
        """(index tensor, padded parameter count): position of every real parameter inside the padded plan's flat vector."""
        Hp, H = self.plan_hidden(), self.hidden_size
        if Hp == H:
            return None
        key = (Hp, dev.index)
        hit = getattr(self, "_pad_cache", None)
        if hit is not None and hit[0] == key:
            return hit[1]
        D, L, F, C = self.n_directions, self.n_layers, self.n_features, self.output_size
        idx, off_p = [], 0

        def rows(n_cols_small, n_cols_pad, col_map):
            # a [3H][cols] block -> padded [3Hp][cols_pad]: row g*H + j -> g*Hp + j, column through col_map
            r = (np.arange(3)[:, None] * Hp + np.arange(H)[None, :]).reshape(-1)
            return (r[:, None] * n_cols_pad + col_map[None, :]).reshape(-1)

        for l in range(L):
            I, Ip = (F, F) if l == 0 else (D * H, D * Hp)
            cm = np.arange(F) if l == 0 else (np.arange(D)[:, None] * Hp + np.arange(H)[None, :]).reshape(-1)
            for d in range(D):
                idx.append(off_p + rows(I, Ip, cm)); off_p += 3 * Hp * Ip                     # W_ih
                idx.append(off_p + rows(H, Hp, np.arange(H))); off_p += 3 * Hp * Hp           # W_hh
                b = (np.arange(3)[:, None] * Hp + np.arange(H)[None, :]).reshape(-1)
                idx.append(off_p + b); off_p += 3 * Hp                                        # b_ih
                idx.append(off_p + b); off_p += 3 * Hp                                        # b_hh
        cmh = (np.arange(3)[:, None] * Hp + np.arange(H)[None, :]).reshape(-1)                # head: last | max | avg, H wide each
        idx.append(off_p + (np.arange(C)[:, None] * 3 * Hp + cmh[None, :]).reshape(-1)); off_p += C * 3 * Hp
        idx.append(off_p + np.arange(C)); off_p += C
        index = torch.from_numpy(np.concatenate(idx).astype(np.int64)).to(dev)
        assert index.numel() == self._flat.numel()
        self._pad_cache = (key, (index, off_p))
        return self._pad_cache[1]

    def _plan_params(self, buf=None):
        """The flat parameter vector as the C plan sees it (zero-padded hidden units scattered in when plan_hidden() > hidden_size)."""
        pm = self._pad_map(self._flat.device)
        if pm is None:
            return self._flat
        index, P = pm
        if buf is None:
            buf = torch.zeros(P, device=self._flat.device, dtype=torch.float32)
        buf.index_copy_(0, index, self._flat.detach())
        return buf

    def _plan_grads(self, pgrad, out=None):
        pm = self._pad_map(self._flat.device)
        if pm is None:
            return pgrad
        return torch.index_select(pgrad, 0, pm[0], out=out) if out is not None else torch.index_select(pgrad, 0, pm[0])

    @staticmethod
    def _pad_last(t, Hp):
        """[.., .., H] -> [.., .., Hp] with zeros (initial hidden states)."""
        if t is None or t.shape[-1] == Hp:
            return t
        out = t.new_zeros(tuple(t.shape[:-1]) + (Hp,))
        out[..., :t.shape[-1]] = t
        return out

    def _padded_batch(self, batch: int) -> int:
        """The tensor-core paths work on whole batch tiles (32 rows at bf16x3, 16 at bf16): other batch sizes run zero-padded
        to the next multiple.  Batch rows are independent and the padded rows receive a zero upstream gradient, so logits,
        loss and every gradient of the real rows are unchanged."""
        prec = self.resolved_precision(batch)
        mult = 32 if (prec == "bf16x3" or (prec == "bf16" and self.plan_hidden(batch) == 512)) else (16 if prec == "bf16" else 1)
        return (batch + mult - 1) // mult * mult

    def _plan_for(self, x) -> _Plan:
        key = (int(x.shape[0]), int(x.shape[1]), self.resolved_precision(int(x.shape[0])), x.device.index)
        plan = self._plans.get(key)
        if plan is None:
            if len(self._plans) > 8:
                self._plans.clear()
            plan = self._plans[key] = _Plan(self, key[0], key[1], x.device)
        return plan

    def _prepare_input(self, input_seq, hidden):
        if not self._is_flat():
            self._flatten()
        dev = self._flat.device
        if dev.type != "cuda":
            raise RuntimeError("BiGRU (B200-native) has no CPU path: move the model to a CUDA device with .cuda() first")
        if input_seq.dim() != 3 or input_seq.shape[2] != self.n_features:
            raise ValueError(f"input_seq must be [batch, seq_len, {self.n_features}], got {tuple(input_seq.shape)}")
        x = input_seq.to(device=dev, dtype=torch.float32, non_blocking=True).contiguous()
        h0 = None
        if hidden is not None:
            want = (self.n_layers * self.n_directions, x.shape[0], self.hidden_size)
            if tuple(hidden.shape) != want:
                raise RuntimeError(f"Expected hidden size {want}, got {tuple(hidden.shape)}")
            h0 = hidden.to(device=dev, dtype=torch.float32).contiguous()
        return x, h0

    def pooled_argmax(self) -> torch.Tensor:
        """argmax_t of the max-pooled direction sum [batch, hidden] as taken by the last ``forward`` (the routing of the
        max-pool gradient, biGRU_model.py:125).  Valid until the next forward of the same shape."""
        plan, stash = self._last_plan_stash
        off = _lib.C.c_size_t()
        _lib.check(_lib.load().bigru_stash_argmax_offset(plan.handle, _lib.C.byref(off)), "bigru_stash_argmax_offset")
        Hp = self.plan_hidden(plan.B)
        n = plan.B * Hp * 4
        return stash[off.value:off.value + n].view(torch.int32).view(plan.B, Hp)[:getattr(self, "_last_batch", plan.B), :self.hidden_size].clone()

    # ------------------------------------------------------------------ reference surface
    def forward(self, input_seq, hidden=None):
        """Logits [batch, output_size] (biGRU_model.py:63-138)."""
        x, h0 = self._prepare_input(input_seq, hidden)
        self.batch_size, self.input_length = x.size(0), x.size(1)          # as the reference sets (:82-85)
        return _BiGRUFunction.apply(self, x, h0, *self._ordered_params())

    def add_loss_fn(self, loss_fn):
        self.loss_fn = loss_fn

    def add_optimizer(self, optimizer):
        self.optimizer = optimizer
        self._adam = None
        self._graphs = {}

    def add_device(self, device=torch.device("cpu")):
        self.device = device

    def enable_data_parallel(self, process_group=None):
        """Batch data parallelism: one process per GPU, every rank holds a replica and a batch shard;
        train_step/train_model all-reduce the flat gradient once per step (NCCL over NVLink)."""
        import torch.distributed as dist
        self._dp_group = process_group if process_group is not None else dist.group.WORLD
        self._dp_world = dist.get_world_size(self._dp_group)

    # ------------------------------------------------------------------ fused training step
    def _loss_spec(self):
        fn = self.loss_fn
        if isinstance(fn, nn.CrossEntropyLoss):
            if fn.weight is None and fn.reduction == "mean" and getattr(fn, "label_smoothing", 0.0) == 0.0 \
                    and fn.ignore_index == -100:
                return _lib.LOSS_CE, None, None
        elif isinstance(fn, nn.BCEWithLogitsLoss):
            per_class = lambda w: w is None or w.numel() in (1, self.output_size)      # per-element weights: autograd path
            if fn.reduction == "mean" and per_class(fn.weight) and per_class(fn.pos_weight):
                return _lib.LOSS_BCE, fn.weight, fn.pos_weight
        elif isinstance(fn, nn.MultiLabelSoftMarginLoss):
            if fn.weight is None and fn.reduction == "mean":
                return _lib.LOSS_MLSM, None, None
        return None

    def _adam_spec(self):
        opt = self.optimizer
        if not isinstance(opt, torch.optim.Adam) or len(opt.param_groups) != 1:
            return None
        g = opt.param_groups[0]
        if g.get("weight_decay", 0) != 0 or g.get("amsgrad", False) or g.get("maximize", False):
            return None
        mine = {id(p) for p in self._ordered_params()}
        if {id(p) for p in g["params"]} != mine:
            return None
        return g

    def can_fuse_step(self) -> bool:
        return self._loss_spec() is not None and self._adam_spec() is not None

    def _loss_vec(self, w, C):
        """Per-class loss weight as a device vector.  Cached (and kept alive across the asynchronous C
        calls) until the source tensor changes."""
        if w is None:
            return None
        key = (id(w), w._version, C)
        hit = self._loss_cache.get(key)
        if hit is None:
            v = w.detach().to(device=self._flat.device, dtype=torch.float32).reshape(-1)
            if v.numel() == 1:
                v = v.expand(C)
            if v.numel() != C:
                raise ValueError("loss weight must have one entry per class")
            if len(self._loss_cache) > 8:
                self._loss_cache.clear()
            hit = self._loss_cache[key] = v.contiguous()
        return hit

    def _fused_state(self, dev):
        """Optimiser state of the fused step.  The flat gradient and the scalar loss share one buffer (``gext`` = P gradients
        + 1 loss), so that data parallelism needs exactly one all-reduce per step.  ``step`` lives on the device too
        (``dstep``), so that a captured CUDA graph of the step stays valid from one step to the next."""
        st = self._adam
        if st is None:
            P = self._flat.numel()
            gext = torch.empty(P + 1, device=dev, dtype=torch.float32)
            st = self._adam = {"m": torch.zeros_like(self._flat), "v": torch.zeros_like(self._flat), "step": 0,
                               "dstep": torch.zeros(1, device=dev, dtype=torch.int32),
                               "gext": gext, "grad": gext[:P], "loss": gext[P:P + 1],
                               "scal": torch.zeros(2, device=dev, dtype=torch.float32)}
            pm = self._pad_map(dev)
            if pm is not None:                                # zero-padded hidden units (plan_hidden): the plan's own parameter / gradient vectors
                st["pflat"] = torch.zeros(pm[1], device=dev, dtype=torch.float32)
                st["pgrad"] = torch.empty(pm[1], device=dev, dtype=torch.float32)
            self._import_optimizer_state(st)
            self._mirror_optimizer_state()
        return st

    @staticmethod
    def _bump_step(st, k):
        st["step"] += k
        ms = st.get("mirror_steps")
        if ms:
            torch._foreach_add_(ms, float(k))

    def _import_optimizer_state(self, st):
        """Moments the user's torch.optim.Adam already holds (generic steps taken before, or a loaded optimizer.state_dict())
        become the fused step's flat moments."""
        opt = getattr(self, "optimizer", None)
        if opt is None:
            return
        steps = []
        for p, (off, n, _) in zip(self._ordered_params(), self._views):
            ps = opt.state.get(p)
            if not ps or "exp_avg" not in ps:
                return
            steps.append(int(float(ps["step"])) if "step" in ps else 0)
        if len(set(steps)) != 1:
            return
        with torch.no_grad():
            for p, (off, n, _) in zip(self._ordered_params(), self._views):
                ps = opt.state[p]
                st["m"][off:off + n].copy_(ps["exp_avg"].reshape(-1).to(st["m"].device))
                st["v"][off:off + n].copy_(ps["exp_avg_sq"].reshape(-1).to(st["v"].device))
        st["step"] = steps[0]
        st["dstep"].fill_(steps[0])

    def _mirror_optimizer_state(self):
        """optimizer.state[p] = views of the flat moments + a step tensor, in torch.optim.Adam's own format: optimizer.state_dict()
        checkpoints carry the fused step's moments, and a later generic optimizer.step() continues from them (in place)."""
        opt, st = getattr(self, "optimizer", None), self._adam
        if opt is None or st is None or self._adam_spec() is None:
            return
        for p, (off, n, shape) in zip(self._ordered_params(), self._views):
            opt.state[p] = {"step": torch.tensor(float(st["step"])), "exp_avg": st["m"][off:off + n].view(shape),
                            "exp_avg_sq": st["v"][off:off + n].view(shape)}
        st["mirror_steps"] = [opt.state[p]["step"] for p in self._ordered_params()]

    def _launch_fwd_loss_bwd(self, lib, plan, x, h0, tgt, kind, wv, pwv, denom, logits, dlogits, stash, args, st, s, part="all"):
        """part = "all": forward, loss, backward.  Data parallelism splits the backward so that the all-reduce of the upper layers'
        gradients overlaps the lowest layer's backward: "upper" = forward + loss + layers L-1 .. 1 (+ head), "lower" = layer 0."""
        # the loss sees the REAL batch rows (tgt's); logits / dlogits may carry zero-padded rows behind them (whole batch tiles)
        B, C = tgt.shape[0], logits.shape[1]
        padded = "pflat" in st
        pflat = (self._plan_params(st["pflat"]) if part != "lower" else st["pflat"]) if padded else self._flat
        pgrad = st["pgrad"] if padded else st["grad"]
        if part != "lower":
            _lib.check(lib.bigru_forward(plan.handle, _lib.ptr(pflat), _lib.ptr(x), _lib.ptr(h0), *args,
                                         _lib.ptr(stash), _lib.ptr(plan.scratch), _lib.ptr(logits), None, s), "bigru_forward")
            _lib.check(lib.bigru_loss(kind, _lib.ptr(logits), _lib.ptr(tgt), _lib.ptr(wv), _lib.ptr(pwv), B, C, denom,
                                      _lib.ptr(st["loss"]), _lib.ptr(dlogits), s), "bigru_loss")
        if part == "all":
            _lib.check(lib.bigru_backward(plan.handle, _lib.ptr(pflat), _lib.ptr(x), _lib.ptr(h0), *args,
                                          _lib.ptr(stash), _lib.ptr(plan.scratch), _lib.ptr(dlogits), _lib.ptr(pgrad),
                                          None, None, s), "bigru_backward")
        else:
            lo_hi = (self.n_layers - 1, 1) if part == "upper" else (0, 0)
            _lib.check(lib.bigru_backward_layers(plan.handle, _lib.ptr(pflat), _lib.ptr(x), _lib.ptr(h0), *args,
                                                 _lib.ptr(stash), _lib.ptr(plan.scratch), _lib.ptr(dlogits), _lib.ptr(pgrad),
                                                 None, None, lo_hi[0], lo_hi[1], s), "bigru_backward_layers")
        if padded and part != "upper":
            self._plan_grads(pgrad, out=st["grad"])

    def _dp_split(self, st) -> int:
        """Offset (in the flat gradient) where the upper layers' parameters start, or 0 when the data-parallel step is not split:
        needs more than one layer, a tensor-core plan (bigru_backward_layers) and no hidden-size padding (the padded plan's
        gradients are gathered only after the whole backward)."""
        if self._dp_world <= 1 or self.n_layers < 2 or "pflat" in st or self.resolved_precision() == "fp32":
            return 0
        if os.environ.get("BIGRU_B200_DP_OVERLAP", "0") != "1":      # opt-in: measured no faster (two collectives cost more than the overlap wins)
            return 0
        per_dir0 = 3 * self.hidden_size * (self.n_features + self.hidden_size + 2)
        return self.n_directions * per_dir0

    def _dp_allreduce_overlapped(self, st, split, dev, lower):
        """All-reduce of [split, P] + loss on a side stream (issued after the upper layers' backward), `lower()` = the lowest
        layer's backward on the main stream meanwhile, then the all-reduce of [0, split) and the join."""
        main = torch.cuda.current_stream(dev)
        side = st.get("side")
        if side is None:
            side = st["side"] = torch.cuda.Stream(device=dev)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            allreduce_flat_(st["gext"][split:], self._dp_group)          # upper layers + head + the loss (last element)
        lower()
        allreduce_flat_(st["gext"][:split], self._dp_group)
        main.wait_stream(side)

    def _launch_update(self, lib, g, st, s):
        """clip_grad_norm_(clip) + Adam on the flat buffers; the step counter is incremented on the device."""
        sq = st["scal"][1:2]
        _lib.check(lib.bigru_adam_tick(_lib.ptr(st["dstep"]), _lib.ptr(sq), s), "bigru_adam_tick")
        _lib.check(lib.bigru_sqnorm(_lib.ptr(st["grad"]), st["grad"].numel(), _lib.ptr(sq), s), "bigru_sqnorm")
        b1, b2 = g["betas"]
        _lib.check(lib.bigru_clip_adam_step_dev(_lib.ptr(self._flat), _lib.ptr(st["grad"]), _lib.ptr(st["m"]),
                                                _lib.ptr(st["v"]), self._flat.numel(), _lib.ptr(sq), float(self.clip),
                                                float(g["lr"]), float(b1), float(b2), float(g["eps"]), _lib.ptr(st["dstep"]),
                                                1.0, s), "bigru_clip_adam_step_dev")
        self._bump_step(st, 1)

    def _graph_for(self, key, x, tgt, kind, wv, pwv, denom, g):
        """CUDA graph(s) of the train step for one (shape, loss) key (SURVEY.md 8(f) N5): static input / output buffers, the
        C-ABI calls captured once.  One graph at world size 1; with data parallelism two (forward+loss+backward | update) with
        the gradient all-reduce issued between them."""
        ent = self._graphs.get(key)
        if ent is not None:
            return ent
        lib = _lib.load()
        dev = x.device
        plan = self._plan_for(x)
        st = self._fused_state(dev)
        B, C = x.shape[0], self.output_size               # x arrives padded to whole batch tiles; tgt has the real rows
        ent = {"x": torch.zeros_like(x), "tgt": torch.empty_like(tgt), "logits": torch.empty(B, C, device=dev, dtype=torch.float32),
               "dlogits": torch.zeros(B, C, device=dev, dtype=torch.float32), "stash": plan.acquire_stash(), "plan": plan}
        args = (float(self.dropout_p), int(bool(self.spatial_dropout)), 0, 0)
        ent["x"].copy_(x); ent["tgt"].copy_(tgt)
        # one eager pass on the static buffers first (first-use work such as shared-memory opt-ins happens outside the capture);
        # its parameter update is real: it is the step the caller asked for
        s = _stream_ptr(dev)
        split = self._dp_split(st)
        fwd_bwd = lambda part, s_: self._launch_fwd_loss_bwd(lib, plan, ent["x"], None, ent["tgt"], kind, wv, pwv, denom, ent["logits"],
                                                             ent["dlogits"], ent["stash"], args, st, s_, part)
        if split:
            fwd_bwd("upper", s)
            self._dp_allreduce_overlapped(st, split, dev, lambda: fwd_bwd("lower", s))
        else:
            fwd_bwd("all", s)
            if self._dp_world > 1:
                allreduce_flat_(st["gext"], self._dp_group)
        self._launch_update(lib, g, st, s)
        torch.cuda.current_stream(dev).synchronize()
        n0 = lib.bigru_launch_count()
        # an explicit capture stream ON THE MODEL'S DEVICE: torch's default capture stream is created once per process, on whichever
        # device was current then
        cap = torch.cuda.Stream(device=dev)
        ga = torch.cuda.CUDAGraph()
        with torch.cuda.graph(ga, stream=cap, capture_error_mode="thread_local"):
            s = _stream_ptr(dev)
            fwd_bwd("upper" if split else "all", s)
            if self._dp_world == 1:
                self._launch_update(lib, g, st, s)
        ga2 = None
        if split:                                         # the lowest layer's backward: replayed while the upper layers' gradients are reduced
            ga2 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(ga2, stream=cap, capture_error_mode="thread_local"):
                fwd_bwd("lower", _stream_ptr(dev))
        gb = None
        if self._dp_world > 1:
            gb = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gb, stream=cap, capture_error_mode="thread_local"):
                self._launch_update(lib, g, st, _stream_ptr(dev))
        self._bump_step(st, -1)                                   # the capture ran the host-side bookkeeping once without stepping
        ent["launches"] = int(lib.bigru_launch_count() - n0)
        lib.bigru_launch_count_add(-ent["launches"])      # captured, not executed
        ent["ga"], ent["ga2"], ent["gb"], ent["fresh"], ent["split"] = ga, ga2, gb, True, split
        if len(self._graphs) > 4:
            self._graphs.clear()
        self._graphs[key] = ent
        return ent

    def train_step(self, input_seq, target, hidden=None):
        """One optimisation step = the body of the reference loop (biGRU_model.py:198-210):
        zero_grad, forward, loss, backward, clip_grad_norm_(clip), Adam step - C-ABI calls with no autograd graph, replayed
        from a captured CUDA graph when the step is replayable (no dropout noise to draw, no initial state).
        Returns (loss, logits) as device tensors (no host sync)."""
        spec, g = self._loss_spec(), self._adam_spec()
        if spec is None or g is None:
            raise RuntimeError("train_step needs add_loss_fn(CrossEntropyLoss | BCEWithLogitsLoss | "
                               "MultiLabelSoftMarginLoss, mean reduction) and add_optimizer(torch.optim.Adam(model.parameters()))")
        lib = _lib.load()
        x, h0 = self._prepare_input(input_seq, hidden)
        dev = x.device
        kind, w, pw = spec
        B, C = x.shape[0], self.output_size
        if kind == _lib.LOSS_CE:
            tgt = target.to(device=dev, dtype=torch.int64, non_blocking=True).contiguous()
            if tgt.shape != (B,):
                raise ValueError(f"CrossEntropyLoss target must be [{B}] class indices")
            denom = float(B * self._dp_world)
        else:
            tgt = target.to(device=dev, dtype=torch.float32, non_blocking=True).contiguous()
            if tuple(tgt.shape) != (B, C):
                raise ValueError(f"target must be [{B}, {C}]")
            denom = float(B * C * self._dp_world)
        training = bool(self.training and self.dropout_p > 0)
        Bp = self._padded_batch(B)
        with torch.cuda.device(dev):
            wv, pwv = self._loss_vec(w, C), self._loss_vec(pw, C)
            st = self._fused_state(dev)
            x_real = x

            def padded(x, h0):                                # whole batch tiles on the tensor-core paths (see _padded_batch)
                if Bp == B:
                    return x, h0
                xp = x.new_zeros(Bp, x.shape[1], x.shape[2])
                xp[:B] = x
                if h0 is not None:
                    hp = h0.new_zeros(h0.shape[0], Bp, h0.shape[2])
                    hp[:, :B] = h0
                    h0 = hp
                return xp, h0
            h0 = self._pad_last(h0, self.plan_hidden(B))
            self._last_batch = B
            if self.use_cuda_graph and not training and h0 is None and not torch.cuda.is_current_stream_capturing():
                key = (B, int(x.shape[1]), self.precision, kind, id(wv), id(pwv), denom, float(g["lr"]), tuple(g["betas"]),
                       float(g["eps"]), float(self.clip), self._dp_world, dev.index)
                try:
                    ent = self._graphs.get(key)
                    if ent is None:
                        ent = self._graph_for(key, padded(x, None)[0], tgt, kind, wv, pwv, denom, g)
                except Exception as e:                        # capture is an optimisation: fall back to plain launches
                    import warnings
                    warnings.warn(f"BiGRU.train_step: CUDA-graph capture failed ({e}); using plain launches")
                    self.use_cuda_graph = False
                    ent = None
                if ent is not None:
                    if ent.pop("fresh", False):               # the warm-up pass inside _graph_for WAS this step
                        return st["loss"].clone(), ent["logits"][:B].clone()
                    ent["x"][:B].copy_(x_real, non_blocking=True)      # rows >= B of the static buffer stay zero
                    ent["tgt"].copy_(tgt, non_blocking=True)
                    ent["ga"].replay()
                    if ent["gb"] is not None:
                        if ent["ga2"] is not None:
                            self._dp_allreduce_overlapped(st, ent["split"], dev, ent["ga2"].replay)
                        else:
                            allreduce_flat_(st["gext"], self._dp_group)
                        ent["gb"].replay()
                    self._bump_step(st, 1)
                    lib.bigru_launch_count_add(ent["launches"])
                    return st["loss"].clone(), ent["logits"][:B].clone()
            x, h0 = padded(x, h0)
            plan = self._plan_for(x)
            logits = torch.empty(Bp, C, device=dev, dtype=torch.float32)
            dlogits = torch.zeros_like(logits) if Bp != B else torch.empty_like(logits)
            stash = plan.acquire_stash()
            seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if training else 0
            self._last_seed = seed
            s = _stream_ptr(dev)
            args = (float(self.dropout_p), int(bool(self.spatial_dropout)), int(training), seed)
            split = self._dp_split(st)
            if split:                                                # upper layers' gradients are reduced while layer 0 runs its backward
                self._launch_fwd_loss_bwd(lib, plan, x, h0, tgt, kind, wv, pwv, denom, logits, dlogits, stash, args, st, s, "upper")
                self._dp_allreduce_overlapped(st, split, dev, lambda: self._launch_fwd_loss_bwd(
                    lib, plan, x, h0, tgt, kind, wv, pwv, denom, logits, dlogits, stash, args, st, s, "lower"))
            else:
                self._launch_fwd_loss_bwd(lib, plan, x, h0, tgt, kind, wv, pwv, denom, logits, dlogits, stash, args, st, s)
                if self._dp_world > 1:
                    allreduce_flat_(st["gext"], self._dp_group)      # ONE all-reduce: shard gradients of the global-mean loss + the loss
            plan.release_stash(stash)
            self._launch_update(lib, g, st, s)
            return st["loss"].clone(), (logits[:B] if Bp != B else logits)

    # ------------------------------------------------------------------ zero-copy windows (SURVEY.md 8(f) N1)
    def _window_args(self, dataset, start, count):
        if dataset.device != self._flat.device:
            raise RuntimeError("dataset and model live on different devices")
        if dataset.n_features != self.n_features:
            raise ValueError(f"dataset has {dataset.n_features} features, the model expects {self.n_features}")
        if count <= 0 or start < 0 or start + count + dataset.window - 1 > dataset.n_rows:
            raise ValueError(f"windows [{start}, {start + count}) of width {dataset.window} exceed the {dataset.n_rows}-row chunk")

    def forward_windows(self, dataset, start: int, count: int):
        """Logits for windows start .. start+count-1 of a chunk-resident ``MySQLBatchLoader`` without materialising
        x[count, window, F]: the first kernel of the path reads (and normalises) the rows of the chunk directly."""
        if not self._is_flat():
            self._flatten()
        lib = _lib.load()
        self._window_args(dataset, start, count)
        if self._padded_batch(count) != count or self.plan_hidden(count) != self.hidden_size:      # padded shapes: collate on the device first
            self._win_ctx = None
            return self.forward(dataset.collate(start, count)[0])
        plan = self._plan_for(torch.empty(count, dataset.window, 0, device=self._flat.device))     # keyed by (B, T)
        logits = torch.empty(count, self.output_size, device=self._flat.device, dtype=torch.float32)
        stash = plan.acquire_stash()
        training = bool(self.training and self.dropout_p > 0)
        seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if training else 0
        with torch.cuda.device(self._flat.device):
            _lib.check(lib.bigru_forward_windows(plan.handle, _lib.ptr(self._flat), _lib.ptr(dataset.x_raw), _lib.ptr(dataset.x_min),
                                                 _lib.ptr(dataset.x_max), int(start), dataset.n_rows, float(self.dropout_p),
                                                 int(bool(self.spatial_dropout)), int(training), seed, _lib.ptr(stash),
                                                 _lib.ptr(plan.scratch), _lib.ptr(logits), None, _stream_ptr(self._flat.device)),
                       "bigru_forward_windows")
        self._win_ctx = (plan, stash, training, seed)
        return logits

    def train_step_windows(self, dataset, start: int, count: int):
        """``train_step`` on windows of a chunk-resident dataset (inputs and targets gathered on the device, the
        fp32 batch never exists).  Returns (loss, logits)."""
        spec, g = self._loss_spec(), self._adam_spec()
        if spec is None or g is None:
            raise RuntimeError("train_step_windows needs a fusable loss and torch.optim.Adam (see train_step)")
        lib = _lib.load()
        kind, w, pw = spec
        if self._padded_batch(count) != count or self.plan_hidden(count) != self.hidden_size:      # padded shapes: collate, then train_step
            self._window_args(dataset, start, count)
            x, y = dataset.collate(start, count)
            tgt = y.reshape(count, -1)[:, 0].to(torch.int64) if kind == _lib.LOSS_CE else y.reshape(count, self.output_size)
            return self.train_step(x, tgt)
        logits = self.forward_windows(dataset, start, count)
        plan, stash, training, seed = self._win_ctx
        dev, B, C = logits.device, count, self.output_size
        with torch.cuda.device(dev):
            y = torch.empty(count, 1, dataset.n_targets, device=dev, dtype=torch.float32)
            s = _stream_ptr(dev)
            _lib.check(lib.bigru_window_targets(_lib.ptr(dataset.y), int(start), dataset.n_rows, count, dataset.window,
                                                dataset.n_targets, _lib.ptr(y), s), "bigru_window_targets")
            if kind == _lib.LOSS_CE:
                tgt = y.reshape(count, -1)[:, 0].to(torch.int64).contiguous()
                denom = float(B * self._dp_world)
            else:
                tgt = y.reshape(count, C).contiguous()
                denom = float(B * C * self._dp_world)
            st = self._fused_state(dev)
            dlogits = torch.empty_like(logits)
            wv, pwv = self._loss_vec(w, C), self._loss_vec(pw, C)
            _lib.check(lib.bigru_loss(kind, _lib.ptr(logits), _lib.ptr(tgt), _lib.ptr(wv), _lib.ptr(pwv), B, C, denom,
                                      _lib.ptr(st["loss"]), _lib.ptr(dlogits), s), "bigru_loss")
            _lib.check(lib.bigru_backward(plan.handle, _lib.ptr(self._flat), None, None, float(self.dropout_p),
                                          int(bool(self.spatial_dropout)), int(training), seed, _lib.ptr(stash),
                                          _lib.ptr(plan.scratch), _lib.ptr(dlogits), _lib.ptr(st["grad"]), None, None, s),
                       "bigru_backward")
            plan.release_stash(stash)
            self._win_ctx = None
            if self._dp_world > 1:
                allreduce_flat_(st["gext"], self._dp_group)
            self._launch_update(lib, g, st, s)
            return st["loss"].clone(), logits

    def _generic_step(self, x, target):
        """Any loss / optimiser: autograd drives the same CUDA forward/backward kernels."""
        self.optimizer.zero_grad()
        pred = self.forward(x)
        if isinstance(self.loss_fn, nn.Module):
            self.loss_fn.to(pred.device)                 # class weights follow the logits
        loss = self.loss_fn(pred, target.to(pred.device))
        loss.backward()
        if self._dp_world > 1:                            # ONE all-reduce of all gradients (flattened), then scattered back
            ps = [p for p in self.parameters() if p.grad is not None]
            flat = torch.cat([p.grad.reshape(-1) for p in ps])
            allreduce_flat_(flat, self._dp_group)
            flat.div_(self._dp_world)
            off = 0
            for p in ps:
                p.grad.copy_(flat[off:off + p.grad.numel()].view_as(p.grad))
                off += p.grad.numel()
        nn.utils.clip_grad_norm_(self.parameters(), self.clip)
        self.optimizer.step()
        return loss.detach().reshape(1), pred.detach()

    # ------------------------------------------------------------------ epoch loops
    def _metric_counts(self, logits, target, counts_row):
        if target.dim() != 2 or target.shape != logits.shape:
            raise ValueError("multilabel metrics need a [batch, n_classes] indicator target "
                             "(biGRU_model.py:213-221 feeds sigmoid(pred) > 0.5 to sklearn)")
        tgt = target.to(device=logits.device, dtype=torch.float32).contiguous()
        with torch.cuda.device(logits.device):
            _lib.check(_lib.load().bigru_multilabel_counts(_lib.ptr(logits), _lib.ptr(tgt), logits.shape[0],
                                                           logits.shape[1], _lib.ptr(counts_row), _stream_ptr(logits.device)),
                       "bigru_multilabel_counts")

    @staticmethod
    def _scores(counts: np.ndarray, sizes, C, beta=0.5):
        """Per-batch accuracy / Hamming loss / F-beta from the device counters, then the mean over
        batches (the reference averages per-batch sklearn scores, :224 / :286)."""
        acc, ham, fb = [], [], []
        b2 = beta * beta
        for row, B in zip(counts, sizes):
            acc.append(row[0] / B)
            ham.append(row[1] / (B * C))
            tp, fp, fn = row[2::3][:C], row[3::3][:C], row[4::3][:C]
            den = (1 + b2) * tp + b2 * fn + fp
            fb.append(np.where(den > 0, (1 + b2) * tp / np.maximum(den, 1), 0.0))
        return float(np.mean(acc)), float(np.mean(ham)), np.mean(np.stack(fb), axis=0)

    def train_model(self, train_iterator):
        """One training epoch (biGRU_model.py:162-224).  Returns
        (mean accuracy, mean Hamming loss, mean loss, mean F-beta(0.5) per class)."""
        self.train()
        fused = self.can_fuse_step()
        losses, sizes, rows = [], [], []
        C = self.output_size
        for input_seq, target in train_iterator:
            target = target.squeeze(1)                                   # [B,1,C] -> [B,C]  (:193)
            if fused:
                loss, logits = self.train_step(input_seq, target)
            else:
                x, _ = self._prepare_input(input_seq, None)
                loss, logits = self._generic_step(x, target)
            row = torch.zeros(2 + 3 * C, dtype=torch.int64, device=logits.device)
            self._metric_counts(logits, target, row)
            losses.append(loss.reshape(1))
            rows.append(row)
            sizes.append(logits.shape[0])
        if not rows:
            return float("nan"), float("nan"), float("nan"), np.full(C, np.nan)
        counts = torch.stack(rows).cpu().numpy().astype(np.float64)      # one host sync per epoch
        acc, ham, fb = self._scores(counts, sizes, C)
        return acc, ham, float(torch.cat(losses).float().mean().item()), fb

    def evaluate_model(self, eval_iterator):
        """One evaluation epoch (biGRU_model.py:227-286).  Returns (mean accuracy, mean Hamming loss,
        mean F-beta(0.5) per class, pred_total LongTensor, target_total LongTensor)."""
        self.eval()
        C = self.output_size
        rows, sizes, preds, targets = [], [], [], []
        with torch.no_grad():
            for input_seq, target in eval_iterator:
                target = target.squeeze(1)
                logits = self.forward(input_seq)
                row = torch.zeros(2 + 3 * C, dtype=torch.int64, device=logits.device)
                self._metric_counts(logits, target, row)
                rows.append(row)
                sizes.append(logits.shape[0])
                preds.append(logits > 0)                                  # sigmoid(x) > 0.5
                targets.append(target)
        if not rows:
            return float("nan"), float("nan"), np.full(C, np.nan), torch.LongTensor(), torch.LongTensor()
        counts = torch.stack(rows).cpu().numpy().astype(np.float64)
        acc, ham, fb = self._scores(counts, sizes, C)
        pred_total = torch.cat(preds).cpu().type(torch.LongTensor)
        target_total = torch.cat([t.cpu() for t in targets]).type(torch.LongTensor)
        return acc, ham, fb, pred_total, target_total
