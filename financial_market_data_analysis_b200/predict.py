"""The model side of the reference's live predictor (``predict.py``) on the B200 path (SURVEY.md 8(f) N5).

``predict.py`` builds ``BiGRU(hidden_size=8, n_features, output_size=4, n_layers=1, clip=50, dropout=0.2,
spatial_dropout=False, bidirectional=True)`` (``:73-88``), loads ``model_params.pt`` (``:104``) and the pickled
``norm_params`` (``:110-122``), and for every Kafka message fetches one window of ``window=5`` rows, normalises it
``(x - min) / (max - min)`` (``:170``), runs ``model.forward`` in eval mode (``:178``), applies a sigmoid (``:181``) and
reports the labels above ``prob_threshold`` (``:186-193``).  The Kafka consumer / producer and the MySQL cursor stay the
reference's own; :class:`LivePredictor` is the part between "rows fetched" and "dict to send".  Small models (the
shipped checkpoint) run in **one kernel launch** (``bigru_infer_window``: normalisation + GRU + pooling head + Linear +
sigmoid, one CTA per window); full-size models (long windows, hidden sizes up to 512) run on ``bigru_infer_cluster``
(one SGEMM and one cluster-resident scan per layer, then the head).  There is no CPU fallback."""
from __future__ import annotations

import pickle

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .biGRU_model import BiGRU

Y_FIELDS = "up1, up2, down1, down2".split(", ")        # predict.py:33

# bigru_infer_window (one CTA per window, one launch) is used where it accepts the shape and hidden_size <=
# SINGLE_CTA_MAX_HIDDEN; otherwise bigru_infer_cluster (2L+1 launches).  The bound keeps the shipped (H 8) and notebook
# (H 32) models on one launch.  The crossover is not measured yet: tools/bench_live_predictor.py measures it (DESIGN §5.7b).
SINGLE_CTA_MAX_HIDDEN = 32


def checkpoint_shape(state):
    """(hidden_size, n_layers) of a BiGRU state dict: the columns of ``gru.weight_hh_l0`` and the number of
    ``gru.weight_ih_l{k}`` keys."""
    hidden = int(state["gru.weight_hh_l0"].shape[1])
    layers = sum(1 for k in state if k.startswith("gru.weight_ih_l") and not k.endswith("_reverse"))
    return hidden, layers


class LivePredictor:
    def __init__(self, model_params="model_params.pt", norm_params="norm_params", n_features=None, y_fields=Y_FIELDS,
                 window=5, hidden_size=None, n_layers=None, clip=50, dropout=0.2, learning_rate=0.001, spatial_dropout=False,
                 prob_threshold=0.5, device="cuda"):
        """``model_params``: path to the checkpoint or a state_dict; ``norm_params``: path to the pickle written by
        ``MySQLChunkLoader`` (``sql_pytorch_dataloader.py:146-153``), the dict itself (name -> {"MIN", "MAX"}), a
        ``(min, max)`` pair of arrays, or ``None`` for already normalised windows.  ``hidden_size`` / ``n_layers`` default to
        the checkpoint's own shape (the shipped one: 8 and 1); other defaults as ``predict.py:73-83``."""
        self.window, self.prob_threshold, self.y_fields = int(window), float(prob_threshold), list(y_fields)
        if isinstance(norm_params, str):
            with open(norm_params, "rb") as fh:
                norm_params = pickle.load(fh)
        if isinstance(norm_params, dict):                                  # predict.py:113-122
            x_min = [norm_params[k]["MIN"] for k in norm_params.keys()]
            x_max = [norm_params[k]["MAX"] for k in norm_params.keys()]
        elif norm_params is not None:
            x_min, x_max = norm_params
        else:
            x_min = x_max = None
        state = torch.load(model_params, map_location="cpu") if isinstance(model_params, str) else model_params
        if n_features is None:
            n_features = int(state["gru.weight_ih_l0"].shape[1])
        self.n_features = int(n_features)
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("LivePredictor runs on the GPU only (no CPU fallback)")
        if hidden_size is None or n_layers is None:
            ck_hidden, ck_layers = checkpoint_shape(state)
            hidden_size = ck_hidden if hidden_size is None else int(hidden_size)
            n_layers = ck_layers if n_layers is None else int(n_layers)
        model = BiGRU(hidden_size, self.n_features, len(self.y_fields), n_layers, clip, dropout, spatial_dropout, bidirectional=True,
                      precision="fp32")
        model.to(dev)                                                      # predict.py:90-91
        model.add_loss_fn(nn.MultiLabelSoftMarginLoss())                   # predict.py:94
        model.add_optimizer(torch.optim.Adam(model.parameters(), lr=learning_rate))
        model.add_device(dev)
        model.load_state_dict({k: torch.as_tensor(v) for k, v in state.items()})
        model.eval()                                                       # predict.py:107
        self.model, self.device = model, dev
        self.x_min = None if x_min is None else torch.as_tensor(np.asarray(x_min, dtype=np.float32), device=dev)
        self.x_max = None if x_max is None else torch.as_tensor(np.asarray(x_max, dtype=np.float32), device=dev)
        if self.x_min is not None and self.x_min.numel() != self.n_features:
            raise ValueError(f"norm_params hold {self.x_min.numel()} features, the model expects {self.n_features}")
        C = len(self.y_fields)
        self._x = torch.empty((1, self.window, self.n_features), dtype=torch.float32, device=dev)
        self._logits = torch.empty((1, C), dtype=torch.float32, device=dev)
        self._probs = torch.empty((1, C), dtype=torch.float32, device=dev)
        self._host = torch.empty((2, C), dtype=torch.float32).pin_memory()
        self._work = torch.empty(0, dtype=torch.float32, device=dev)     # bigru_infer_cluster workspace, grown as needed

    def forward_windows(self, windows):
        """Raw (un-normalised) windows [B, window, n_features] -> (logits, probabilities) on the device."""
        m = self.model
        x = torch.as_tensor(windows, dtype=torch.float32).to(self.device, non_blocking=True).contiguous()
        if x.dim() == 2:
            x = x.unsqueeze(0)                                             # predict.py:167
        if x.dim() != 3 or x.shape[2] != self.n_features:
            raise ValueError(f"expected [batch, window, {self.n_features}] rows, got {tuple(x.shape)}")
        B, T = int(x.shape[0]), int(x.shape[1])
        logits = self._logits if B == 1 else torch.empty((B, len(self.y_fields)), dtype=torch.float32, device=self.device)
        probs = self._probs if B == 1 else torch.empty_like(logits)
        lib = _lib.load()
        H, L, C, bi = m.hidden_size, m.n_layers, m.output_size, 1 if m.bidirectional else 0
        xmin, xmax = _lib.ptr(self.x_min), _lib.ptr(self.x_max)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            params = m.flat_parameters()
            rc = _lib.ERR_UNSUPPORTED
            if H <= SINGLE_CTA_MAX_HIDDEN:
                rc = lib.bigru_infer_window(_lib.ptr(params), _lib.ptr(x), xmin, xmax, B, T, self.n_features, H, L, C, bi,
                                            _lib.ptr(logits), _lib.ptr(probs), stream)
                if rc != _lib.ERR_UNSUPPORTED:
                    _lib.check(rc, "bigru_infer_window")
            if rc == _lib.ERR_UNSUPPORTED:
                nbytes = _lib.C.c_size_t()
                _lib.check(lib.bigru_infer_cluster_workspace_bytes(B, T, self.n_features, H, L, bi, _lib.C.byref(nbytes)),
                           "bigru_infer_cluster_workspace_bytes")
                if self._work.numel() * 4 < nbytes.value:
                    self._work = torch.empty((nbytes.value + 3) // 4, dtype=torch.float32, device=self.device)
                rc = lib.bigru_infer_cluster(_lib.ptr(params), _lib.ptr(x), xmin, xmax, B, T, self.n_features, H, L, C, bi,
                                             _lib.ptr(self._work), _lib.ptr(logits), _lib.ptr(probs), stream)
                if rc != _lib.ERR_UNSUPPORTED:
                    _lib.check(rc, "bigru_infer_cluster")
            if rc == _lib.ERR_UNSUPPORTED:
                # neither live kernel takes the shape: the model's own fp32 forward (eval mode, no dropout)
                xn = x if self.x_min is None else (x - self.x_min) / (self.x_max - self.x_min)
                with torch.no_grad():
                    logits.copy_(m(xn))
                torch.sigmoid(logits, out=probs)
        return logits, probs

    def predict(self, input_data, timestamp_str=None):
        """``input_data``: the rows of one window as fetched at ``predict.py:159-163`` ([window, n_features]).  Returns the
        dict the reference sends to its 'predict' topic (``predict.py:195-196``)."""
        logits, probs = self.forward_windows(input_data)
        self._host[0].copy_(probs[0], non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        pred = self._host[0].clone()                                        # pred.squeeze(0), predict.py:183
        pred_idx = np.where(pred.numpy() > self.prob_threshold)[0]          # predict.py:186
        pred_labels = [self.y_fields[i] for i in pred_idx]
        return {"timestamp": timestamp_str, "probabilities": pred, "prob_threshold": self.prob_threshold,
                "pred_indices": pred_idx, "pred_labels": pred_labels}
