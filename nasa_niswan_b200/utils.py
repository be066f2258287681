"""Checkpoint and validation helpers with the reference's contracts (utils.py:23-75), SURVEY.md section 8f rank 4.

`save_checkpoint` / `load_checkpoint` keep the reference's file format -- a dict with `model_state_dict`,
`optimizer_state_dict`, `learning_rate`, `epoch` -- so checkpoints move freely between the reference ConvLSTM and
this one (same `state_dict` keys and shapes) and between `torch.optim.Adam` and `NativeAdam` (same optimizer
`state_dict` layout).  `val_loop` is utils.py:52-75 without its per-batch device-to-host copies: R^2 is reduced on
the GPU by the fused loss kernel and read back once per batch as five floats."""
import ctypes
from typing import Optional, Tuple

import torch

from . import _lib
from .preprocess import fuse_inputs_adjoint


def save_checkpoint(model, optimizer, filename, learning_rate=None, epoch=None):
    """utils.py:23-32"""
    checkpoint = {
        "model_state_dict": model.state_dict(),
        "optimizer_state_dict": optimizer.state_dict(),
        "learning_rate": learning_rate,
        "epoch": epoch,
    }
    torch.save(checkpoint, filename)


def load_checkpoint(checkpoint_file, model, optimizer=None, lr=None, map_location=None):
    """utils.py:34-50 (the learning-rate override rules included)"""
    checkpoint = torch.load(checkpoint_file, map_location=map_location, weights_only=False)
    model.load_state_dict(checkpoint["model_state_dict"])
    if optimizer is not None:
        optimizer.load_state_dict(checkpoint["optimizer_state_dict"])
        if lr is not None:
            for param_group in optimizer.param_groups:
                param_group["lr"] = lr
        elif checkpoint["learning_rate"] is not None:
            for param_group in optimizer.param_groups:
                param_group["lr"] = checkpoint["learning_rate"]
    return checkpoint


def r2_from_stats(stats: torch.Tensor, n: int) -> float:
    """sklearn.metrics.r2_score(y.flatten(), pred.flatten()) (train.py:114, utils.py:73) from the sums the fused loss
    kernel leaves in its scratch: stats = {sum (p-y)^2, sum |p-y|, sum y, sum y^2, -}."""
    s = stats[:4].double().cpu()
    ss_res, sy, syy = float(s[0]), float(s[2]), float(s[3])
    ss_tot = syy - sy * sy / n
    return 1.0 - ss_res / ss_tot if ss_tot > 0 else float("nan")


def r2_score_device(pred: torch.Tensor, y: torch.Tensor, crop: Optional[Tuple[int, int, int, int]] = None) -> float:
    """R^2 of pred[:, 0, y0:y1, x0:x1] against y on the GPU (one kernel, 20 bytes read back)."""
    if not pred.is_cuda:
        raise RuntimeError("r2_score_device needs CUDA tensors (no CPU fallback)")
    B, _, H, W = pred.shape
    y0, y1, x0, x1 = crop if crop is not None else (0, H, 0, W)
    stats = torch.zeros(8, dtype=torch.float32, device=pred.device)
    loss = torch.empty(1, dtype=torch.float32, device=pred.device)
    vp = _lib.ptr
    with _lib.on_device(pred.device):
        _lib.check(_lib.load().nint_loss_mse_l1(vp(pred.detach().contiguous().float()), vp(y.contiguous().float()), B, H, W,
                                                y0, y1, x0, x1, None, vp(loss), vp(stats), _lib.stream_ptr(pred.device)),
                   "nint_loss_mse_l1")
    return r2_from_stats(stats, B * (y1 - y0) * (x1 - x0))


_CROPS = {"LSTM": (5, 95, 5, 149), "PIX2PIX": (83, 173, 56, 200), "UNet": (83, 173, 56, 200)}   # utils.py:67-71


def val_loop(args, dataloader, model, crop="auto") -> float:
    """utils.py:52-75, same signature and call (`val_loop(args, val_dataloader, generator)`, train.py:122): mean over
    batches of R^2 on the cropped prediction, with the crop chosen by the `args.model` prefix like the reference.
    `args` may be None (or anything without `.model`): the LSTM crop is used.  `crop=None` disables cropping, a
    4-tuple (y0, y1, x0, x1) overrides it.  R^2 is reduced on the GPU; only five floats per batch cross to the host."""
    if crop == "auto":
        kind = str(getattr(args, "model", "LSTM")).split("-")[0]
        crop = _CROPS.get(kind, _CROPS["LSTM"])
    model.eval()
    r2, n = 0.0, 0
    device = next(model.parameters()).device
    with torch.no_grad():
        for X, y in dataloader:
            X, y = X.to(device, non_blocking=True), y.to(device, non_blocking=True)
            out = model(X)
            pred = out[0] if isinstance(out, tuple) else out
            r2 += r2_score_device(pred, y, crop)
            n += 1
    return r2 / max(n, 1)


def seed(seed=0):
    """utils.py:77-88: seeds python / numpy / torch and asks for deterministic kernels.  Here `cudnn.deterministic`
    also selects the fixed-order gradient reductions of the ConvLSTM kernels (model._deterministic_default)."""
    import random
    import numpy as np
    random.seed(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)
    if torch.cuda.is_available():
        torch.cuda.manual_seed(seed)
        torch.cuda.manual_seed_all(seed)
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.benchmark = False


def sensitivity_sweep(dataloader, model, num_features: int, perturbation: float = 0.05,
                      crop: Optional[Tuple[int, int, int, int]] = (5, 95, 5, 149), y_mean: float = 0.0,
                      y_std: float = 1.0) -> torch.Tensor:
    """One-at-a-time input sensitivity (test.ipynb:2430-2462): for every feature i, predictions with channel i of the
    whole window scaled by (1 + perturbation), cropped and de-normalised -> [num_features, N, Hc, Wc] on the host.

    The notebook walks the dataloader once per feature and uploads every batch again each time; here a batch is
    uploaded once, the perturbation is applied and undone on the device, and only the cropped predictions come back."""
    model.eval()
    chunks = [[] for _ in range(num_features)]
    with torch.no_grad():
        for X, _ in dataloader:
            X = X.to(next(model.parameters()).device, non_blocking=True)
            for i in range(num_features):
                saved = X[:, :, i].clone()
                X[:, :, i] *= (1 + perturbation)
                out = model(X)
                pred = out[0] if isinstance(out, tuple) else out
                if crop is not None:
                    pred = pred[:, :, crop[0]:crop[1], crop[2]:crop[3]]
                chunks[i].append((pred[:, 0] * y_std + y_mean).cpu())
                X[:, :, i] = saved
    return torch.stack([torch.cat(c, dim=0) for c in chunks], dim=0)


def input_sensitivity(model, bank, win_start, seq_len: int,
                      crop: Optional[Tuple[int, int, int, int]] = (5, 95, 5, 149), y_std: float = 1.0):
    """The gradient counterpart of `sensitivity_sweep`: d(sum of the de-normalised, cropped predictions of the windows
    `win_start`) / d(inputs) in one forward and one backward, at every pixel, channel and lag instead of one +5 %
    perturbation per feature.  Returns `bank.field_grads()` for banks built by `FrameBank.from_fields` (gradients w.r.t.
    the raw levels, emission and static fields), else dL/d(frames) [N, C, Hp, Wp].  The bank's own gradient state is
    left as it was, and no parameter gets a .grad."""
    saved = bank.grad, bank._anchor
    bank.grad = bank._anchor = None
    try:
        bank.requires_grad_()
        with torch.enable_grad():
            out = model.forward_windows(bank, win_start, seq_len)
            pred = out[0] if isinstance(out, tuple) else out
            if crop is not None:
                pred = pred[:, :, crop[0]:crop[1], crop[2]:crop[3]]
            torch.autograd.grad(pred.sum() * y_std, bank._anchor, allow_unused=True)
        return bank.field_grads() if bank._fields is not None else bank.grad
    finally:
        bank.grad, bank._anchor = saved


def tangent_sweep(dataloader, model, num_features: int, perturbation: float = 0.05,
                  crop: Optional[Tuple[int, int, int, int]] = (5, 95, 5, 149), y_std: float = 1.0) -> torch.Tensor:
    """The linearised counterpart of `sensitivity_sweep`: for every feature i, the change of the cropped, de-normalised
    prediction when channel i of the whole window is scaled by (1 + perturbation), taken from the tangent-linear model
    (ConvLSTM.jvp) in the direction v = perturbation * x restricted to channel i -> [num_features, N, Hc, Wc] on the
    host.  `sensitivity_sweep` returns the perturbed predictions; this returns their first-order difference from the
    unperturbed one, without the rounding of two nonlinear runs.  One forward per batch, then one tangent pass per
    feature on the same forward."""
    model.eval()
    chunks = [[] for _ in range(num_features)]
    device = next(model.parameters()).device
    with torch.no_grad():
        for X, _ in dataloader:
            X = X.to(device, non_blocking=True)
            plan = model.plan_for(X, True, tangent=True)
            plan.forward(X)
            dx = torch.zeros_like(X, dtype=torch.float32)
            for i in range(num_features):
                dx[:, :, i] = X[:, :, i] * perturbation
                dpred = plan.forward_tangent(dx)[0]
                dx[:, :, i] = 0
                if crop is not None:
                    dpred = dpred[:, :, crop[0]:crop[1], crop[2]:crop[3]]
                chunks[i].append((dpred[:, 0] * y_std).cpu())
    return torch.stack([torch.cat(c, dim=0) for c in chunks], dim=0)


def emission_response(model, bank, win_start, seq_len: int, d_emis2d: torch.Tensor,
                      crop: Optional[Tuple[int, int, int, int]] = (5, 95, 5, 149), y_std: float = 1.0) -> torch.Tensor:
    """The source-oriented question the adjoint cannot answer in one pass: how the de-normalised, cropped prediction of
    every window `win_start` changes, to first order, when the raw emission field of a bank built by
    `FrameBank.from_fields` changes by d_emis2d [N, H, W] (e.g. +10 % over a region and a few days) -> [B, Hc, Wc].  One
    forward and one tangent pass over the windows (FrameBank.tangent_from_fields, then ConvLSTM.jvp_windows)."""
    _, dout = model.jvp_windows(bank, win_start, seq_len, bank.tangent_from_fields(d_emis2d=d_emis2d))
    dpred = dout[0] if isinstance(dout, tuple) else dout
    if crop is not None:
        dpred = dpred[:, :, crop[0]:crop[1], crop[2]:crop[3]]
    return dpred[:, 0] * y_std


def emission_hvp(model, bank, win_start, seq_len: int, d_emis2d: torch.Tensor, loss_fn):
    """The Hessian-vector product of loss_fn(model.forward_windows(bank, win_start, seq_len)) w.r.t. the raw fields of
    a bank built by `FrameBank.from_fields`, in the direction of an emission perturbation d_emis2d [N, H, W]: the
    curvature a Newton-CG or truncated-Newton emission inversion needs.  The fusion is affine in the fields, so H v in
    field space is its adjoint applied to the frame-space H of its tangent: FrameBank.tangent_from_fields, then
    ConvLSTM.hvp_windows, then the preprocessing adjoint (nint_fuse_inputs_adjoint) of the HVP frames.  Returns the dict
    of `field_grads()` ({"levels3d", "emis2d", "statics"}) holding H v."""
    if bank._fields is None:
        raise RuntimeError("emission_hvp needs a bank built by FrameBank.from_fields")
    _, _, (hv, _) = model.hvp_windows(bank, win_start, seq_len, bank.tangent_from_fields(d_emis2d=d_emis2d), loss_fn)
    return fuse_inputs_adjoint(hv, **bank._fields)
