"""CPU oracle for the Smart-NINT ConvLSTM hot path.  TEST INFRASTRUCTURE ONLY.

This file is a from-scratch restatement (plain torch fp32 on the CPU + numpy) of
the arithmetic of the reference's ``model.py`` hot path.  It is imported only by
``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl
reference`` legs of ``bench.py``; the product package never imports it and has
no CPU fallback.

Parity status: PINNED.  ``oracle/make_golden.py`` imports the unmodified
reference ``model.py`` from an upstream checkout, runs it on seeded inputs and
writes ``tests/golden/*.npz`` (``oracle/golden.py``); ``tests/test_oracle.py`` checks every
function here against those vectors and against the structural known answers
the reference's notebooks print (param counts ``test.ipynb:4698-4699``, padding
print ``dataset_config.ipynb:484-496``).  The arithmetic itself lives in a
third-party dependency of the reference (PyTorch ``nn.Conv2d``; unpinned in the
reference, ``README.md:23``); golden vectors were produced with torch
2.11.0+cu128 on CPU.

Reference citations are ``file:line`` into the upstream repo.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F

Tensor = torch.Tensor


# --------------------------------------------------------------------------
# parameters
# --------------------------------------------------------------------------
def param_shapes(input_channels: int, hidden_channels: Sequence[int],
                 kernel_size: Sequence[int]) -> Dict[str, Tuple[int, ...]]:
    """state_dict names/shapes of the reference ``ConvLSTM`` (model.py:235-251;
    checkpoint contract utils.py:27,39)."""
    assert len(hidden_channels) == len(kernel_size)
    shapes: Dict[str, Tuple[int, ...]] = {}
    cin = input_channels
    for l, (hc, k) in enumerate(zip(hidden_channels, kernel_size)):
        shapes[f"layers.{l}.conv.weight"] = (4 * hc, cin + hc, k, k)   # model.py:207-211
        shapes[f"layers.{l}.conv.bias"] = (4 * hc,)
        cin = hc                                                       # model.py:248
    shapes["conv.weight"] = (1, hidden_channels[-1], 1, 1)             # model.py:251
    shapes["conv.bias"] = (1,)
    return shapes


def init_params(input_channels: int, hidden_channels: Sequence[int],
                kernel_size: Sequence[int], seed: int = 0) -> Dict[str, Tensor]:
    """PyTorch-default Conv2d init restated: weight and bias ~ U(+-1/sqrt(fan_in))
    (kaiming_uniform(a=sqrt(5)) reduces to that bound).  Values differ from the
    reference's RNG stream; parity tests always copy weights, never re-draw."""
    g = torch.Generator().manual_seed(seed)
    out: Dict[str, Tensor] = {}
    for name, shape in param_shapes(input_channels, hidden_channels, kernel_size).items():
        if name.endswith("weight"):
            fan_in = shape[1] * shape[2] * shape[3]
            last_bound = 1.0 / fan_in ** 0.5
        out[name] = (torch.rand(shape, generator=g) * 2 - 1) * last_bound
    return out


# --------------------------------------------------------------------------
# forward
# --------------------------------------------------------------------------
def cell_forward(x: Tensor, h: Tensor, c: Tensor, weight: Tensor,
                 bias: Optional[Tensor]) -> Tuple[Tensor, Tensor]:
    """One recurrent step (model.py:216-231).

    ``combined = cat([x, h], 1)`` (x first), zero-padded k x k conv with
    ``padding = k // 2`` (model.py:204-211), split in four ``hidden`` blocks
    ordered i, f, g, o (model.py:221), sigma/sigma/tanh/sigma (model.py:223-226),
    ``c' = c*f + i*g`` (model.py:228), ``h' = o*tanh(c')`` (model.py:229)."""
    k = weight.shape[-1]
    gates = F.conv2d(torch.cat([x, h], dim=1), weight, bias, padding=k // 2)
    i, f, g, o = torch.split(gates, h.shape[1], dim=1)
    i, f, g, o = torch.sigmoid(i), torch.sigmoid(f), torch.tanh(g), torch.sigmoid(o)
    c_new = c * f + i * g
    h_new = o * torch.tanh(c_new)
    return h_new, c_new


def convlstm_forward(x: Tensor, params: Dict[str, Tensor], num_layers: int,
                     return_sequence: bool = False):
    """``ConvLSTM.forward`` (model.py:253-274): zero (h, c) per layer, loop t then
    layers, 1x1 head on the last layer's h at the last t -> [B,1,H,W].
    ``return_sequence`` restates the commented-out variant (model.py:264,272,274)
    that also returns the head applied at every t -> [B,T,H,W]."""
    B, T, _, H, W = x.shape
    hs: List[Tensor] = []
    cs: List[Tensor] = []
    for l in range(num_layers):
        hc = params[f"layers.{l}.conv.bias"].shape[0] // 4
        hs.append(torch.zeros(B, hc, H, W, dtype=x.dtype))       # model.py:260-261
        cs.append(torch.zeros(B, hc, H, W, dtype=x.dtype))
    outs = []
    h = None
    for t in range(T):                                           # model.py:265
        inp = x[:, t]
        for l in range(num_layers):                              # model.py:267
            h, c = cell_forward(inp, hs[l], cs[l], params[f"layers.{l}.conv.weight"],
                                params[f"layers.{l}.conv.bias"])
            hs[l], cs[l] = h, c
            inp = h                                              # model.py:271
        if return_sequence:
            outs.append(F.conv2d(h, params["conv.weight"], params["conv.bias"]))
    pred = F.conv2d(h, params["conv.weight"], params["conv.bias"])   # model.py:274
    if return_sequence:
        return pred, torch.cat(outs, dim=1)
    return pred


def training_loss(pred: Tensor, y: Tensor, crop: Optional[Tuple[int, int, int, int]] = None) -> Tensor:
    """``MSELoss(y,pred) + L1Loss(y,pred)`` on the (optionally cropped) squeezed
    prediction (train.py:74-75,102,105).  ``crop = (y0, y1, x0, x1)``."""
    if crop is not None:
        y0, y1, x0, x1 = crop
        pred = pred[:, :, y0:y1, x0:x1]
    p = pred.squeeze(1)
    return F.mse_loss(p, y) + F.l1_loss(p, y)


def forward_backward(x: Tensor, y: Tensor, params: Dict[str, Tensor], num_layers: int,
                     crop=None) -> Tuple[Tensor, Tensor, Dict[str, Tensor]]:
    """fwd + loss + autograd backward (train.py:96-109).  Returns (pred, loss, grads)."""
    leaf = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
    pred = convlstm_forward(x, leaf, num_layers)
    loss = training_loss(pred, y, crop)
    loss.backward()
    return pred.detach(), loss.detach(), {k: v.grad.detach() for k, v in leaf.items()}


# --------------------------------------------------------------------------
# explicit BPTT (what the CUDA backward kernels implement; checked against
# autograd in tests/test_oracle.py)
# --------------------------------------------------------------------------
def manual_backward(x: Tensor, params: Dict[str, Tensor], num_layers: int,
                    dpred: Tensor) -> Dict[str, Tensor]:
    """Hand-derived backward of ``convlstm_forward`` for an upstream gradient
    ``dpred`` [B,1,H,W] (SURVEY.md section 8 a10): per step in reverse t,
    ``tc=tanh(c_t)``, ``do=dh*tc``, ``dc=dc_next+dh*o*(1-tc^2)``, ``di=dc*g``,
    ``dg=dc*i``, ``df=dc*c_{t-1}``, ``dc_{t-1}=dc*f``; pre-activation grads
    ``di*i(1-i)``, ``df*f(1-f)``, ``dg*(1-g^2)``, ``do*o(1-o)``; wgrad / dgrad of
    the gate conv.  No autograd is used."""
    B, T, _, H, W = x.shape
    L = num_layers
    Wt = [params[f"layers.{l}.conv.weight"] for l in range(L)]
    bs = [params[f"layers.{l}.conv.bias"] for l in range(L)]
    hc = [b.shape[0] // 4 for b in bs]
    # ---- forward, saving what backward needs
    hs = [[torch.zeros(B, hc[l], H, W)] for l in range(L)]     # hs[l][t] = h_{t-1}
    cs = [[torch.zeros(B, hc[l], H, W)] for l in range(L)]
    gates = [[None] * T for _ in range(L)]
    for t in range(T):
        inp = x[:, t]
        for l in range(L):
            k = Wt[l].shape[-1]
            pre = F.conv2d(torch.cat([inp, hs[l][t]], 1), Wt[l], bs[l], padding=k // 2)
            i, f, g, o = torch.split(pre, hc[l], 1)
            i, f, g, o = torch.sigmoid(i), torch.sigmoid(f), torch.tanh(g), torch.sigmoid(o)
            c = cs[l][t] * f + i * g
            h = o * torch.tanh(c)
            gates[l][t] = (i, f, g, o)
            hs[l].append(h)
            cs[l].append(c)
            inp = h
    # ---- backward
    grads = {k: torch.zeros_like(v) for k, v in params.items()}
    h_last = hs[L - 1][T]
    grads["conv.weight"] = (dpred * h_last).sum(dim=(0, 2, 3)).reshape(1, -1, 1, 1)
    grads["conv.bias"] = dpred.sum().reshape(1)
    dh_next = [torch.zeros(B, hc[l], H, W) for l in range(L)]   # from own dgrad at t+1
    dc_next = [torch.zeros(B, hc[l], H, W) for l in range(L)]
    for t in reversed(range(T)):
        dx_from_above = None
        for l in reversed(range(L)):
            dh = dh_next[l].clone()
            if l == L - 1 and t == T - 1:
                dh = dh + dpred * params["conv.weight"].reshape(1, -1, 1, 1)
            if dx_from_above is not None:
                dh = dh + dx_from_above
            i, f, g, o = gates[l][t]
            tc = torch.tanh(cs[l][t + 1])
            do = dh * tc
            dc = dc_next[l] + dh * o * (1 - tc * tc)
            di, dg, df = dc * g, dc * i, dc * cs[l][t]
            dc_next[l] = dc * f
            dpre = torch.cat([di * i * (1 - i), df * f * (1 - f), dg * (1 - g * g), do * o * (1 - o)], 1)
            inp = x[:, t] if l == 0 else hs[l - 1][t + 1]
            comb = torch.cat([inp, hs[l][t]], 1)
            k = Wt[l].shape[-1]
            p = k // 2
            # wgrad: dW[n,c,dy,dx] = sum_{b,y,x} dpre[b,n,y,x] * comb[b,c,y+dy-p,x+dx-p]
            cp = F.pad(comb, (p, p, p, p))
            for dy in range(k):
                for dx in range(k):
                    win = cp[:, :, dy:dy + H, dx:dx + W]
                    grads[f"layers.{l}.conv.weight"][:, :, dy, dx] += torch.einsum("bnyx,bcyx->nc", dpre, win)
            grads[f"layers.{l}.conv.bias"] += dpre.sum(dim=(0, 2, 3))
            # dgrad: dcomb = dpre (*) flip(W)   (transposed conv, same zero padding)
            dcomb = F.conv_transpose2d(dpre, Wt[l], padding=p)
            cin = inp.shape[1]
            dx_from_above = dcomb[:, :cin] if l > 0 else None
            dh_next[l] = dcomb[:, cin:]
    return grads


# --------------------------------------------------------------------------
# host-side preprocessing restated (north-star item 4 / SURVEY 5.9)
# --------------------------------------------------------------------------
def cyclic_pad_lon(data: np.ndarray, target_w: int) -> np.ndarray:
    """Cyclic longitude halo on the last axis (dataset.py:22-36, dataset.py:67-80)."""
    W = data.shape[-1]
    left = (target_w - W) // 2
    right = target_w - W - left
    if left > W or right > W:
        raise AttributeError("The requested padding size is larger than width size of the input image.")
    lhs = data[..., W - left:] if left > 0 else data[..., :0]
    return np.concatenate([lhs, data, data[..., :right]], axis=-1)


def reflect_pad_lat(data: np.ndarray, target_h: int, mode: str = "reflect") -> np.ndarray:
    """Latitude halo on axis -2.

    ``mode='reflect'``: true reflect without edge repeat, what the 3-D variant
    computes (dataset.py:38-53; equals ``np.pad(mode='reflect')``).
    ``mode='reference_rnn'``: bug-compatible with the 4-D variant
    (dataset.py:82-98): ``np.fliplr`` acts on axis 1 (= channels for a
    ``(T,C,rows,W)`` slab), so the halo rows keep their row order (rows 1..top,
    and H-bottom-1..H-2) while the channel order is reversed."""
    H = data.shape[-2]
    top = (target_h - H) // 2
    bot = target_h - H - top
    if top + 1 > H or bot + 1 > H:
        raise AttributeError("The requested padding size is larger than height size of the input image.")
    upper = data[..., 1:top + 1, :]
    lower = data[..., H - bot - 1:H - 1, :]
    if mode == "reflect":
        upper, lower = upper[..., ::-1, :], lower[..., ::-1, :]
    elif mode == "reference_rnn":
        assert data.ndim == 4, "reference_rnn mode is defined for (T,C,H,W) slabs"
        upper, lower = upper[:, ::-1], lower[:, ::-1]
    else:
        raise ValueError(mode)
    return np.concatenate([upper, data, lower], axis=-2)


def halo_pad(data: np.ndarray, target_hw: Tuple[int, int], mode: str = "reflect") -> np.ndarray:
    """cyclic longitude then latitude halo (dataset.py:55-58)."""
    return reflect_pad_lat(cyclic_pad_lon(data, target_hw[1]), target_hw[0], mode)


def normalise_static_attributes(fields: np.ndarray) -> np.ndarray:
    """dataset.py:109-116: per-field spatial z-score of the static attributes [S,H,W]."""
    S = np.asarray(fields)
    return (S - S.mean(axis=(1, 2)).reshape(-1, 1, 1)) / S.std(axis=(1, 2)).reshape(-1, 1, 1)


def fuse_inputs(levels3d: np.ndarray, emis2d: np.ndarray, mean: np.ndarray, std: np.ndarray,
                target_hw: Optional[Tuple[int, int]] = None, mode: str = "reflect",
                statics: Optional[np.ndarray] = None) -> np.ndarray:
    """Preprocessing fusion: stack ``levels3d`` [T,L,H,W] (first L model levels of
    the 3-D forcings) with the 2-D emission field ``emis2d`` [T,H,W] as channel L,
    z-score per channel, then halo-pad.  Follows the shipped single-level code
    (stack dataset.py:526, z-score dataset.py:520-529, pad dataset.py:535-536).
    PARITY UNPINNED for L > 1: the README's 20-level module has no shipped code
    (SURVEY.md section 0, discrepancy 2)."""
    X = np.concatenate([levels3d, emis2d[:, None]], axis=1).astype(np.float32)
    X = (X - mean.reshape(1, -1, 1, 1).astype(np.float32)) / std.reshape(1, -1, 1, 1).astype(np.float32)
    if statics is not None:   # dataset.py:118-122, 532-533: normalised static fields repeated over the sequence
        rep = np.repeat(np.expand_dims(statics.astype(np.float32), 0), repeats=X.shape[0], axis=0)
        X = np.concatenate((X, rep), axis=1)
    if target_hw is not None:
        X = halo_pad(X, target_hw, mode)
    return X.astype(np.float32)


# --------------------------------------------------------------------------
# error metric (SURVEY 8d "Parity metric")
# --------------------------------------------------------------------------
def max_abs_normalised(a, b) -> float:
    """max|a-b| / max|b| with b the fp32 oracle."""
    a = torch.as_tensor(a, dtype=torch.float64)
    b = torch.as_tensor(b, dtype=torch.float64)
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def rel_l2(a, b) -> float:
    a = torch.as_tensor(a, dtype=torch.float64)
    b = torch.as_tensor(b, dtype=torch.float64)
    return float((a - b).norm() / b.norm().clamp_min(1e-30))
