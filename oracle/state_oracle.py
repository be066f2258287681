"""CPU reference for the stateful ConvLSTM surface.  TEST INFRASTRUCTURE ONLY.

``ConvLSTM.forward`` (model.py:253-274) always starts from zeros; this is the same
loop started from a given per-layer state, returning the final one, built from
the pinned ``convlstm_oracle.cell_forward``.  The tests compare the CUDA path's
``hidden_state`` / ``return_state`` results and their gradients (autograd through
this loop) against it.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

from .convlstm_oracle import cell_forward

Tensor = torch.Tensor


def convlstm_forward_state(x: Tensor, params: Dict[str, Tensor], num_layers: int,
                           state: Optional[Sequence[Tuple[Optional[Tensor], Optional[Tensor]]]] = None,
                           return_sequence: bool = False):
    """``convlstm_oracle.convlstm_forward`` (the loop of model.py:253-274) started from a given
    per-layer ``state`` = [(h_l, c_l)] [B,Hc_l,H,W] instead of zeros (None, or a
    None tensor: zeros).  Returns ``(out, [(h_T, c_T) per layer])`` with ``out``
    what ``convlstm_forward`` returns; differentiable w.r.t. the state."""
    B, T, _, H, W = x.shape
    hs: List[Tensor] = []
    cs: List[Tensor] = []
    for l in range(num_layers):
        hc = params[f"layers.{l}.conv.bias"].shape[0] // 4
        h0, c0 = state[l] if state is not None else (None, None)
        hs.append(torch.zeros(B, hc, H, W, dtype=x.dtype) if h0 is None else h0)
        cs.append(torch.zeros(B, hc, H, W, dtype=x.dtype) if c0 is None else c0)
    outs = []
    h = None
    for t in range(T):
        inp = x[:, t]
        for l in range(num_layers):
            h, c = cell_forward(inp, hs[l], cs[l], params[f"layers.{l}.conv.weight"],
                                params[f"layers.{l}.conv.bias"])
            hs[l], cs[l] = h, c
            inp = h
        if return_sequence:
            outs.append(F.conv2d(h, params["conv.weight"], params["conv.bias"]))
    pred = F.conv2d(h, params["conv.weight"], params["conv.bias"])
    out = (pred, torch.cat(outs, dim=1)) if return_sequence else pred
    return out, list(zip(hs, cs))


