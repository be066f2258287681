"""CPU reference for the parameter-space tangent (J dtheta jointly with J dx, J dstate).  TEST INFRASTRUCTURE ONLY.

An explicit restatement of what ``nint_forward_tangent`` computes once a parameter direction is set
(``nint_plan_set_weight_tangent`` / ``nint_plan_set_head_tangent``): the forward loop of
``state_oracle.convlstm_forward_state`` and, next to it, the tangent-linear recursion with the
parameter terms written out as formulas.  No autograd is used for the model.  The CPU tests check it
against ``torch.func.jvp`` of the reference loop with the parameters as an argument; the GPU tests
compare the CUDA path against ``torch.func.jvp`` of the fp32 reference loop.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

Tensor = torch.Tensor
Pairs = Optional[Sequence[Tuple[Optional[Tensor], Optional[Tensor]]]]


def jvp_restatement(x: Tensor, params: Dict[str, Tensor], num_layers: int, state: Pairs = None,
                    dx: Optional[Tensor] = None, dstate: Pairs = None, dparams: Optional[Dict[str, Tensor]] = None,
                    return_sequence: bool = False):
    """((out, [(h_T, c_T)]), (dout, [(dh_T, dc_T)])) with out what
    ``convlstm_forward_state(x, params, num_layers, state, return_sequence)[0]`` returns and dout its
    derivative in the joint direction (dx, dstate, dparams); dparams is keyed like ``params`` and a
    missing key (or None) is zero.

    Per step t and layer l, with comb = [x_t^l, h_{t-1}^l] (x_t^l = h_t^{l-1} for l >= 1) and dcomb
    likewise:
      dpre = W (*) dcomb + dW (*) comb + db
      di = i(1-i) dpre_i  df = f(1-f) dpre_f  dg = (1-g^2) dpre_g  do = o(1-o) dpre_o
      dc = f dc_{t-1} + c_{t-1} df + g di + i dg      dh = tanh(c) do + o (1 - tanh^2 c) dc
    and the head dpred_t = w_head . dh_t + dw_head . h_t + db_head."""
    B, T, _, H, W = x.shape
    L = num_layers
    dparams = dparams or {}
    Wt = [params[f"layers.{l}.conv.weight"] for l in range(L)]
    bs = [params[f"layers.{l}.conv.bias"] for l in range(L)]
    hc = [b.shape[0] // 4 for b in bs]
    zero = lambda name: torch.zeros_like(params[name])
    dWt = [dparams.get(f"layers.{l}.conv.weight") for l in range(L)]
    dWt = [zero(f"layers.{l}.conv.weight") if d is None else d for l, d in enumerate(dWt)]
    dbs = [dparams.get(f"layers.{l}.conv.bias") for l in range(L)]
    dbs = [zero(f"layers.{l}.conv.bias") if d is None else d for l, d in enumerate(dbs)]
    hw, hb = params["conv.weight"], params["conv.bias"]
    dhw = dparams.get("conv.weight")
    dhw = zero("conv.weight") if dhw is None else dhw
    dhb = dparams.get("conv.bias")
    dhb = zero("conv.bias") if dhb is None else dhb
    zeros = lambda l: torch.zeros(B, hc[l], H, W, dtype=x.dtype)
    pick = lambda pairs, l, j: (pairs[l][j] if pairs is not None and pairs[l][j] is not None else zeros(l))
    dx = torch.zeros_like(x) if dx is None else dx
    h = [pick(state, l, 0) for l in range(L)]
    c = [pick(state, l, 1) for l in range(L)]
    dh = [pick(dstate, l, 0) for l in range(L)]
    dc = [pick(dstate, l, 1) for l in range(L)]
    preds, dpreds = [], []
    for t in range(T):
        inp, dinp = x[:, t], dx[:, t]
        for l in range(L):
            p = Wt[l].shape[-1] // 2
            comb = torch.cat([inp, h[l]], 1)
            dcomb = torch.cat([dinp, dh[l]], 1)
            pre = F.conv2d(comb, Wt[l], bs[l], padding=p)
            dpre = F.conv2d(dcomb, Wt[l], None, padding=p) + F.conv2d(comb, dWt[l], dbs[l], padding=p)
            ai, af, ag, ao = torch.split(pre, hc[l], 1)
            i, f, g, o = torch.sigmoid(ai), torch.sigmoid(af), torch.tanh(ag), torch.sigmoid(ao)
            dai, daf, dag, dao = torch.split(dpre, hc[l], 1)
            di, df, dg, do = i * (1 - i) * dai, f * (1 - f) * daf, (1 - g * g) * dag, o * (1 - o) * dao
            c_new = f * c[l] + i * g
            dc_new = f * dc[l] + c[l] * df + g * di + i * dg
            tau = torch.tanh(c_new)
            h[l], c[l] = o * tau, c_new
            dh[l], dc[l] = tau * do + o * (1 - tau * tau) * dc_new, dc_new
            inp, dinp = h[l], dh[l]
        if return_sequence or t == T - 1:
            preds.append(F.conv2d(inp, hw, hb))
            dpreds.append(F.conv2d(dinp, hw, None) + F.conv2d(inp, dhw, dhb))
    out = (preds[-1], torch.cat(preds, 1)) if return_sequence else preds[-1]
    dout = (dpreds[-1], torch.cat(dpreds, 1)) if return_sequence else dpreds[-1]
    return (out, list(zip(h, c))), (dout, list(zip(dh, dc)))
