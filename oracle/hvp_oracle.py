"""CPU reference for the second-order adjoint (Hessian-vector products).  TEST INFRASTRUCTURE ONLY.

An explicit restatement, in the style of ``convlstm_oracle.manual_backward``, of what
``nint_backward_second_order`` computes: the forward of ``state_oracle.convlstm_forward_state``
saving gates and cell states, the tangent-linear pass saving the gate pre-activation tangents and
the cell-state tangents, and one reverse pass that carries the adjoint (eta = dL/dh_t,
kappa = dL/dc_t) together with its tangent.  No autograd is used for the model; the loss's own
gradient u and its tangent du come from torch.func on the output tensors, as in ConvLSTM.hvp.
The CPU tests check it against torch.func.jvp(torch.func.grad(L o f)); the GPU tests compare the
CUDA path against torch.func on the fp32 oracle.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

Tensor = torch.Tensor
Pairs = Optional[Sequence[Tuple[Optional[Tensor], Optional[Tensor]]]]


def _split4(t: Tensor, hc: int):
    return torch.split(t, hc, 1)


def hvp_restatement(x: Tensor, params: Dict[str, Tensor], num_layers: int, loss_fn: Callable,
                    state: Pairs = None, dx: Optional[Tensor] = None, dstate: Pairs = None,
                    return_sequence: bool = False):
    """(loss, (grad_x, [(grad_h0, grad_c0)]), (hvp_x, [(hvp_h0, hvp_c0)])) of loss_fn(out) with out what
    ``convlstm_forward_state(x, params, num_layers, state, return_sequence)[0]`` returns, w.r.t. x and
    the initial state, in the direction v = (dx, dstate) (None: zero), at fixed parameters.

    Per step t (descending) and layer l (top first), with gates i, f, g, o, c_p = c_{t-1}, c = c_t,
    tau = tanh c, and the tangents di = i(1-i) da_i, df = f(1-f) da_f, dg = (1-g^2) da_g,
    do = o(1-o) da_o, dtau = (1-tau^2) dc:
      kt   = k + eta o (1-tau^2)        dkt  = dk + deta o (1-tau^2) + eta do (1-tau^2) - 2 eta o tau dtau
      ai   = kt g i(1-i)                dai  = dkt g i(1-i) + kt dg i(1-i) + kt g (1-2i) di
      af   = kt c_p f(1-f)              daf  = dkt c_p f(1-f) + kt dc_p f(1-f) + kt c_p (1-2f) df
      ag   = kt i (1-g^2)               dag  = dkt i (1-g^2) + kt di (1-g^2) - 2 kt i g dg
      ao   = eta tau o(1-o)             dao  = deta tau o(1-o) + eta dtau o(1-o) + eta tau (1-2o) do
      k   <- kt f                       dk  <- dkt f + kt df
    eta / deta at (t, l) = the h part of (a, da)_{t+1} (*) flip(W_l) + the x part of (a, da)_t of layer
    l+1 (*) flip(W_{l+1}) + u_t w_head / du_t w_head on the top layer.  Layer 0's x part of (a, da)_t is
    (grad, H v) w.r.t. x_t; at t = 0 the h part of (a, da)_0 and (k, dk) are those w.r.t. (h0, c0)."""
    B, T, _, H, W = x.shape
    L = num_layers
    Wt = [params[f"layers.{l}.conv.weight"] for l in range(L)]
    bs = [params[f"layers.{l}.conv.bias"] for l in range(L)]
    hc = [b.shape[0] // 4 for b in bs]
    hw = params["conv.weight"]
    zeros = lambda l: torch.zeros(B, hc[l], H, W, dtype=x.dtype)
    pick = lambda pairs, l, j: (pairs[l][j] if pairs is not None and pairs[l][j] is not None else zeros(l))
    dx = torch.zeros_like(x) if dx is None else dx
    # ---- forward and tangent, saving gates, c, and the tangents of the pre-activations and of c
    hs = [[pick(state, l, 0)] for l in range(L)]        # hs[l][t] = h_{t-1}
    cs = [[pick(state, l, 1)] for l in range(L)]
    dhs = [[pick(dstate, l, 0)] for l in range(L)]
    dcs = [[pick(dstate, l, 1)] for l in range(L)]
    gates = [[None] * T for _ in range(L)]
    dgates = [[None] * T for _ in range(L)]             # (di, df, dg, do)
    preds, dpreds = [], []
    for t in range(T):
        inp, dinp = x[:, t], dx[:, t]
        for l in range(L):
            p = Wt[l].shape[-1] // 2
            a = F.conv2d(torch.cat([inp, hs[l][t]], 1), Wt[l], bs[l], padding=p)
            da = F.conv2d(torch.cat([dinp, dhs[l][t]], 1), Wt[l], None, padding=p)
            ai, af, ag, ao = _split4(a, hc[l])
            i, f, g, o = torch.sigmoid(ai), torch.sigmoid(af), torch.tanh(ag), torch.sigmoid(ao)
            dai, daf, dag, dao = _split4(da, hc[l])
            di, df, dg, do = i * (1 - i) * dai, f * (1 - f) * daf, (1 - g * g) * dag, o * (1 - o) * dao
            c = cs[l][t] * f + i * g
            dc = dcs[l][t] * f + cs[l][t] * df + di * g + i * dg
            tau = torch.tanh(c)
            h = o * tau
            dh = do * tau + o * (1 - tau * tau) * dc
            gates[l][t], dgates[l][t] = (i, f, g, o), (di, df, dg, do)
            hs[l].append(h)
            cs[l].append(c)
            dhs[l].append(dh)
            dcs[l].append(dc)
            inp, dinp = h, dh
        if return_sequence or t == T - 1:
            preds.append(F.conv2d(inp, hw, params["conv.bias"]))
            dpreds.append(F.conv2d(dinp, hw, None))
    pred, dpred = preds[-1], dpreds[-1]
    out = (pred, torch.cat(preds, 1)) if return_sequence else pred
    dout = (dpred, torch.cat(dpreds, 1)) if return_sequence else dpred
    # ---- the loss's gradient u and its tangent du (small output tensors)
    (u, loss), (du, _) = torch.func.jvp(torch.func.grad_and_value(loss_fn), (out,), (dout,))
    if return_sequence:       # pred is the last step of seq: fold its seed into the per-step ones
        us, dus = u[1].clone(), du[1].clone()
        us[:, -1] += u[0][:, 0]
        dus[:, -1] += du[0][:, 0]
    else:
        us, dus = torch.zeros(B, T, H, W, dtype=x.dtype), torch.zeros(B, T, H, W, dtype=x.dtype)
        us[:, -1], dus[:, -1] = u[:, 0], du[:, 0]
    # ---- reverse pass: the adjoint and its tangent together
    gx, hx = torch.zeros_like(x), torch.zeros_like(x)
    eta_next = [zeros(l) for l in range(L)]              # h part of the dgrad of (a, da)_{t+1}
    deta_next = [zeros(l) for l in range(L)]
    k = [zeros(l) for l in range(L)]
    dk = [zeros(l) for l in range(L)]
    gh0: List[Tensor] = [zeros(l) for l in range(L)]
    hh0: List[Tensor] = [zeros(l) for l in range(L)]
    for t in reversed(range(T)):
        up, dup = None, None                             # x part of the layer above's dgrad at t
        for l in reversed(range(L)):
            eta, deta = eta_next[l].clone(), deta_next[l].clone()
            if l == L - 1:
                eta = eta + us[:, t:t + 1] * hw.reshape(1, -1, 1, 1)
                deta = deta + dus[:, t:t + 1] * hw.reshape(1, -1, 1, 1)
            if up is not None:
                eta, deta = eta + up, deta + dup
            i, f, g, o = gates[l][t]
            di, df, dg, do = dgates[l][t]
            cp, c, dcp, dc = cs[l][t], cs[l][t + 1], dcs[l][t], dcs[l][t + 1]
            tau = torch.tanh(c)
            tt = 1 - tau * tau
            dtau = tt * dc
            kt = k[l] + eta * o * tt
            dkt = dk[l] + deta * o * tt + eta * do * tt - 2 * eta * o * tau * dtau
            si, sf, so, tg = i * (1 - i), f * (1 - f), o * (1 - o), 1 - g * g
            a = torch.cat([kt * g * si, kt * cp * sf, kt * i * tg, eta * tau * so], 1)
            da = torch.cat([dkt * g * si + kt * dg * si + kt * g * (1 - 2 * i) * di,
                            dkt * cp * sf + kt * dcp * sf + kt * cp * (1 - 2 * f) * df,
                            dkt * i * tg + kt * di * tg - 2 * kt * i * g * dg,
                            deta * tau * so + eta * dtau * so + eta * tau * (1 - 2 * o) * do], 1)
            k[l], dk[l] = kt * f, dkt * f + kt * df
            p = Wt[l].shape[-1] // 2
            comb = F.conv_transpose2d(a, Wt[l], padding=p)
            dcomb = F.conv_transpose2d(da, Wt[l], padding=p)
            cin = comb.shape[1] - hc[l]
            eta_next[l], deta_next[l] = comb[:, cin:], dcomb[:, cin:]
            if l == 0:
                gx[:, t], hx[:, t] = comb[:, :cin], dcomb[:, :cin]
            else:
                up, dup = comb[:, :cin], dcomb[:, :cin]
            if t == 0:
                gh0[l], hh0[l] = comb[:, cin:], dcomb[:, cin:]
    return loss, (gx, list(zip(gh0, k))), (hx, list(zip(hh0, dk)))
