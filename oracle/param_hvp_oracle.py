"""CPU reference for Hessian-vector products over the parameters jointly with the inputs and the initial state.
TEST INFRASTRUCTURE ONLY.

An explicit restatement of what the tangent pass with a parameter direction, ``nint_backward_second_order`` on a plan
with ``NINT_FLAG_PARAM_TANGENT`` and ``nint_backward_second_order_params`` compute, written as the formulas of
DESIGN.md section 10 (f9) on top of the recursion of ``hvp_oracle.hvp_restatement``.  No autograd is used for the
model; the loss's gradient u and its tangent du come from torch.func on the output tensors.  The CPU tests check it
against torch.func.jvp(torch.func.grad(L o f)) over (theta, x, h0, c0); the GPU tests compare the CUDA path against
torch.func on the fp32 reference loop.
"""
from __future__ import annotations

from typing import Callable, Dict, Optional

import torch
import torch.nn.functional as F

from .hvp_oracle import Pairs

Tensor = torch.Tensor


def _wgrad(a: Tensor, comb: Tensor, shape, p: int) -> Tensor:
    """dL/dW of pre = W (*) comb for dL/dpre = a (the wgrad of one step)"""
    return torch.nn.grad.conv2d_weight(comb, shape, a, padding=p)


def param_hvp_restatement(x: Tensor, params: Dict[str, Tensor], num_layers: int, loss_fn: Callable,
                          state: Pairs = None, dx: Optional[Tensor] = None, dstate: Pairs = None,
                          dparams: Optional[Dict[str, Tensor]] = None, return_sequence: bool = False):
    """(loss, grad, hvp) with grad = (d/dx, [(d/dh0, d/dc0)], {name: d/dtheta}) of loss_fn(out), out what
    ``convlstm_forward_state(x, params, num_layers, state, return_sequence)[0]`` returns, and hvp the same blocks of
    H v for the joint direction v = (dx, dstate, dparams) (None / missing keys: zero).

    Tangent pass: dpre = W (*) dcomb + dW (*) comb + db, dpred_t = w_head . dh_t + dw_head . h_t + db_head.
    Reverse pass (hvp_oracle's recursion for (a, da) = dL/dpre and its tangent) with the parameter terms
      deta_t^l   += dW_h^l^T (*) a_{t+1}^l + dW_x^{l+1}^T (*) a_t^{l+1}     (+ u_t dw_head on the top layer)
      (H v)_x_t  += dW_x^0^T (*) a_t^0,     (H v)_h0^l += dW_h^l^T (*) a_0^l
    and the parameter outputs
      grad_W = sum_t wgrad(a_t, comb_t)          grad_b = sum a
      Hv_W   = sum_t wgrad(da_t, comb_t) + wgrad(a_t, dcomb_t)      Hv_b = sum da
      grad_w_head = sum u h,  grad_b_head = sum u,  Hv_w_head = sum du h + u dh,  Hv_b_head = sum du."""
    B, T, _, H, W = x.shape
    L = num_layers
    dparams = dparams or {}
    d = lambda name: dparams[name] if dparams.get(name) is not None else torch.zeros_like(params[name])
    Wt = [params[f"layers.{l}.conv.weight"] for l in range(L)]
    bs = [params[f"layers.{l}.conv.bias"] for l in range(L)]
    dWt = [d(f"layers.{l}.conv.weight") for l in range(L)]
    dbs = [d(f"layers.{l}.conv.bias") for l in range(L)]
    hw, hb, dhw, dhb = params["conv.weight"], params["conv.bias"], d("conv.weight"), d("conv.bias")
    hc = [b.shape[0] // 4 for b in bs]
    pad = [w.shape[-1] // 2 for w in Wt]
    zeros = lambda l: torch.zeros(B, hc[l], H, W, dtype=x.dtype)
    pick = lambda pairs, l, j: (pairs[l][j] if pairs is not None and pairs[l][j] is not None else zeros(l))
    dx = torch.zeros_like(x) if dx is None else dx
    # ---- forward and tangent, saving comb, dcomb, gates, their tangents, c and dc
    h = [pick(state, l, 0) for l in range(L)]
    dh = [pick(dstate, l, 0) for l in range(L)]
    cs = [[pick(state, l, 1)] for l in range(L)]
    dcs = [[pick(dstate, l, 1)] for l in range(L)]
    combs = [[None] * T for _ in range(L)]
    dcombs = [[None] * T for _ in range(L)]
    gates = [[None] * T for _ in range(L)]
    dgates = [[None] * T for _ in range(L)]
    top_h, top_dh = [], []
    preds, dpreds = [], []
    for t in range(T):
        inp, dinp = x[:, t], dx[:, t]
        for l in range(L):
            comb, dcomb = torch.cat([inp, h[l]], 1), torch.cat([dinp, dh[l]], 1)
            a = F.conv2d(comb, Wt[l], bs[l], padding=pad[l])
            da = F.conv2d(dcomb, Wt[l], None, padding=pad[l]) + F.conv2d(comb, dWt[l], dbs[l], padding=pad[l])
            ai, af, ag, ao = torch.split(a, hc[l], 1)
            i, f, g, o = torch.sigmoid(ai), torch.sigmoid(af), torch.tanh(ag), torch.sigmoid(ao)
            dai, daf, dag, dao = torch.split(da, hc[l], 1)
            di, df, dg, do = i * (1 - i) * dai, f * (1 - f) * daf, (1 - g * g) * dag, o * (1 - o) * dao
            c = cs[l][t] * f + i * g
            dc = dcs[l][t] * f + cs[l][t] * df + di * g + i * dg
            tau = torch.tanh(c)
            h[l], dh[l] = o * tau, do * tau + o * (1 - tau * tau) * dc
            combs[l][t], dcombs[l][t] = comb, dcomb
            gates[l][t], dgates[l][t] = (i, f, g, o), (di, df, dg, do)
            cs[l].append(c)
            dcs[l].append(dc)
            inp, dinp = h[l], dh[l]
        top_h.append(inp)
        top_dh.append(dinp)
        if return_sequence or t == T - 1:
            preds.append(F.conv2d(inp, hw, hb))
            dpreds.append(F.conv2d(dinp, hw, None) + F.conv2d(inp, dhw, dhb))
    out = (preds[-1], torch.cat(preds, 1)) if return_sequence else preds[-1]
    dout = (dpreds[-1], torch.cat(dpreds, 1)) if return_sequence else dpreds[-1]
    (u, loss), (du, _) = torch.func.jvp(torch.func.grad_and_value(loss_fn), (out,), (dout,))
    if return_sequence:
        us, dus = u[1].clone(), du[1].clone()
        us[:, -1] += u[0][:, 0]
        dus[:, -1] += du[0][:, 0]
    else:
        us, dus = torch.zeros(B, T, H, W, dtype=x.dtype), torch.zeros(B, T, H, W, dtype=x.dtype)
        us[:, -1], dus[:, -1] = u[:, 0], du[:, 0]
    # ---- reverse pass: the adjoint and its tangent together, and the parameter reductions
    gx, hx = torch.zeros_like(x), torch.zeros_like(x)
    eta_next = [zeros(l) for l in range(L)]
    deta_next = [zeros(l) for l in range(L)]
    k = [zeros(l) for l in range(L)]
    dk = [zeros(l) for l in range(L)]
    gh0, hh0 = [zeros(l) for l in range(L)], [zeros(l) for l in range(L)]
    gW = [torch.zeros_like(w) for w in Wt]
    hW = [torch.zeros_like(w) for w in Wt]
    gb = [torch.zeros_like(b) for b in bs]
    hbv = [torch.zeros_like(b) for b in bs]
    ghw, ghb, hhw, hhb = (torch.zeros_like(hw), torch.zeros_like(hb), torch.zeros_like(hw), torch.zeros_like(hb))
    for t in reversed(range(T)):
        ut, dut = us[:, t:t + 1], dus[:, t:t + 1]
        ghw += (ut * top_h[t]).sum((0, 2, 3)).reshape(hw.shape)
        ghb += ut.sum().reshape(1)
        hhw += (dut * top_h[t] + ut * top_dh[t]).sum((0, 2, 3)).reshape(hw.shape)
        hhb += dut.sum().reshape(1)
        up, dup = None, None
        for l in reversed(range(L)):
            eta, deta = eta_next[l].clone(), deta_next[l].clone()
            if l == L - 1:
                eta = eta + ut * hw.reshape(1, -1, 1, 1)
                deta = deta + dut * hw.reshape(1, -1, 1, 1) + ut * dhw.reshape(1, -1, 1, 1)
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
            gW[l] += _wgrad(a, combs[l][t], Wt[l].shape, pad[l])
            hW[l] += _wgrad(da, combs[l][t], Wt[l].shape, pad[l]) + _wgrad(a, dcombs[l][t], Wt[l].shape, pad[l])
            gb[l] += a.sum((0, 2, 3))
            hbv[l] += da.sum((0, 2, 3))
            comb = F.conv_transpose2d(a, Wt[l], padding=pad[l])
            dcomb = F.conv_transpose2d(da, Wt[l], padding=pad[l]) + F.conv_transpose2d(a, dWt[l], padding=pad[l])
            cin = comb.shape[1] - hc[l]
            eta_next[l], deta_next[l] = comb[:, cin:], dcomb[:, cin:]
            if l == 0:
                gx[:, t], hx[:, t] = comb[:, :cin], dcomb[:, :cin]
            else:
                up, dup = comb[:, :cin], dcomb[:, :cin]
            if t == 0:
                gh0[l], hh0[l] = comb[:, cin:], dcomb[:, cin:]
    gp, hp = {}, {}
    for l in range(L):
        gp[f"layers.{l}.conv.weight"], gp[f"layers.{l}.conv.bias"] = gW[l], gb[l]
        hp[f"layers.{l}.conv.weight"], hp[f"layers.{l}.conv.bias"] = hW[l], hbv[l]
    gp["conv.weight"], gp["conv.bias"], hp["conv.weight"], hp["conv.bias"] = ghw, ghb, hhw, hhb
    return loss, (gx, list(zip(gh0, k)), gp), (hx, list(zip(hh0, dk)), hp)
