"""Integer-lattice case D: carried state, the tangent pass, the second-order pass and the params call, exactly.
TEST INFRASTRUCTURE ONLY.

Case D extends ``lattice.case_b``'s interleaving to every layer and every step of a whole ConvLSTM that starts from an
explicit initial state.  *Live* channels hold nonzero values and get zero weight columns; *silent* channels hold zero
values and get lattice weight columns.  Every gate pre-activation is then exactly its bias at every step, and layer 0's
live hidden channels are layer 1's live x channels.  Each hidden channel is in one of three modes:

* silent (odd channels): b = 0, h0 = c0 = 0, so c = h = 0 at every step (tanh' = 1): the g row of dgates and the
  recurrent dgrad;
* live F (f = 1/2, g = 0): c0 = +-24 * 2^T, so |c_t| >= 24, tanh(c_t) = +-1 and h_t = +-1/2 at every step: the f and o
  rows;
* live G (b_g = +-40, g = +-1): c0 = g * 24 * 2^T, so c_t keeps its sign and |c_t| >= 24: the i row.

Both activation variants of the kernels (nint_common.cuh act_tanh / act_sigmoid_halved, FAST and precise) give exactly
sigmoid(0) = 1/2 and tanh(x) = +-1 for |x| >= 24, and tangent_cell_body / soa_cell_body call the same functions as the
forward epilogue.  Every seed (x, h0, c0, dpred, dseq, dh_T, dc_T, the directions dx, dh0, dc0 and dtheta -- dW on
every column, live ones included, so dW (*) comb sees h = +-1/2 -- and the second-order seeds u, du) is a sparse small
integer, so every product is on a power-of-two grid and every sum is exact in fp32 (``headroom``).

``reference`` evaluates the case for every pass, with the kernels' roundings emulated where they happen:
* the ordinary backward (Plan.backward with dh_T / dc_T): dgates rounded to the operand format, the tf32 bias
  residuals under ``lattice.resid_on``;
* the tangent pass: dX and dh0 rounded to the operand format (input packing), dh_t rounded as tangent_cell_body
  stores it (nint_pointwise.cu round_for: bf16 round-to-nearest-even, tf32 cvt.rna);
* the second-order pass: (a, da) rounded to the operand format (soa_cell_body); eta, deta, kappa, dkappa stay fp32;
* the params call (Plan.backward_second_order_params): wgrads over the rounded (a, da) and the rounded tangent
  activations, and bias sums of the rounded (a, da) with NO tf32 residuals (param_wgrad passes none).

At every lattice point sigma(1-sigma)(1-2sigma) = 0 and tanh(1-tanh^2) = 0, so the second-derivative terms of
soa_cell_body are exactly zero here; they stay covered by the tolerance tests only.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import torch
import torch.nn.functional as F

from . import lattice as Lt
from .lattice import _Rng, _conv, _dgrad, _note, _pixsum, _tap_hits, _tile_mask, _wgrad, grid, live_channels

DEFECTS = ("tangent_recurrent_slot", "tangent_t0_drops_h0", "dw_ifo_not_halved", "params_reads_a_for_da",
           "soa_recurrent_slot", "dh_T_not_joined", "dc0_one_step_early", "params_drop_ragged_tile",
           "params_drop_splitk_share")
SATURATE = 24.0


def _modes(hc):
    """0 silent (odd channels), 1 live F, 2 live G (alternating over the even channels)"""
    j = torch.arange(hc)
    return torch.where(j % 2 == 1, 0, torch.where((j // 2) % 2 == 0, 1, 2))


def case_d(B, T, C, H, W, hidden, ks, precision, seed=0, wdensity=0.06, ddensity=0.1, xdensity=0.5, tdensity=0.1,
           sdensity=1.0, return_sequence=False, shared_frames=False, repeat_starts=False, wide=False):
    """whole-model case with carried state, upstream seeds, directions and second-order seeds.  shared_frames: the
    windows are frames[starts[b] : starts[b] + T] of one record; repeat_starts: pairs of samples share a start.
    tdensity: share of nonzero direction entries (dx, dW).  sdensity: share of the pixels where the live F channels
    saturate.  wide: 12-bit dtop, u and dx entries, so that dgates, (a, da) and the tangent's dh round"""
    r = _Rng(seed)
    L = len(hidden)
    dd = min(ddensity, 400.0 / (B * H * W))
    lx = live_channels(C)
    frames = starts = None
    if shared_frames:
        starts = torch.arange(B) // 2 if repeat_starts else torch.arange(B)
        n = int(starts.max()) + T
        frames = r.ints((n, C, H, W), -2, 2, xdensity) * lx.view(1, C, 1, 1)
        dframes = r.ints((n, C, H, W), -1, 1, tdensity)
        x = torch.stack([frames[s:s + T] for s in starts.tolist()])
        dx = torch.stack([dframes[s:s + T] for s in starts.tolist()])
    else:
        x = r.ints((B, T, C, H, W), -2, 2, xdensity) * lx.view(1, 1, C, 1, 1)
        dx = r.ints((B, T, C, H, W), -1, 1, tdensity)
        dframes = None
    ws, bs, dws, dbs, h0, c0, dh0, dc0, dh_T, dc_T = ([] for _ in range(10))
    cin = C
    for hc, k in zip(hidden, ks):
        m = _modes(hc)
        live = m > 0
        w = r.ints((4 * hc, cin + hc, k, k), -1, 1, wdensity)
        w[:, torch.cat([live_channels(cin), live])] = 0
        ws.append(w)
        gsign = r.signs((hc,))
        b = torch.zeros(4 * hc, dtype=torch.float64)
        b[2 * hc:3 * hc] = torch.where(m == 2, 40.0 * gsign, 0.0)
        bs.append(b)
        dws.append(r.ints((4 * hc, cin + hc, k, k), -1, 1, tdensity))
        dbs.append(r.ints((4 * hc,), -1, 1, 0.5))
        big = SATURATE * 2.0 ** T
        cm = lambda i: (m == i).view(1, hc, 1, 1).double()
        # live F channels saturate at a share sdensity of the pixels; elsewhere c0 = 0 keeps them at c = h = 0 (their
        # weight columns are zero, so there they act as silent channels and the large c_{t-1} terms stay sparse)
        fsat = r.signs((B, hc, H, W)) * (torch.rand((B, hc, H, W), generator=r.g) < sdensity).double()
        c0.append(big * (fsat * cm(1) + gsign.view(1, hc, 1, 1) * cm(2)))
        h0.append(r.ints((B, hc, H, W), -2, 2, 0.5) * live.view(1, hc, 1, 1).double())
        dh0.append(r.ints((B, hc, H, W), -1, 1, max(dd, 0.02)))
        dc0.append(r.ints((B, hc, H, W), -1, 1, max(dd, 0.02)))
        dh_T.append(r.ints((B, hc, H, W), -1, 1, dd))
        dc_T.append(r.ints((B, hc, H, W), -1, 1, dd))
        cin = hc
    hw = r.ints((1, hidden[-1], 1, 1), -2, 2)
    hw.view(-1)[0] = 1.0
    hb = torch.tensor([0.75], dtype=torch.float64)
    dhw = r.ints((1, hidden[-1], 1, 1), -1, 1)
    dhb = torch.tensor([0.5], dtype=torch.float64)

    def seed_pair():
        top = torch.zeros(B, T, H, W, dtype=torch.float64)
        top[:, T - 1] = r.ints((B, H, W), -1, 1, dd * 2)
        for y, xx in Lt._edge_pixels(H, W):
            top[:, T - 1, y, xx] = r.ints((B,), -1, 1, nonzero=True)
        if return_sequence:
            top[:, :T - 1] = r.ints((B, T - 1, H, W), -1, 1, dd)
        return top
    dtop, u, du = seed_pair(), seed_pair(), seed_pair()
    if wide:
        # 12-bit values, dtop and u at step 0 (so that they are not carried down the finer grids of the earlier steps)
        # and dx at the last step (so that it meets u only where u is small): dtop makes
        # the ordinary backward's dgates round (and, in tf32, reach the bias through the rounding residuals), u makes
        # (a, da) round, and dx on a silent channel makes the tangent's dh round
        assert return_sequence
        dtop[0, 0, H // 2, W // 2] = 2049.0
        u[0, 0, H // 2, W // 2] = 2049.0
        dx[0, T - 1, 1, H // 2, W // 2] = 2049.0
    return dict(kind="D", precision=precision, B=B, T=T, C=C, H=H, W=W, hidden=list(hidden), ks=list(ks), x=x,
                h0=h0, c0=c0, ws=ws, bs=bs, hw=hw, hb=hb, dtop=dtop, dh_T=dh_T, dc_T=dc_T, dx=dx, dh0=dh0, dc0=dc0,
                dws=dws, dbs=dbs, dhw=dhw, dhb=dhb, u=u, du=du, return_sequence=return_sequence, frames=frames,
                dframes=dframes, starts=starts, wide=wide)


def with_direction(case, which):
    """the case with only some parts of the joint direction: 'input', 'state', 'input_state', 'param' or 'joint'"""
    out = dict(case)
    z = lambda ts: [torch.zeros_like(t) for t in ts]
    if which not in ("input", "input_state", "joint"):
        out["dx"] = torch.zeros_like(case["dx"])
        if case["dframes"] is not None:
            out["dframes"] = torch.zeros_like(case["dframes"])
    if which not in ("state", "input_state", "joint"):
        out["dh0"], out["dc0"] = z(case["dh0"]), z(case["dc0"])
    if which not in ("param", "joint"):
        out["dws"], out["dbs"] = z(case["dws"]), z(case["dbs"])
        out["dhw"], out["dhb"] = torch.zeros_like(case["dhw"]), torch.zeros_like(case["dhb"])
    return out


def _round(t, precision):
    return t if precision is None else Lt.to_operand(t, precision)


def _round_dh(t, precision):
    """dh_t as tangent_cell_body stores it: round_for (tf32 cvt.rna) or the bf16 store (round-to-nearest-even)"""
    return _round(t, precision)


def _halve_ifo(t, hc):
    """the i, f, o quarters of a gate tensor (dim 1)"""
    m = torch.ones(4 * hc, dtype=t.dtype)
    m[2 * hc:3 * hc] = 0
    return t * m.view(1, -1, 1, 1)


def reference(case, dtype=torch.float64, order: Optional[int] = None, defect: Optional[str] = None,
              stats: Optional[dict] = None, rounding: bool = True) -> Dict[str, torch.Tensor]:
    """Every pass of a case D evaluated at ``dtype``.  ``order``: permutes the pixel order of every wgrad / bias sum and
    the time order of every sum over steps.  ``defect``: one of DEFECTS, planted.  ``stats``: filled with headroom
    (``stats['headroom']``) and coverage.  rounding=False: no operand rounding at all (the pure fp64 formulas)."""
    prec = case["precision"] if rounding else None
    B, T, C, H, W = case["B"], case["T"], case["C"], case["H"], case["W"]
    hidden, ks = case["hidden"], case["ks"]
    L = len(hidden)
    cv = lambda t: t.to(dtype)
    x, dX = cv(case["x"]), _round(cv(case["dx"]), prec)
    Ws, bs = [cv(w) for w in case["ws"]], [cv(b) for b in case["bs"]]
    dWs, dbs = [cv(w) for w in case["dws"]], [cv(b) for b in case["dbs"]]
    hw, hb, dhw, dhb = cv(case["hw"]), cv(case["hb"]), cv(case["dhw"]), cv(case["dhb"])
    resid = Lt.resid_on(case) and rounding
    perm = tperm = None
    if order is not None:
        g = torch.Generator().manual_seed(order)
        perm = torch.randperm(B * H * W, generator=g)
        tperm = torch.randperm(T, generator=g).tolist()
    steps = tperm if tperm is not None else list(reversed(range(T)))
    pads = [k // 2 for k in ks]
    cov = _new_cov(stats, case) if stats is not None else None
    hr = (lambda name, a, gam: _note(stats, name, a, gam)) if stats is not None else (lambda *a: None)
    A = lambda t: t.abs().double()
    out: Dict[str, torch.Tensor] = {}

    # ---- forward from the initial state
    hs = [[cv(case["h0"][l])] for l in range(L)]        # hs[l][t] = h_{t-1}
    cs = [[cv(case["c0"][l])] for l in range(L)]
    gates = [[None] * T for _ in range(L)]
    combs = [[None] * T for _ in range(L)]
    for t in range(T):
        inp = x[:, t]
        for l in range(L):
            hc = hidden[l]
            comb = torch.cat([inp, hs[l][t]], 1)
            pre = _conv(comb, Ws[l], pads[l]) + bs[l].view(1, -1, 1, 1)
            hr(f"gates{l}", F.conv2d(A(comb), A(Ws[l]), padding=pads[l]), grid(comb) * grid(Ws[l]))
            i, f, gg, o = torch.split(pre, hc, 1)
            i, f, gg, o = torch.sigmoid(i), torch.sigmoid(f), torch.tanh(gg), torch.sigmoid(o)
            c = cs[l][t] * f + i * gg
            h = o * torch.tanh(c)
            gates[l][t], combs[l][t] = (i, f, gg, o), comb
            if stats is not None:
                stats.setdefault("pre", []).append((l, pre - bs[l].view(1, -1, 1, 1)))
                stats.setdefault("c", []).append((l, c))
                stats.setdefault("h", []).append((l, h))
            hs[l].append(h)
            cs[l].append(c)
            inp = h
    top = [hs[L - 1][t + 1] for t in range(T)]
    seq = torch.cat([F.conv2d(h, hw, hb) for h in top], 1)
    out["pred"] = seq[:, T - 1:T]
    if case["return_sequence"]:
        out["seq"] = seq
    for l in range(L):
        out[f"hT{l}"], out[f"cT{l}"] = hs[l][T], cs[l][T]

    # ---- ordinary backward with the final-state seeds (Plan.backward(dh_T=, dc_T=))
    dtop = cv(case["dtop"])
    dh_next = [cv(case["dh_T"][l]) if defect != "dh_T_not_joined" else torch.zeros_like(hs[l][0]) for l in range(L)]
    dc_next = [cv(case["dc_T"][l]) for l in range(L)]
    habs = [A(t) for t in dh_next]
    hgam = [grid(t) for t in dh_next]
    contrib = [[None] * T for _ in range(L)]
    wabs = [torch.zeros(w.shape, dtype=torch.float64) for w in Ws]
    babs = [torch.zeros(b.shape, dtype=torch.float64) for b in bs]
    wgam, bgam = [math.inf] * L, [math.inf] * L
    dx = torch.zeros(B, T, C, H, W, dtype=dtype)
    dc0 = [None] * L
    for t in reversed(range(T)):
        up, up_abs, up_gam = None, None, math.inf
        for l in reversed(range(L)):
            hc = hidden[l]
            dh = dh_next[l] if up is None else dh_next[l] + up
            terms, gam = [habs[l]] + ([up_abs] if up_abs is not None else []), min(hgam[l], up_gam)
            if l == L - 1:
                head = dtop[:, t:t + 1] * hw.view(1, -1, 1, 1)
                dh = dh + head
                terms.append(A(head))
                gam = min(gam, grid(head))
            hr(f"dh{l}", sum(terms), gam)
            i, f, gg, o = gates[l][t]
            tc = torch.tanh(cs[l][t + 1])
            a1 = dh * o * (1 - tc * tc)
            dcv = dc_next[l] + a1
            hr(f"dc{l}", A(a1) + A(dc_next[l]), min(grid(a1), grid(dc_next[l])))
            dpre = torch.cat([dcv * gg * i * (1 - i), dcv * cs[l][t] * f * (1 - f), dcv * i * (1 - gg * gg),
                              dh * tc * o * (1 - o)], 1)
            dc_next[l] = dcv * f
            if t == 0:
                dc0[l] = dcv if defect == "dc0_one_step_early" else dc_next[l]
            dg = _round(dpre, prec)
            comb = combs[l][t]
            contrib[l][t] = (_wgrad(dg, comb, ks[l], perm), _pixsum(dpre if resid else dg, perm))
            dcomb = _dgrad(dg, Ws[l], pads[l])
            cin = comb.shape[1] - hc
            if stats is not None:
                ad = _dgrad(A(dg), A(Ws[l]), pads[l])
                gd = grid(dg) * grid(Ws[l])
                habs[l], hgam[l] = ad[:, cin:], gd
                up_abs, up_gam = ad[:, :cin], gd
                wabs[l] += _wgrad(A(dg), A(comb), ks[l])
                wgam[l] = min(wgam[l], grid(dg) * grid(comb))
                babs[l] += A(dpre).sum((0, 2, 3)) + A(dpre - dg).sum((0, 2, 3))
                bgam[l] = min(bgam[l], grid(dg), grid(dpre))
                _cover(cov, "bwd", l, t, dg, comb, Ws[l], ks[l], hc, cin)
            up = dcomb[:, :cin] if l > 0 else None
            if l == 0:
                dx[:, t] = dcomb[:, :cin]
            dh_next[l] = dcomb[:, cin:]
    for l in range(L):
        out[f"gw{l}"] = sum(contrib[l][t][0] for t in steps)
        out[f"gb{l}"] = sum(contrib[l][t][1] for t in steps)
        out[f"dh0_{l}"], out[f"dc0_{l}"] = dh_next[l], dc0[l]
        hr(f"dw{l}", wabs[l], wgam[l])
        hr(f"db{l}", babs[l], bgam[l])
        if stats is not None:
            cov["bwd_hcols_late"][l] = any(bool((contrib[l][t][0][:, comb_cin(case, l):] != 0).any()) for t in range(1, T))
    out["ghw"] = sum((dtop[:, t:t + 1] * top[t]).sum((0, 2, 3)) for t in steps).view(1, -1, 1, 1)
    out["ghb"] = sum(dtop[:, t].sum() for t in steps).view(1)
    out["dx"] = dx

    # ---- tangent pass (f7 + f9): dpre = W (*) dcomb + dW (*) comb + db
    dhs = [[_round(cv(case["dh0"][l]), prec)] for l in range(L)]
    dcs = [[cv(case["dc0"][l])] for l in range(L)]
    dgates = [[None] * T for _ in range(L)]
    dcombs = [[None] * T for _ in range(L)]
    for t in range(T):
        dinp = dX[:, t]
        for l in range(L):
            hc = hidden[l]
            comb = combs[l][t]
            dhr = dhs[l][t]
            if defect == "tangent_recurrent_slot" and t > 0:    # reads the neighbouring slot: dh_{t-2} for dh_{t-1}
                dhr = dhs[l][t - 1]
            dcomb = torch.cat([dinp, dhr], 1)
            pcomb = comb
            if defect == "tangent_t0_drops_h0" and t == 0:     # the zero-state rule applied to dW (*) comb
                pcomb = torch.cat([comb[:, :comb.shape[1] - hc], torch.zeros_like(comb[:, comb.shape[1] - hc:])], 1)
            pterm = _conv(pcomb, dWs[l], pads[l])
            if defect == "dw_ifo_not_halved":
                pterm = pterm + _halve_ifo(pterm, hc)
            dpre = _conv(dcomb, Ws[l], pads[l]) + pterm + dbs[l].view(1, -1, 1, 1)
            hr(f"tgates{l}", F.conv2d(A(dcomb), A(Ws[l]), padding=pads[l]) + F.conv2d(A(comb), A(dWs[l]), padding=pads[l])
               + A(dbs[l]).view(1, -1, 1, 1), min(grid(dcomb) * grid(Ws[l]), grid(comb) * grid(dWs[l]), grid(dbs[l])))
            i, f, gg, o = gates[l][t]
            dai, daf, dag, dao = torch.split(dpre, hc, 1)
            di, df, dgv, do = i * (1 - i) * dai, f * (1 - f) * daf, (1 - gg * gg) * dag, o * (1 - o) * dao
            dc = f * dcs[l][t] + cs[l][t] * df + gg * di + i * dgv
            tc = torch.tanh(cs[l][t + 1])
            dh = _round_dh(tc * do + o * (1 - tc * tc) * dc, prec)
            dgates[l][t], dcombs[l][t] = (di, df, dgv, do), dcomb
            if stats is not None:
                cov["dh_steps"][l][t] = bool((dh != 0).any())
            dhs[l].append(dh)
            dcs[l].append(dc)
            dinp = dh
    tseq = torch.cat([F.conv2d(dhs[L - 1][t + 1], hw) + F.conv2d(top[t], dhw, dhb) for t in range(T)], 1)
    for t in range(T):
        hr("head_tangent", F.conv2d(A(dhs[L - 1][t + 1]), A(hw)) + F.conv2d(A(top[t]), A(dhw)) + A(dhb),
           min(grid(dhs[L - 1][t + 1]) * grid(hw), grid(top[t]) * grid(dhw), grid(dhb)))
    out["t_pred"] = tseq[:, T - 1:T]
    if case["return_sequence"]:
        out["t_seq"] = tseq
    for l in range(L):
        out[f"t_hT{l}"], out[f"t_cT{l}"] = dhs[l][T], dcs[l][T]

    # ---- second-order pass (f8 + f9) and the params call
    us, dus = cv(case["u"]), cv(case["du"])
    eta_next = [torch.zeros_like(hs[l][0]) for l in range(L)]
    deta_next = [torch.zeros_like(hs[l][0]) for l in range(L)]
    late = [(torch.zeros_like(hs[l][0]), torch.zeros_like(hs[l][0])) for l in range(L)]   # the h part of step t+2
    eabs, egam = [None] * L, [math.inf] * L
    k_ = [torch.zeros_like(hs[l][0]) for l in range(L)]
    dk = [torch.zeros_like(hs[l][0]) for l in range(L)]
    sgx, shx = torch.zeros(B, T, C, H, W, dtype=dtype), torch.zeros(B, T, C, H, W, dtype=dtype)
    pc = [[None] * T for _ in range(L)]          # (grad W, grad b, Hv W, Hv b) of every (layer, step)
    mask = _tile_mask(B, H, W, defect[len("params_"):]) if defect and defect.startswith("params_drop") else None
    pw_abs = [[torch.zeros(w.shape, dtype=torch.float64) for w in Ws] for _ in range(3)]
    pw_gam = [[math.inf] * L for _ in range(3)]
    pb_abs = [[torch.zeros(b.shape, dtype=torch.float64) for b in bs] for _ in range(2)]
    pb_gam = [[math.inf] * L for _ in range(2)]
    for t in reversed(range(T)):
        ut, dut = us[:, t:t + 1], dus[:, t:t + 1]
        up = dup = None
        up_abs, up_gam = None, math.inf
        for l in reversed(range(L)):
            hc = hidden[l]
            eta, deta = eta_next[l], deta_next[l]
            terms, gam = ([eabs[l]] if eabs[l] is not None else []), egam[l]
            if l == L - 1:
                eta = eta + ut * hw.view(1, -1, 1, 1)
                deta = deta + dut * hw.view(1, -1, 1, 1) + ut * dhw.view(1, -1, 1, 1)
                terms += [A(ut * hw.view(1, -1, 1, 1)) + A(dut * hw.view(1, -1, 1, 1)) + A(ut * dhw.view(1, -1, 1, 1))]
                gam = min(gam, grid(ut) * grid(hw), grid(dut) * grid(hw), grid(ut) * grid(dhw))
            if up is not None:
                eta, deta = eta + up, deta + dup
                if up_abs is not None:
                    terms.append(up_abs)
                    gam = min(gam, up_gam)
            if terms:
                hr(f"eta{l}", sum(terms), gam)
            i, f, gg, o = gates[l][t]
            di, df, dgv, do = dgates[l][t]
            cp, c, dcp, dc = cs[l][t], cs[l][t + 1], dcs[l][t], dcs[l][t + 1]
            tau = torch.tanh(c)
            tt = 1 - tau * tau
            dtau = tt * dc
            kt = k_[l] + eta * o * tt
            dkt = dk[l] + deta * o * tt + eta * do * tt - 2 * eta * o * tau * dtau
            hr(f"kappa{l}", A(k_[l]) + A(eta * o * tt) + A(dk[l]) + A(deta * o * tt) + A(eta * do * tt),
               min(grid(k_[l]), grid(eta * o * tt), grid(dk[l]), grid(deta * o * tt), grid(eta * do * tt)))
            si, sf, so, tg = i * (1 - i), f * (1 - f), o * (1 - o), 1 - gg * gg
            a = torch.cat([kt * gg * si, kt * cp * sf, kt * i * tg, eta * tau * so], 1)
            da = torch.cat([dkt * gg * si + kt * dgv * si + kt * gg * (1 - 2 * i) * di,
                            dkt * cp * sf + kt * dcp * sf + kt * cp * (1 - 2 * f) * df,
                            dkt * i * tg + kt * di * tg - 2 * kt * i * gg * dgv,
                            deta * tau * so + eta * dtau * so + eta * tau * (1 - 2 * o) * do], 1)
            k_[l], dk[l] = kt * f, dkt * f + kt * df
            a, da = _round(a, prec), _round(da, prec)
            comb, dcomb = combs[l][t], dcombs[l][t]
            wa, wd = (a, da) if mask is None else (a * mask.to(dtype), da * mask.to(dtype))
            kind1 = wa if defect == "params_reads_a_for_da" else wd
            pc[l][t] = (_wgrad(wa, comb, ks[l], perm), _pixsum(wa, perm),
                        _wgrad(kind1, comb, ks[l], perm) + _wgrad(wa, dcomb, ks[l], perm), _pixsum(kind1, perm))
            # eta / deta of the step before: the h part of (a, da) (*) flip(W) (+ dW's terms over a)
            ec = _dgrad(a, Ws[l], pads[l])
            dec = _dgrad(da, Ws[l], pads[l]) + _dgrad(a, dWs[l], pads[l])
            cin = comb.shape[1] - hc
            if stats is not None:
                ad = _dgrad(A(a), A(Ws[l]), pads[l]) + _dgrad(A(da), A(Ws[l]), pads[l]) + _dgrad(A(a), A(dWs[l]), pads[l])
                gd = min(grid(a) * grid(Ws[l]), grid(da) * grid(Ws[l]), grid(a) * grid(dWs[l]))
                eabs[l], egam[l] = ad[:, cin:], gd
                up_abs, up_gam = ad[:, :cin], gd
                for j, (g_, c_) in enumerate(((a, comb), (da, comb), (a, dcomb))):
                    pw_abs[j][l] += _wgrad(A(g_), A(c_), ks[l])
                    pw_gam[j][l] = min(pw_gam[j][l], grid(g_) * grid(c_))
                    if j < 2:       # the bias sums of the gradient and of H v (kind 2 has none)
                        pb_abs[j][l] += A(g_).sum((0, 2, 3))
                        pb_gam[j][l] = min(pb_gam[j][l], grid(g_))
                ad2 = torch.cat([a, da], 0)
                _cover(cov, "soa", l, t, ad2, torch.cat([comb, dcomb], 0), Ws[l], ks[l], hc, cin)
            if defect == "soa_recurrent_slot":      # dh_{t-1} reads the neighbouring slot: (a, da) of step t+1
                (eta_next[l], deta_next[l]), late[l] = late[l], (ec[:, cin:], dec[:, cin:])
            else:
                eta_next[l], deta_next[l] = ec[:, cin:], dec[:, cin:]
            if l == 0:
                sgx[:, t], shx[:, t] = ec[:, :cin], dec[:, :cin]
                hr("soa_dx", up_abs if up_abs is not None else A(ec[:, :cin]), up_gam)
            else:
                up, dup = ec[:, :cin], dec[:, :cin]
            if t == 0:
                out[f"s_dh0_{l}"], out[f"s_ddh0_{l}"] = ec[:, cin:], dec[:, cin:]
    out["s_dx"], out["s_ddx"] = sgx, shx
    for l in range(L):
        out[f"s_dc0_{l}"], out[f"s_ddc0_{l}"] = k_[l], dk[l]
        out[f"p_gw{l}"] = sum(pc[l][t][0] for t in steps)
        out[f"p_gb{l}"] = sum(pc[l][t][1] for t in steps)
        out[f"p_hw{l}"] = sum(pc[l][t][2] for t in steps)
        out[f"p_hb{l}"] = sum(pc[l][t][3] for t in steps)
        for j in range(3):
            hr(f"params_wgrad{j}_{l}", pw_abs[j][l], pw_gam[j][l])
            if j < 2:
                hr(f"params_bias{j}_{l}", pb_abs[j][l], pb_gam[j][l])
        if stats is not None:
            cc = comb_cin(case, l)
            cov["soa_hcols_late"][l] = any(bool((pc[l][t][2][:, cc:] != 0).any()) for t in range(1, T))
    tdh = [dhs[L - 1][t + 1] for t in range(T)]
    out["p_ghw"] = sum((us[:, t:t + 1] * top[t]).sum((0, 2, 3)) for t in steps).view(1, -1, 1, 1)
    out["p_ghb"] = sum(us[:, t].sum() for t in steps).view(1)
    out["p_hhw"] = sum((dus[:, t:t + 1] * top[t] + us[:, t:t + 1] * tdh[t]).sum((0, 2, 3)) for t in steps).view(1, -1, 1, 1)
    out["p_hhb"] = sum(dus[:, t].sum() for t in steps).view(1)
    hr("head_sums", sum((A(dus[:, t:t + 1] * top[t]) + A(us[:, t:t + 1] * tdh[t])).sum((0, 2, 3)) for t in range(T)),
       min(min(grid(dus) * grid(top[t]), grid(us) * grid(tdh[t])) for t in range(T)))
    if case["frames"] is not None:
        out["dframes"] = bank_scatter(case, dx)
        out["s_dframes"], out["s_ddframes"] = bank_scatter(case, sgx), bank_scatter(case, shx)
    return out


def bank_scatter(case, g):
    """the per-window gradient [B, T, C, H, W] added into the frames: frame starts[b] + t gets sample b's step t"""
    n = case["frames"].shape[0]
    out = g.new_zeros(n, *g.shape[2:])
    for b, s in enumerate(case["starts"].tolist()):
        for t in range(case["T"]):
            out[s + t] += g[b, t]
    return out


def comb_cin(case, l):
    return case["C"] if l == 0 else case["hidden"][l - 1]


# ------------------------------------------------------------------------------------------------ coverage
def _new_cov(stats, case):
    if "cov" not in stats:
        B, H, W, T, L = case["B"], case["H"], case["W"], case["T"], len(case["hidden"])
        stats["cov"] = dict(
            pix={p: torch.zeros(B, H, W, dtype=torch.bool) for p in PARTS},
            rows={p: [torch.zeros(T, 4, dtype=torch.bool) for _ in range(L)] for p in ("bwd", "soa")},
            taps={p: [torch.zeros(k, k, dtype=torch.bool) for k in case["ks"]] for p in ("bwd", "soa")},
            cols=[torch.zeros(comb_cin(case, l) + hc, dtype=torch.bool) for l, hc in enumerate(case["hidden"])],
            dh_steps=[[False] * T for _ in range(L)],
            bwd_hcols_late=[False] * L, soa_hcols_late=[False] * L)
    return stats["cov"]


PARTS = ("bwd", "a", "da")      # the ordinary backward's dgates; the primal and tangent halves of the 2B-image view


def _cover(cov, pas, l, t, dg, comb, w, k, hc, cin):
    nz = dg != 0
    if pas == "soa":
        n = nz.shape[0] // 2
        cov["pix"]["a"] |= nz[:n].any(1)
        cov["pix"]["da"] |= nz[n:].any(1)
    else:
        cov["pix"]["bwd"] |= nz.any(1)
    rows = nz.flatten(2).any(2).any(0)
    cov["rows"][pas][l][t] |= rows.view(4, hc).any(1)
    wg_cols = (comb != 0).flatten(2).any(2).any(0) & bool(rows.any())
    dg_cols = (w[rows] != 0).flatten(2).any(2).any(0) if bool(rows.any()) else torch.zeros(w.shape[1], dtype=torch.bool)
    cov["cols"][l] |= wg_cols | dg_cols
    cov["taps"][pas][l] |= _tap_hits(dg, w, k, forward=False)


def row_exceptions(case):
    """(pass, layer, gate row) that the construction cannot reach at two or more steps: the live o rows of dgates see
    dh only from the head (top layer, every step with dseq, else T-1) and from dh_T (every layer, T-1), because live
    weight columns are zero, so dgrad never reaches a live channel"""
    L = len(case["hidden"])
    ex = {("bwd", l, 3) for l in range(L - 1)}
    if not case["return_sequence"]:
        ex.add(("bwd", L - 1, 3))
    return ex


def summarize_coverage(case, cov) -> Dict[str, bool]:
    H, W = case["H"], case["W"]
    ty, tx = Lt.TILE_H * ((H - 1) // Lt.TILE_H), Lt.TILE_W * ((W - 1) // Lt.TILE_W)
    res = {}
    for p in PARTS:        # every edge of every part, the tangent half of the 2B view included
        pix = cov["pix"][p]
        res[f"{p}_corners"] = all(bool(pix[:, y, xx].any()) for y, xx in ((0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1)))
        res[f"{p}_last_tile_row"] = bool(pix[:, ty:].any())
        res[f"{p}_last_tile_col"] = bool(pix[:, :, tx:].any())
        res[f"{p}_every_image"] = bool(pix.flatten(1).any(1).all())
    res["every_tap"] = all(bool(t.all()) for p in cov["taps"].values() for t in p)
    # every gate row of every layer's dgates, and of its (a, da) together, at two or more steps, but the exceptions
    ex = row_exceptions(case)
    for p in ("bwd", "soa"):
        for l, r in enumerate(cov["rows"][p]):
            n = r.sum(0)
            res[f"{p}_rows_2_steps_layer{l}"] = all(int(n[q]) >= (1 if (p, l, q) in ex else 2) for q in range(4))
    res["dh_every_step"] = all(all(s) for s in cov["dh_steps"])
    res["dW_h_cols_from_t_ge_1"] = all(cov["bwd_hcols_late"])
    res["HvW_h_cols_from_t_ge_1"] = all(cov["soa_hcols_late"])
    ok = True
    for l, c in enumerate(cov["cols"]):
        ci = comb_cin(case, l)
        for lo, hi in ((0, ci), (ci, c.numel())):
            for s in range(lo, hi, Lt.CHUNK):
                ok &= bool(c[s:min(s + Lt.CHUNK, hi)].any())
    res["every_channel_chunk"] = ok
    return res


def headroom(stats) -> float:
    return max(stats["headroom"].values())


# ------------------------------------------------------------------------------------------------ the suite's cases
D_CASES = {
    # one layer, hidden 64, k 3, ragged in both directions, T = 3
    "h64_k3_19x21": dict(B=2, T=3, C=9, H=19, W=21, hidden=[64], ks=[3], return_sequence=True, ddensity=0.01,
                         tdensity=0.02),
    # two layers, a padded hidden size (40), k 5 / 3, frame-bank windows with repeated starts
    "h40_h16_k5_k3_17x13": dict(B=4, T=2, C=9, H=17, W=13, hidden=[40, 16], ks=[5, 3], return_sequence=True,
                                shared_frames=True, repeat_starts=True, ddensity=0.01, wdensity=0.04, tdensity=0.02),
    # wide dtop, u and dx entries: dgates, (a, da) and the tangent's dh round in both operand formats
    "h32_k3_wide_12x20": dict(B=2, T=2, C=9, H=12, W=20, hidden=[32], ks=[3], return_sequence=True, wide=True,
                              ddensity=0.01, tdensity=0.02),
    # the shipped geometry: hidden 64/32/16, k 5/3/3, 100 x 154 (layer-0 dgrad: K segments of 25 and 9 taps), pred
    # only (seeds at T-1), sparse saturated pixels.  T = 2: at T = 3 the c_{t-1} = 24 * 2^T factor of the saturated
    # channels takes the bias sum of (H v)_b past the 2^20 headroom
    "shipped_100x154_T2": dict(B=2, T=2, C=21, H=100, W=154, hidden=[64, 32, 16], ks=[5, 3, 3], wdensity=0.015,
                               ddensity=0.0005, xdensity=0.05, tdensity=0.003, sdensity=0.01),
}
LARGE = ("shipped_100x154_T2",)     # the CPU suite plants the defects into the first image of these


def d_case(name, precision):
    kw = dict(D_CASES[name])
    return case_d(kw.pop("B"), kw.pop("T"), kw.pop("C"), kw.pop("H"), kw.pop("W"), kw.pop("hidden"), kw.pop("ks"),
                  precision, **kw)


def suite_cases():
    return [(f"D-{p}-{n}", d_case(n, p)) for p in ("tf32", "bf16") for n in D_CASES]


def first_images(case, n):
    """the case cut to its first n images (same grid, weights and seeds)"""
    out = dict(case, B=n)
    for k in ("x", "dx", "dtop", "u", "du"):
        out[k] = case[k][:n]
    for k in ("h0", "c0", "dh0", "dc0", "dh_T", "dc_T"):
        out[k] = [t[:n] for t in case[k]]
    if case["frames"] is not None:
        out["starts"] = case["starts"][:n]
        m = int(out["starts"].max()) + case["T"]
        out["frames"], out["dframes"] = case["frames"][:m], case["dframes"][:m]
    return out
