"""CPU: the stateful lattice cases of test_gpu_exact_derivatives.py are exact by construction (no GPU, no libnint.so).

For every case: the fp64 reference of every pass (stateful forward and BPTT, tangent pass, second-order pass, params
call) equals the same reference evaluated in fp32 with the pixels and time steps of every sum in another order; every
sum stays within 2^20 grid steps; nonzero terms reach the corners, the last ragged tile row and column, every tap,
channel chunk and image, both image halves of the (a, da) view, every gate row at two or more steps, the h columns of
dW and (Hv)_W from steps t >= 1 and dh of the tangent at every step; every planted defect changes an asserted output;
and with the roundings switched off the reference equals the torch.func-validated fp64 restatements."""
import functools

import pytest
import torch

from oracle import lattice as Lt
from oracle import lattice_derivatives as D
from oracle.hvp_oracle import hvp_restatement
from oracle.param_hvp_oracle import param_hvp_restatement
from oracle.param_tangent_oracle import jvp_restatement
from oracle.state_oracle import convlstm_forward_state

CASES = dict(D.suite_cases())
LARGE = [c for c in CASES if c.split("-", 2)[2] in D.LARGE]


@functools.lru_cache(maxsize=None)
def _ref(cid):
    stats = {}
    return D.reference(CASES[cid], stats=stats), stats


@pytest.mark.parametrize("cid", list(CASES))
def test_fp32_in_another_order_equals_fp64(cid):
    ref = _ref(cid)[0]
    for order in ((1,) if cid in LARGE else (1, 2)):     # one evaluation of a large case takes seconds
        got = D.reference(CASES[cid], torch.float32, order=order)
        for k in ref:
            assert torch.equal(got[k].double(), ref[k]), (k, order)


@pytest.mark.parametrize("cid", list(CASES))
def test_headroom(cid):
    hr = _ref(cid)[1]["headroom"]
    worst = max(hr, key=hr.get)
    assert hr[worst] <= 2.0 ** Lt.HEADROOM_BITS, (worst, hr[worst])


@pytest.mark.parametrize("cid", list(CASES))
def test_coverage_and_non_vacuous_outputs(cid):
    ref, stats = _ref(cid)
    cov = D.summarize_coverage(CASES[cid], stats["cov"])
    assert all(cov.values()), [k for k, v in cov.items() if not v]
    assert not [k for k, v in ref.items() if not bool((v != 0).any())]


@pytest.mark.parametrize("cid", list(CASES))
def test_construction_sits_on_the_exact_points(cid):
    """pre-activations equal the bias at every step; live channels sit at |c_t| >= 24, h_t = +-1/2 (live F channels only
    where they saturate, c = h = 0 elsewhere); silent channels at c = h = 0"""
    case = CASES[cid]
    stats = _ref(cid)[1]
    for l, pre in stats["pre"]:
        assert bool((pre == 0).all()), l
    for (l, c), (_, h) in zip(stats["c"], stats["h"]):
        m = D._modes(case["hidden"][l]).view(1, -1, 1, 1).expand_as(c)
        sat = (m == 2) | ((m == 1) & (case["c0"][l] != 0))
        assert bool((c[sat].abs() >= D.SATURATE).all()) and bool((h[sat].abs() == 0.5).all()), l
        assert bool((c[(m == 1) & ~sat] == 0).all()) and bool((h[(m == 1) & ~sat] == 0).all()), l
        assert bool((c[m == 0] == 0).all()) and bool((h[m == 0] == 0).all()), l


@pytest.mark.parametrize("cid", [c for c in CASES if CASES[c]["wide"]])
def test_the_wide_case_rounds(cid):
    """the operand roundings of every pass are exercised, not only emulated: the ordinary backward's dgates (and in tf32
    its bias residuals), the tangent's dh and the second-order (a, da)"""
    ref, raw = _ref(cid)[0], D.reference(CASES[cid], rounding=False)
    for keys in (("gw0", "dx"), ("t_seq",), ("s_dx", "s_ddx", "p_hw0")):
        assert any(not torch.equal(ref[k], raw[k]) for k in keys), keys
    if CASES[cid]["precision"] == "tf32":       # the residuals put the unrounded dgates back into the bias gradient
        assert torch.equal(ref["gb0"], raw["gb0"]) and not torch.equal(ref["p_gb0"], raw["p_gb0"])


@pytest.mark.parametrize("cid", list(CASES))
def test_planted_defects_change_the_exact_result(cid):
    case = CASES[cid]
    if cid in LARGE:        # planted into the first image: same grid, tiles, halos and weights
        case = D.first_images(case, 1)
        ref = D.reference(case)
    else:
        ref = _ref(cid)[0]
    for d in D.DEFECTS:
        bad = D.reference(case, defect=d)
        assert any(not torch.equal(bad[k], ref[k]) for k in ref), f"{d} leaves every asserted output unchanged"


def test_every_defect_is_planted_somewhere():
    assert set(D.DEFECTS) == {"tangent_recurrent_slot", "tangent_t0_drops_h0", "dw_ifo_not_halved",
                              "params_reads_a_for_da", "soa_recurrent_slot", "dh_T_not_joined", "dc0_one_step_early",
                              "params_drop_ragged_tile", "params_drop_splitk_share"}


def _params(case):
    p, d = {}, {}
    for l in range(len(case["hidden"])):
        p[f"layers.{l}.conv.weight"], p[f"layers.{l}.conv.bias"] = case["ws"][l], case["bs"][l]
        d[f"layers.{l}.conv.weight"], d[f"layers.{l}.conv.bias"] = case["dws"][l], case["dbs"][l]
    p["conv.weight"], p["conv.bias"], d["conv.weight"], d["conv.bias"] = case["hw"], case["hb"], case["dhw"], case["dhb"]
    return p, d


@pytest.mark.parametrize("cid", [c for c in CASES if c.startswith("D-bf16")])
def test_unrounded_reference_equals_the_restatements(cid):
    """with no rounding the lattice reference is the fp64 restatements of f5-f9: the loss <u, out> + (s/2)|out - out*|^2
    (out* the case's own output, s = 1/2) has gradient u and Hessian-vector product s * dout there, and the ordinary
    backward with dtop = u and no final-state seeds is its gradient.  Large cases: their first image"""
    case = D.first_images(CASES[cid], 1) if cid in LARGE else dict(CASES[cid])
    L, T, s, rs = len(case["hidden"]), case["T"], 0.5, case["return_sequence"]
    params, dparams = _params(case)
    state = list(zip(case["h0"], case["c0"]))
    dstate = list(zip(case["dh0"], case["dc0"]))
    (out, fin), (dout, dfin) = jvp_restatement(case["x"], params, L, state, case["dx"], dstate, dparams, rs)
    o, do = (out[1], dout[1]) if rs else (out, dout)
    u = case["u"] if rs else case["u"][:, T - 1:]
    du = s * do
    dus = du if rs else torch.cat([torch.zeros_like(case["u"][:, :T - 1]), du], 1)
    case.update(dtop=case["u"], du=dus, dh_T=[torch.zeros_like(h) for h in case["h0"]],
                dc_T=[torch.zeros_like(c) for c in case["c0"]])
    ref = D.reference(case, rounding=False)
    close = lambda a, b, k: torch.testing.assert_close(a, b, rtol=0, atol=1e-12 * max(1.0, float(b.abs().max())),
                                                       msg=lambda m: f"{k}: {m}")
    close(ref["seq" if rs else "pred"], o, "out")
    close(ref["t_seq" if rs else "t_pred"], do, "t_out")
    fout, ffin = convlstm_forward_state(case["x"], params, L, state, rs)
    close(ref["seq" if rs else "pred"], fout[1] if rs else fout, "state_oracle out")
    for l in range(L):
        close(ref[f"hT{l}"], fin[l][0], f"hT{l}")
        close(ref[f"cT{l}"], fin[l][1], f"cT{l}")
        close(ref[f"hT{l}"], ffin[l][0], f"state_oracle hT{l}")
        close(ref[f"cT{l}"], ffin[l][1], f"state_oracle cT{l}")
        close(ref[f"t_hT{l}"], dfin[l][0], f"t_hT{l}")
        close(ref[f"t_cT{l}"], dfin[l][1], f"t_cT{l}")
    pick = (lambda q: q[1]) if rs else (lambda q: q)
    loss = lambda q: (u * pick(q)).sum() + 0.5 * s * ((pick(q) - o) ** 2).sum()
    _, (gx, gst, gp), (hx, hst, hp) = param_hvp_restatement(case["x"], params, L, loss, state, case["dx"], dstate,
                                                            dparams, return_sequence=rs)
    close(ref["s_dx"], gx, "s_dx")
    close(ref["s_ddx"], hx, "s_ddx")
    close(ref["dx"], gx, "dx")
    for l in range(L):
        for k, v in ((f"s_dh0_{l}", gst[l][0]), (f"s_dc0_{l}", gst[l][1]), (f"s_ddh0_{l}", hst[l][0]),
                     (f"s_ddc0_{l}", hst[l][1]), (f"dh0_{l}", gst[l][0]), (f"dc0_{l}", gst[l][1]),
                     (f"p_gw{l}", gp[f"layers.{l}.conv.weight"]), (f"p_gb{l}", gp[f"layers.{l}.conv.bias"]),
                     (f"gw{l}", gp[f"layers.{l}.conv.weight"]), (f"gb{l}", gp[f"layers.{l}.conv.bias"]),
                     (f"p_hw{l}", hp[f"layers.{l}.conv.weight"]), (f"p_hb{l}", hp[f"layers.{l}.conv.bias"])):
            close(ref[k], v, k)
    for k, n in (("p_ghw", "conv.weight"), ("p_ghb", "conv.bias"), ("ghw", "conv.weight"), ("ghb", "conv.bias")):
        close(ref[k], gp[n], k)
    close(ref["p_hhw"], hp["conv.weight"], "p_hhw")
    close(ref["p_hhb"], hp["conv.bias"], "p_hhb")
    # at fixed parameters: hvp_restatement (f8), with the input and state directions only
    fixed = D.with_direction(case, "input")
    fixed.update(dh0=case["dh0"], dc0=case["dc0"])
    (_, _), (dout0, _) = jvp_restatement(case["x"], params, L, state, case["dx"], dstate, None, rs)
    d0 = dout0[1] if rs else dout0
    fixed["du"] = s * d0 if rs else torch.cat([torch.zeros_like(case["u"][:, :T - 1]), s * d0], 1)
    ref0 = D.reference(fixed, rounding=False)
    _, (gx0, gst0), (hx0, hst0) = hvp_restatement(case["x"], params, L, loss, state, case["dx"], dstate, rs)
    close(ref0["s_dx"], gx0, "f8 s_dx")
    close(ref0["s_ddx"], hx0, "f8 s_ddx")
    for l in range(L):
        close(ref0[f"s_ddh0_{l}"], hst0[l][0], f"f8 s_ddh0_{l}")
        close(ref0[f"s_ddc0_{l}"], hst0[l][1], f"f8 s_ddc0_{l}")
