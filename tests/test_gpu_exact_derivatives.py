"""GPU (B200): bit-exact checks of carried state, the tangent pass, the second-order pass and the params call on the
stateful integer-lattice cases (oracle/lattice_derivatives.py, case D).

test_lattice_derivatives_cpu.py proves on the CPU that every sum of these cases is exact in fp32 whatever the order,
so every asserted tensor must equal the fp64 reference with torch.equal.  Everything runs through Plan:
  - stateful forward and BPTT with dh_T / dc_T seeds (deterministic and atomic, NINT_FUSE_STEPS 0 and 3);
  - the tangent pass with input, state and parameter directions, alone and jointly, explicit and frame-bank windows;
  - the second-order pass and the params call (grad=True and grad=False), two directions on one forward;
  - an ordinary backward of the same forward after the derivative passes;
  - every derivative plan layout: tangent / param_tangent plans (the tangent's dh in a two-slot ring), second_order
    plans ((a, da) of one step), and plans with both flags (every step kept for the params call);
  - the params call after the caller dropped the tangent frames of a frame-bank tangent pass."""
import functools

import pytest
import torch

from oracle import lattice_derivatives as D

pytestmark = pytest.mark.gpu

CASES = dict(D.suite_cases())


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists)")


@functools.lru_cache(maxsize=None)
def _ref(cid, which="joint"):
    return D.reference(D.with_direction(CASES[cid], which))


def _cu(t):
    return t.float().cuda()


def _assert_exact(got, ref, tag=""):
    for k, v in got.items():
        assert torch.equal(v.detach().cpu().double(), ref[k]), f"{tag} {k}: {int((v.detach().cpu().double() != ref[k]).sum())} " \
                                                               f"elements differ, max |diff| {float((v.detach().cpu().double() - ref[k]).abs().max()):.3e}"


# the derivative flag sets: each keeps the tangent's dh and the second-order (a, da) in a different layout -- only
# second_order + param_tangent keeps every step (the history the params call reads); tangent and param_tangent alone
# keep dh in a two-slot ring, second_order alone keeps (a, da) of one step as one 2B-image buffer
FLAGS = {"tangent": dict(tangent=True), "param_tangent": dict(param_tangent=True),
         "second_order": dict(second_order=True), "both": dict(second_order=True, param_tangent=True), "none": {}}


def _plan(case, deterministic, derivatives=True, flags="both"):
    from nasa_niswan_b200 import Plan
    L = len(case["hidden"])
    plan = Plan(case["B"], case["T"], case["H"], case["W"], case["C"], case["hidden"], case["ks"],
                precision=case["precision"], training=True, return_sequence=case["return_sequence"],
                deterministic=deterministic, input_grad=True, state_grad=True,
                **FLAGS[flags if derivatives else "none"])
    for l in range(L):
        plan.set_weights(l, _cu(case["ws"][l]), _cu(case["bs"][l]))
    plan.set_head(_cu(case["hw"]), _cu(case["hb"]))
    return plan


def _forward(plan, case, bank):
    """the forward from the case's initial state; returns (outputs, frame bank or None)"""
    L = len(case["hidden"])
    state = [(_cu(case["h0"][l]), _cu(case["c0"][l])) for l in range(L)]
    fb = None
    if bank:
        from nasa_niswan_b200.preprocess import FrameBank
        fb = FrameBank.from_frames(_cu(case["frames"]), case["precision"])
        pred, seq = plan.forward_bank(fb.frames, case["starts"].to(torch.int32).cuda(), state)
    else:
        pred, seq = plan.forward(_cu(case["x"]), state)
    out = {"pred": pred}
    if seq is not None:
        out["seq"] = seq
    for l, (h, c) in enumerate(plan.final_state()):
        out[f"hT{l}"], out[f"cT{l}"] = h, c
    return out, fb


def _seed(case, key):
    s = _cu(case[key])
    return (None, s) if case["return_sequence"] else s[:, -1:].contiguous()


def _derivatives(plan, case, fb, grad=True, keep_tangent=True):
    """tangent pass, then (on second-order plans) the second-order pass, then (on plans with both flags) the params
    call, for the case's direction.  keep_tangent=False: drop the tangent frames after the tangent pass and fill a new
    tensor of the same size, so that the params call reads garbage unless the plan keeps them"""
    L = len(case["hidden"])
    if plan.param_tangent:
        plan.set_param_tangent([(_cu(case["dws"][l]), _cu(case["dbs"][l])) for l in range(L)],
                               (_cu(case["dhw"]), _cu(case["dhb"])))
    dh0 = [_cu(t) for t in case["dh0"]]
    dc0 = [_cu(t) for t in case["dc0"]]
    if fb is not None:
        tpred, tseq, tfin = plan.forward_tangent_bank(fb.tangent(_cu(case["dframes"])), dh0, dc0)
    else:
        tpred, tseq, tfin = plan.forward_tangent(_cu(case["dx"]), dh0, dc0)
    out = {"t_pred": tpred}
    if tseq is not None:
        out["t_seq"] = tseq
    for l, (h, c) in enumerate(tfin):
        out[f"t_hT{l}"], out[f"t_cT{l}"] = h, c
    if not keep_tangent:
        garbage = torch.full_like(fb.frames, 3.0)      # the caching allocator hands out the freed block again
    if not plan.second_order:
        return out
    u, du = _seed(case, "u"), _seed(case, "du")
    if fb is not None:
        shape = (case["frames"].shape[0], case["C"], case["H"], case["W"])
        dfr = torch.zeros(shape, device="cuda")
        ddfr = torch.zeros(shape, device="cuda")
        st, dst = plan.backward_second_order_bank(u, du, dfr, ddfr, state=True)
        out["s_dframes"], out["s_ddframes"] = dfr, ddfr
    else:
        dx, ddx, st, dst = plan.backward_second_order(u, du, state=True)
        out["s_dx"], out["s_ddx"] = dx, ddx
    for l in range(L):
        out[f"s_dh0_{l}"], out[f"s_dc0_{l}"] = st[l]
        out[f"s_ddh0_{l}"], out[f"s_ddc0_{l}"] = dst[l]
    if not plan.param_tangent:
        return out
    g, h = plan.backward_second_order_params(grad=grad)
    for l in range(L):
        if grad:
            out[f"p_gw{l}"], out[f"p_gb{l}"] = g[2 * l], g[2 * l + 1]
        out[f"p_hw{l}"], out[f"p_hb{l}"] = h[2 * l], h[2 * l + 1]
    if grad:
        out["p_ghw"], out["p_ghb"] = g[-2], g[-1]
    out["p_hhw"], out["p_hhb"] = h[-2], h[-1]
    return out


def _backward(plan, case, fb):
    L = len(case["hidden"])
    dtop = _cu(case["dtop"])
    dpred, dseq = (None, dtop) if case["return_sequence"] else (dtop[:, -1:].contiguous(), None)
    gw, gb, ghw, ghb = plan.backward(dpred, dseq, dh_T=[_cu(t) for t in case["dh_T"]],
                                     dc_T=[_cu(t) for t in case["dc_T"]])
    out = {"ghw": ghw, "ghb": ghb}
    dh0, dc0 = plan.backward_initial_state()
    for l in range(L):
        out[f"gw{l}"], out[f"gb{l}"] = gw[l], gb[l]
        out[f"dh0_{l}"], out[f"dc0_{l}"] = dh0[l], dc0[l]
    if fb is not None:
        dfr = torch.zeros((case["frames"].shape[0], case["C"], case["H"], case["W"]), device="cuda")
        plan.backward_input_bank(dfr)
        out["dframes"] = dfr
    else:
        out["dx"] = plan.backward_input()
    return out


def _bank(cid):
    return CASES[cid]["frames"] is not None


@pytest.mark.parametrize("cid", list(CASES))
def test_every_pass_is_exact(cid):
    """one forward: the joint direction (grad=True), then the input direction alone (grad=False), each against its own
    reference, then the ordinary backward of the same forward; deterministic plan"""
    case, bank = CASES[cid], _bank(cid)
    plan = _plan(case, deterministic=True)
    out, fb = _forward(plan, case, bank)
    _assert_exact(out, _ref(cid), "forward")
    _assert_exact(_derivatives(plan, D.with_direction(case, "joint"), fb), _ref(cid), "joint")
    _assert_exact(_derivatives(plan, D.with_direction(case, "input"), fb, grad=False), _ref(cid, "input"), "input")
    plan.clear_param_tangent()
    _assert_exact(_backward(plan, case, fb), _ref(cid), "backward")
    torch.cuda.synchronize()


@pytest.mark.parametrize("flags", ["tangent", "param_tangent", "second_order"])
@pytest.mark.parametrize("cid", [c for c in CASES if "shipped" not in c])
def test_every_plan_layout_is_exact(cid, flags):
    """the flag sets without the full history: the tangent's dh in a two-slot ring, (a, da) of one step as one 2B-image
    buffer; two directions on one forward, then the ordinary backward.  Plans without param_tangent take the input and
    state directions (their tangent pass runs at fixed parameters)"""
    case, bank = CASES[cid], _bank(cid)
    plan = _plan(case, deterministic=True, flags=flags)
    out, fb = _forward(plan, case, bank)
    _assert_exact(out, _ref(cid), "forward")
    first = "joint" if flags == "param_tangent" else "input_state"
    for which in (first, "state"):
        _assert_exact(_derivatives(plan, D.with_direction(case, which), fb), _ref(cid, which), f"{flags} {which}")
    _assert_exact(_backward(plan, case, fb), _ref(cid), "backward")


@pytest.mark.parametrize("cid", [c for c in CASES if _bank(c)])
def test_the_plan_keeps_the_tangent_frames(cid):
    """the params call reads the bank's tangent frames again: dropping them after the tangent pass must not matter"""
    case = CASES[cid]
    plan = _plan(case, deterministic=True)
    _, fb = _forward(plan, case, True)
    _assert_exact(_derivatives(plan, D.with_direction(case, "joint"), fb, keep_tangent=False), _ref(cid), "joint")


@pytest.mark.parametrize("which", ["state", "param"])
@pytest.mark.parametrize("cid", [c for c in CASES if "h64" in c or "h40" in c])
def test_single_directions_are_exact(cid, which):
    """the state and parameter directions alone, on an atomic plan"""
    case, bank = CASES[cid], _bank(cid)
    plan = _plan(case, deterministic=False)
    _, fb = _forward(plan, case, bank)
    _assert_exact(_derivatives(plan, D.with_direction(case, which), fb), _ref(cid, which), which)


@pytest.mark.parametrize("det", [True, False], ids=["deterministic", "atomic"])
@pytest.mark.parametrize("fuse", ["0", "3"], ids=["per_step", "fused"])
@pytest.mark.parametrize("cid", list(CASES))
def test_stateful_bptt_is_exact(monkeypatch, cid, fuse, det):
    """forward from the initial state and backward with dh_T / dc_T on a plan without the derivative flags, with one
    launch per step (NINT_FUSE_STEPS=0) and with time-fused launches (NINT_FUSE_STEPS=3)"""
    monkeypatch.setenv("NINT_FUSE_STEPS", fuse)
    case, bank = CASES[cid], _bank(cid)
    plan = _plan(case, deterministic=det, derivatives=False)
    out, fb = _forward(plan, case, bank)
    _assert_exact(out, _ref(cid), "forward")
    _assert_exact(_backward(plan, case, fb), _ref(cid), "backward")
