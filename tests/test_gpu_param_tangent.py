"""GPU (B200): the parameter-space tangent -- ConvLSTM.jvp / jvp_windows with param_tangent, Plan.set_param_tangent /
clear_param_tangent, and forward_tangent with a parameter direction.

References: torch.func.jvp of the fp32 oracle (convlstm_forward_state) with the parameters as an argument, at the bars of
the parity tests (max|a-b| / max|b| <= 2e-2 in bf16, <= 1e-3 in tf32); the ordinary backward of the same forward for the
dot-product identity; and bit-for-bit identities wherever the arithmetic is the same (no or a zero direction against a
plan without the flag, linearity, directions in sequence, explicit vs frame-bank windows, a following backward)."""
import ctypes

import pytest
import torch

from oracle import convlstm_oracle as O
from oracle.state_oracle import convlstm_forward_state

pytestmark = pytest.mark.gpu

TOL = {"tf32": 1e-3, "bf16": 2e-2}
PRECISIONS = ["bf16", "tf32"]


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists)")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.deterministic = False


def _net(C, hidden, ks, precision, seed=0, return_sequence=True):
    """(net on the GPU, CPU copies of its parameters)"""
    from nasa_niswan_b200 import ConvLSTM
    torch.manual_seed(seed)
    net = ConvLSTM(C, hidden, ks, len(hidden), precision=precision, return_sequence=return_sequence)
    params = {k: v.detach().clone() for k, v in net.state_dict().items()}
    return net.cuda(), params


def _rand(g, *shape, scale=1.0):
    return torch.randn(*shape, generator=g) * scale


def _direction(params, g, keys=None):
    """a parameter direction scaled like each parameter (every key, or `keys`)"""
    return {k: _rand(g, *v.shape) * float(v.abs().mean()) for k, v in params.items() if keys is None or k in keys}


def _cuda(d):
    return {k: v.cuda() for k, v in d.items()}


def _cuda_pairs(pairs):
    return None if pairs is None else [(h.cuda(), c.cuda()) for h, c in pairs]


def _oracle_jvp(params, L, x, state, dx, dstate, dparams):
    """torch.func.jvp of the fp32 oracle over (params, x, h0, c0): tangents of (pred, seq, [h_T], [c_T])"""
    dparams = {k: dparams.get(k, torch.zeros_like(v)) for k, v in params.items()}

    def f(p, x, hs, cs):
        (pred, seq), final = convlstm_forward_state(x, p, L, list(zip(hs, cs)), return_sequence=True)
        return pred, seq, tuple(h for h, _ in final), tuple(c for _, c in final)
    primals = (params, x, tuple(h for h, _ in state), tuple(c for _, c in state))
    tangents = (dparams, dx, tuple(h for h, _ in dstate), tuple(c for _, c in dstate))
    with torch.no_grad():
        return torch.func.jvp(f, primals, tangents)[1]


# (B, T, C, H, W, hidden, ks, precisions): the tangent tests' list -- one layer on the 90x144 grid, ragged tiles with a
# padded hidden size and k = 5, the shipped three-layer model on its 100x154 halo grid, BASELINE cfg 2 at B = 32
CASES = {
    "one_layer_90x144": (2, 4, 7, 90, 144, [32], [3], PRECISIONS),
    "edge_h20_k5": (2, 4, 5, 18, 22, [20], [5], PRECISIONS),
    "edge_two_layers_padded": (3, 3, 5, 20, 26, [20, 48], [5, 3], PRECISIONS),
    "shipped_3layer": (2, 6, 5, 100, 154, [64, 32, 16], [5, 3, 3], PRECISIONS),
    "cfg2": (32, 12, 21, 90, 144, [64], [3], ["bf16"]),
}


@pytest.mark.parametrize("joint", [False, True], ids=["params_only", "joint_with_input_and_state"])
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", list(CASES))
def test_param_tangent_matches_the_oracle_jvp(name, precision, joint):
    """dpred, dseq, dh_T and dc_T of J (dtheta) and of J (dx, dh0, dc0, dtheta) against torch.func.jvp"""
    B, T, C, H, W, hidden, ks, precisions = CASES[name]
    if precision not in precisions:
        pytest.skip(f"{name} runs in {precisions} only")
    net, params = _net(C, hidden, ks, precision)
    g = torch.Generator().manual_seed(41)
    x = _rand(g, B, T, C, H, W)
    dtheta = _direction(params, g)
    zero = [(torch.zeros(B, hc, H, W), torch.zeros(B, hc, H, W)) for hc in hidden]
    if joint:
        dx = _rand(g, B, T, C, H, W)
        state = [(_rand(g, B, hc, H, W, scale=0.5), _rand(g, B, hc, H, W, scale=0.5)) for hc in hidden]
        dstate = [(_rand(g, B, hc, H, W), _rand(g, B, hc, H, W)) for hc in hidden]
    else:
        dx, state, dstate = torch.zeros_like(x), zero, zero
    ref = _oracle_jvp(params, len(hidden), x, state, dx, dstate, dtheta)
    (_, _), ((dpred, dseq), dfinal) = net.jvp(
        x.cuda(), dx.cuda() if joint else None, hidden_state=_cuda_pairs(state) if joint else None,
        state_tangent=_cuda_pairs(dstate) if joint else None, return_state=True, param_tangent=_cuda(dtheta))
    errs = {"dpred": O.max_abs_normalised(dpred.cpu(), ref[0]), "dseq": O.max_abs_normalised(dseq.cpu(), ref[1])}
    for l, (dh, dc) in enumerate(dfinal):
        errs[f"dh_T[{l}]"] = O.max_abs_normalised(dh.cpu(), ref[2][l])
        errs[f"dc_T[{l}]"] = O.max_abs_normalised(dc.cpu(), ref[3][l])
    print(f"{name} {precision} joint={joint}: worst {max(errs.values()):.2e}")
    bad = {k: e for k, e in errs.items() if not e < TOL[precision]}
    assert not bad, bad


def _plan(net, B, T, H, W, C, hidden, ks, precision, **flags):
    from nasa_niswan_b200.engine import Plan
    plan = Plan(B, T, H, W, C, hidden, ks, precision=precision, training=True, return_sequence=True, **flags)
    for l, cell in enumerate(net.layers):
        plan.set_weights(l, cell.conv.weight, cell.conv.bias)
    plan.set_head(net.conv.weight, net.conv.bias)
    return plan


def _launches():
    from nasa_niswan_b200 import _lib
    return _lib.load().nint_launch_count(-1)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_no_or_zero_direction_equals_the_tangent_plan_bitwise(precision):
    """a param_tangent plan without a direction issues the tangent plan's launches and gives its outputs bit for bit; a
    zero direction gives the same outputs"""
    B, T, C, H, W, hidden, ks = 2, 4, 5, 20, 24, [32, 16], [5, 3]
    net, params = _net(C, hidden, ks, precision)
    g = torch.Generator().manual_seed(3)
    r = lambda *s: _rand(g, *s).cuda()
    x, dx = r(B, T, C, H, W), r(B, T, C, H, W)
    dh0 = [r(B, hc, H, W) for hc in hidden]
    ref_plan = _plan(net, B, T, H, W, C, hidden, ks, precision, tangent=True)
    ref_plan.forward(x)
    n0 = _launches()
    ref = ref_plan.forward_tangent(dx, dh0)
    n_ref = _launches() - n0
    plan = _plan(net, B, T, H, W, C, hidden, ks, precision, param_tangent=True)
    plan.forward(x)
    n0 = _launches()
    got = plan.forward_tangent(dx, dh0)
    assert _launches() - n0 == n_ref
    zero = {k: torch.zeros_like(v).cuda() for k, v in params.items()}
    plan.set_param_tangent(*net.param_direction(zero))
    got0 = plan.forward_tangent(dx, dh0)
    for a in (got, got0):
        assert torch.equal(a[0], ref[0]) and torch.equal(a[1], ref[1])
        assert all(torch.equal(p, q) and torch.equal(s, t) for (p, s), (q, t) in zip(a[2], ref[2]))
    plan.clear_param_tangent()
    n0 = _launches()
    plan.forward_tangent(dx, dh0)
    assert _launches() - n0 == n_ref


@pytest.mark.parametrize("precision", PRECISIONS)
def test_exact_linearity(precision):
    """J (2 v) = 2 J v bit for bit for a joint direction (doubling is exact through every rounding)"""
    B, T, C, H, W, hidden, ks = 2, 4, 5, 20, 24, [32, 16], [3, 5]
    net, params = _net(C, hidden, ks, precision)
    g = torch.Generator().manual_seed(4)
    x, dx = _rand(g, B, T, C, H, W).cuda(), _rand(g, B, T, C, H, W).cuda()
    d = _cuda(_direction(params, g))
    _, dout = net.jvp(x, dx, param_tangent=d)
    _, dout2 = net.jvp(x, 2 * dx, param_tangent={k: 2 * v for k, v in d.items()})
    assert torch.equal(dout2[0], 2 * dout[0]) and torch.equal(dout2[1], 2 * dout[1])


@pytest.mark.parametrize("precision", PRECISIONS)
def test_dot_product_identity_with_the_parameter_gradients(precision):
    """<u, J_theta v> from the tangent pass against <J_theta^T u, v> from the ordinary backward of the same forward,
    with u = J_theta v itself (no cancellation in the sum)"""
    B, T, C, H, W, hidden, ks = 2, 5, 5, 20, 26, [32, 16], [3, 5]
    net, params = _net(C, hidden, ks, precision)
    g = torch.Generator().manual_seed(8)
    x = _rand(g, B, T, C, H, W).cuda()
    d = _cuda(_direction(params, g))
    _, (dpred, dseq) = net.jvp(x, None, param_tangent=d)
    net.zero_grad()
    pred, seq = net(x)
    (pred * dpred).sum().add_((seq * dseq).sum()).backward()
    dot = lambda a, b: sum(float((p.double() * q.double()).sum()) for p, q in zip(a, b))
    lhs = dot([dpred, dseq], [dpred, dseq])
    rhs = dot([p.grad for _, p in net.named_parameters()], [d[n] for n, _ in net.named_parameters()])
    print(f"dot product {precision}: {lhs:.6e} vs {rhs:.6e}")
    assert abs(lhs - rhs) <= TOL[precision] * max(abs(lhs), abs(rhs))


@pytest.mark.parametrize("precision", PRECISIONS)
def test_two_directions_on_one_forward_equal_separate_calls(precision):
    B, T, C, H, W, hidden, ks = 2, 4, 5, 20, 24, [32, 16], [3, 5]
    net, params = _net(C, hidden, ks, precision)
    g = torch.Generator().manual_seed(6)
    x, dx = _rand(g, B, T, C, H, W).cuda(), _rand(g, B, T, C, H, W).cuda()
    d1 = net.param_direction(_cuda(_direction(params, g)))
    d2 = net.param_direction(_cuda(_direction(params, g, keys={"layers.1.conv.bias", "conv.weight"})))
    plan = _plan(net, B, T, H, W, C, hidden, ks, precision, param_tangent=True)
    plan.forward(x)
    plan.set_param_tangent(*d1)
    a1 = plan.forward_tangent(dx)
    plan.set_param_tangent(*d2)
    a2 = plan.forward_tangent(None)
    for d, a, ddx in ((d2, a2, None), (d1, a1, dx)):
        plan.forward(x)
        plan.set_param_tangent(*d)
        b = plan.forward_tangent(ddx)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        assert all(torch.equal(p, q) and torch.equal(s, t) for (p, s), (q, t) in zip(a[2], b[2]))


@pytest.mark.parametrize("precision", PRECISIONS)
def test_backward_after_parameter_tangents_is_bitwise_unchanged(precision):
    """deterministic plan: a backward that follows two tangent passes with parameter directions equals the backward of a
    forward without them"""
    B, T, C, H, W, hidden, ks = 2, 5, 5, 20, 24, [32, 16], [3, 5]
    net, params = _net(C, hidden, ks, precision)
    plan = _plan(net, B, T, H, W, C, hidden, ks, precision, deterministic=True, param_tangent=True)
    g = torch.Generator().manual_seed(5)
    x, dseq = _rand(g, B, T, C, H, W).cuda(), _rand(g, B, T, H, W).cuda()
    d = net.param_direction(_cuda(_direction(params, g)))

    def step(tangents):
        plan.forward(x)
        for _ in range(tangents):
            plan.set_param_tangent(*d)
            plan.forward_tangent(None)
        return plan.backward(None, dseq)
    ref = step(0)
    got = step(2)
    for a, b in zip(ref[:2], got[:2]):
        assert all(torch.equal(p, q) for p, q in zip(a, b))
    assert torch.equal(ref[2], got[2]) and torch.equal(ref[3], got[3])


@pytest.mark.parametrize("precision", PRECISIONS)
def test_frame_bank_windows_equal_explicit_windows_bitwise(precision):
    from nasa_niswan_b200.preprocess import FrameBank
    T, C, H, W, N, hidden, ks = 4, 5, 20, 24, 9, [32, 16], [5, 3]
    net, params = _net(C, hidden, ks, precision)
    g = torch.Generator().manual_seed(10)
    record, drecord = _rand(g, N, C, H, W).cuda(), _rand(g, N, C, H, W).cuda()
    if precision == "bf16":     # the bank holds bf16 frames: explicit windows of the same values
        record, drecord = record.bfloat16().float(), drecord.bfloat16().float()
    bank = FrameBank.from_frames(record, precision)
    dbank = bank.tangent(drecord)
    starts = torch.tensor([3, 0, 3, 5])
    state = _cuda_pairs([(_rand(g, 4, hc, H, W), _rand(g, 4, hc, H, W)) for hc in hidden])
    d = _cuda(_direction(params, g))
    win = lambda r: torch.stack([r[s:s + T] for s in starts.tolist()])
    a = net.jvp_windows(bank, starts, T, dbank, hidden_state=state, return_state=True, param_tangent=d)
    b = net.jvp(win(record), win(drecord), hidden_state=state, return_state=True, param_tangent=d)
    (da, dsa), dfa = a[1]
    (db, dsb), dfb = b[1]
    assert torch.equal(da, db) and torch.equal(dsa, dsb)
    assert all(torch.equal(p, q) and torch.equal(s, t) for (p, s), (q, t) in zip(dfa, dfb))


def test_refusals():
    from nasa_niswan_b200.engine import Plan
    B, T, C, H, W, hidden = 2, 3, 5, 12, 16, [16]
    net, params = _net(C, hidden, [3], "bf16")
    x = torch.randn(B, T, C, H, W, device="cuda")
    d = net.param_direction(_cuda(_direction(params, torch.Generator().manual_seed(1))))
    tp = _plan(net, B, T, H, W, C, hidden, [3], "bf16", tangent=True)          # no NINT_FLAG_PARAM_TANGENT
    with pytest.raises(RuntimeError, match="NINT_FLAG_PARAM_TANGENT"):
        tp.set_param_tangent(*d)
    with pytest.raises(RuntimeError, match="NINT_FLAG_PARAM_TANGENT"):
        tp.clear_param_tangent()
    inf = Plan(B, T, H, W, C, hidden, [3], training=False, param_tangent=True)
    with pytest.raises(RuntimeError, match="training plan"):
        inf.set_param_tangent(*d)
    pp = _plan(net, B, T, H, W, C, hidden, [3], "bf16", param_tangent=True)
    with pytest.raises(RuntimeError, match="null weight"):
        from nasa_niswan_b200 import _lib
        _lib.check(pp.lib.nint_plan_set_weight_tangent(pp._h, 0, None, None, pp._stream()), "set_weight_tangent")
    with pytest.raises(ValueError, match="shape"):
        pp.set_param_tangent([(torch.zeros(3, 3, device="cuda"), None)])
    with pytest.raises(KeyError, match="unknown"):
        net.param_direction({"layers.0.weight": torch.zeros(1)})
    with pytest.raises(ValueError, match="shape"):
        net.param_direction({"conv.bias": torch.zeros(2, device="cuda")})
    # a direction set or cleared after the tangent pass makes the second-order pass refuse until the tangent pass runs
    sp = _plan(net, B, T, H, W, C, hidden, [3], "bf16", second_order=True, param_tangent=True)
    u = torch.randn(B, 1, H, W, device="cuda")
    sp.forward(x)
    sp.set_param_tangent(*d)
    sp.forward_tangent(torch.randn_like(x))
    sp.backward_second_order(u, u)
    sp.clear_param_tangent()
    with pytest.raises(RuntimeError, match="before nint_forward_tangent"):
        sp.backward_second_order(u, u)
    sp.forward_tangent(torch.randn_like(x))
    sp.backward_second_order(u, u)
    torch.cuda.synchronize()
