"""GPU (B200): Hessian-vector products over the parameters jointly with the inputs and the initial state --
ConvLSTM.hvp / hvp_windows(param_direction=, wrt_params=), Plan.backward_second_order_params.

References: torch.func.jvp(torch.func.grad(L o f)) of the fp32 reference loop over (theta, x, h0, c0) at the bars of the
parity tests (max|a-b| / max|b| <= 2e-2 in bf16, <= 1e-3 in tf32), with L1 differentiated on the piece of the device's
own prediction as tests/test_gpu_hvp.py does (the same loss, gradient and curvature there); the ordinary backward for
the gradient; bit-for-bit identities on deterministic plans."""
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


def _net(C, hidden, ks, precision, seed=0):
    from nasa_niswan_b200 import ConvLSTM
    torch.manual_seed(seed)
    net = ConvLSTM(C, hidden, ks, len(hidden), precision=precision, return_sequence=True).cuda()
    return net, {k: v.detach().clone() for k, v in net.state_dict().items()}


def _inputs(B, T, C, H, W, hidden, params, seed=41):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s, scale=1.0: (torch.randn(*s, generator=g) * scale).cuda()
    x, dx = r(B, T, C, H, W), r(B, T, C, H, W)
    state = [(r(B, hc, H, W, scale=0.5), r(B, hc, H, W, scale=0.5)) for hc in hidden]
    dstate = [(r(B, hc, H, W), r(B, hc, H, W)) for hc in hidden]
    dtheta = {k: r(*v.shape) * float(v.abs().mean()) for k, v in params.items()}
    y, ys = r(B, 1, H, W), r(B, T, H, W)
    return x, dx, state, dstate, dtheta, y, ys


def _losses(net, x, state, y, ys, linear):
    """(device loss, oracle loss): MSE + L1 on pred and seq, the oracle's L1 taken on the device prediction's piece; or
    a loss linear in the outputs (pure model curvature)"""
    if linear:
        f = lambda out: (out[0] * y).mean() + 0.5 * (out[1] * ys).mean()
        return f, f
    with torch.no_grad():
        pred, seq = net(x, hidden_state=state)
    s, ss = torch.sign(pred - y), torch.sign(seq - ys)
    dev = lambda out: (((out[0] - y) ** 2).mean() + (out[0] - y).abs().mean() +
                       0.5 * (((out[1] - ys) ** 2).mean() + (out[1] - ys).abs().mean()))
    ref = lambda out: (((out[0] - y) ** 2).mean() + (s * (out[0] - y)).mean() +
                       0.5 * (((out[1] - ys) ** 2).mean() + (ss * (out[1] - ys)).mean()))
    return dev, ref


def _oracle(params, L, loss_fn, x, state, dx, dstate, dtheta):
    """torch.func forward-over-reverse of the fp32 reference loop (on the GPU, tf32 off)"""
    p = {k: v.cuda() for k, v in params.items()}

    def lf(p, x, hs, cs):
        out, _ = convlstm_forward_state(x, p, L, list(zip(hs, cs)), return_sequence=True)
        return loss_fn(out)
    primals = (p, x, tuple(h for h, _ in state), tuple(c for _, c in state))
    tangents = (dtheta, dx, tuple(h for h, _ in dstate), tuple(c for _, c in dstate))
    return torch.func.jvp(torch.func.grad(lf, argnums=(0, 1, 2, 3)), primals, tangents)


CASES = {
    "one_layer_90x144": (2, 4, 7, 90, 144, [32], [3], PRECISIONS),
    "shipped_3layer": (2, 6, 5, 100, 154, [64, 32, 16], [5, 3, 3], PRECISIONS),
    "cfg2": (32, 12, 21, 90, 144, [64], [3], ["bf16"]),
}


def _errors(ours, ref, L):
    gx, gst, gp = ours
    rp, rx, rh, rc = ref
    e = {"x": O.max_abs_normalised(gx.cpu(), rx.cpu())}
    for l in range(L):
        e[f"h0[{l}]"] = O.max_abs_normalised(gst[l][0].cpu(), rh[l].cpu())
        e[f"c0[{l}]"] = O.max_abs_normalised(gst[l][1].cpu(), rc[l].cpu())
    for k, v in rp.items():
        e[k] = O.max_abs_normalised(gp[k].cpu(), v.cpu())
    return e


@pytest.mark.parametrize("linear", [False, True], ids=["mse_l1", "linear_loss"])
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", list(CASES))
def test_joint_hvp_matches_the_oracle(name, precision, linear):
    """gradient and H v over (x, h0, c0, theta), every parameter output included, for a joint direction"""
    B, T, C, H, W, hidden, ks, precisions = CASES[name]
    if precision not in precisions:
        pytest.skip(f"{name} runs in {precisions} only")
    if linear and name == "cfg2":
        pytest.skip("the linear loss runs on the smaller cases")
    net, params = _net(C, hidden, ks, precision)
    x, dx, state, dstate, dtheta, y, ys = _inputs(B, T, C, H, W, hidden, params)
    dev, ref_loss = _losses(net, x, state, y, ys, linear)
    g_ref, h_ref = _oracle(params, len(hidden), ref_loss, x, state, dx, dstate, dtheta)
    _, g, h = net.hvp(x, dx, dev, hidden_state=state, state_tangent=dstate, param_direction=dtheta, wrt_params=True)
    eg, eh = _errors(g, g_ref, len(hidden)), _errors(h, h_ref, len(hidden))
    # the bar of a parameter block is the parity bar, or, where larger, twice the error of the ordinary backward's
    # gradient of that parameter at the same point (tf32 5x5 layer-0 weights: 3e-3..5e-3 with these inputs): H v's
    # weight block is the sum of two wgrad reductions, each over operands rounded like the backward's
    net.zero_grad()
    dev(net(x, hidden_state=state)).backward()
    bar = {k: TOL[precision] for k in eg}
    for n, p in net.named_parameters():
        bar[n] = max(TOL[precision], 2.0 * O.max_abs_normalised(p.grad.cpu(), g_ref[0][n].cpu()))
    print(f"{name} {precision} linear={linear}: grad worst {max(eg.values()):.2e}, hvp worst {max(eh.values()):.2e}, "
          f"bars above the parity bar {({k: round(v, 4) for k, v in bar.items() if v > TOL[precision]})}")
    bad = {**{'g:' + k: v for k, v in eg.items() if not v < bar[k]}, **{'h:' + k: v for k, v in eh.items() if not v < bar[k]}}
    assert not bad, bad


@pytest.mark.parametrize("precision", PRECISIONS)
def test_gradient_output_matches_the_ordinary_backward(precision):
    B, T, C, H, W, hidden, ks = 2, 4, 7, 90, 144, [32, 16], [3, 5]
    net, params = _net(C, hidden, ks, precision)
    x, dx, state, dstate, dtheta, y, ys = _inputs(B, T, C, H, W, hidden, params)
    dev, _ = _losses(net, x, state, y, ys, False)
    _, g, _ = net.hvp(x, dx, dev, hidden_state=state, param_direction=dtheta, wrt_params=True)
    net.zero_grad()
    dev(net(x, hidden_state=state)).backward()
    errs = {n: O.max_abs_normalised(g[2][n].cpu(), p.grad.cpu()) for n, p in net.named_parameters()}
    print(f"grad vs backward {precision}: worst {max(errs.values()):.2e}")
    assert max(errs.values()) < TOL[precision], errs


def test_absent_direction_gives_the_input_hvp_bitwise():
    """wrt_params on a plan with both flags and no parameter direction: the x and state parts equal hvp's"""
    B, T, C, H, W, hidden, ks = 2, 4, 5, 20, 24, [32, 16], [3, 5]
    net, params = _net(C, hidden, ks, "bf16")
    x, dx, state, dstate, _, y, ys = _inputs(B, T, C, H, W, hidden, params)
    dev, _ = _losses(net, x, state, y, ys, False)
    _, g0, h0 = net.hvp(x, dx, dev, hidden_state=state, state_tangent=dstate)
    _, g1, h1 = net.hvp(x, dx, dev, hidden_state=state, state_tangent=dstate, wrt_params=True)
    for a, b in ((g0, g1), (h0, h1)):
        assert torch.equal(a[0], b[0])
        assert all(torch.equal(p, q) and torch.equal(r, s) for (p, r), (q, s) in zip(a[1], b[1]))


def _det_plan(net, B, T, H, W, C, hidden, ks, precision):
    from nasa_niswan_b200.engine import Plan
    plan = Plan(B, T, H, W, C, hidden, ks, precision=precision, training=True, return_sequence=True,
                deterministic=True, second_order=True, param_tangent=True, input_grad=True)
    for l, cell in enumerate(net.layers):
        plan.set_weights(l, cell.conv.weight, cell.conv.bias)
    plan.set_head(net.conv.weight, net.conv.bias)
    return plan


@pytest.mark.parametrize("precision", PRECISIONS)
def test_deterministic_identities(precision):
    """deterministic plan: the params call is run-to-run bit-identical; H(2v) = 2 H v bit for bit; two directions on
    one forward equal separate calls; a following ordinary backward equals one without the new calls"""
    B, T, C, H, W, hidden, ks = 2, 4, 5, 20, 24, [32, 16], [3, 5]
    net, params = _net(C, hidden, ks, precision)
    x, dx, _, _, dtheta, y, ys = _inputs(B, T, C, H, W, hidden, params)
    d1 = net.param_direction(dtheta)
    d2 = net.param_direction({k: 2 * v for k, v in dtheta.items()})
    d3 = net.param_direction({"layers.1.conv.weight": dtheta["layers.1.conv.weight"], "conv.bias": dtheta["conv.bias"]})
    plan = _det_plan(net, B, T, H, W, C, hidden, ks, precision)
    u, u_seq = y, ys

    def run(d, scale=1.0):
        plan.set_param_tangent(*d)
        dpred, dseq, _ = plan.forward_tangent(scale * dx)
        _, ddx, _, _ = plan.backward_second_order((u, u_seq), (dpred, dseq))    # a loss with d2L/dout2 = identity
        return ddx, plan.backward_second_order_params()
    plan.forward(x)
    a = run(d1)
    b = run(d1)
    c = run(d2, 2.0)
    e = run(d3)
    same = lambda p, q: all(torch.equal(s, t) for s, t in zip(p, q))
    assert torch.equal(a[0], b[0]) and same(a[1][0], b[1][0]) and same(a[1][1], b[1][1])
    assert torch.equal(c[0], 2 * a[0]) and same(c[1][1], [2 * t for t in a[1][1]]) and same(c[1][0], a[1][0])
    ref_bwd = plan.backward(None, ys)
    plan.forward(x)
    e2 = run(d3)
    assert torch.equal(e[0], e2[0]) and same(e[1][1], e2[1][1])
    plan.clear_param_tangent()
    plan.forward(x)
    bwd = plan.backward(None, ys)
    assert same(ref_bwd[0], bwd[0]) and same(ref_bwd[1], bwd[1])
    assert torch.equal(ref_bwd[2], bwd[2]) and torch.equal(ref_bwd[3], bwd[3])


@pytest.mark.parametrize("precision", PRECISIONS)
def test_frame_bank_windows_agree_with_explicit_windows(precision):
    from nasa_niswan_b200.preprocess import FrameBank
    T, C, H, W, N, hidden, ks = 4, 5, 20, 24, 9, [32, 16], [5, 3]
    net, params = _net(C, hidden, ks, precision)
    g = torch.Generator().manual_seed(10)
    record, drecord = torch.randn(N, C, H, W, generator=g).cuda(), torch.randn(N, C, H, W, generator=g).cuda()
    if precision == "bf16":
        record, drecord = record.bfloat16().float(), drecord.bfloat16().float()
    bank = FrameBank.from_frames(record, precision)
    dbank = bank.tangent(drecord)
    starts = torch.tensor([3, 0, 3, 5])
    dtheta = {k: (torch.randn(v.shape, generator=g) * float(v.abs().mean())).cuda() for k, v in params.items()}
    y = torch.randn(4, 1, H, W, generator=g).cuda()
    loss = lambda out: ((out[0] - y) ** 2).mean()
    win = lambda r: torch.stack([r[s:s + T] for s in starts.tolist()])
    _, ga, ha = net.hvp_windows(bank, starts, T, dbank, loss, param_direction=dtheta, wrt_params=True)
    _, gb, hb = net.hvp(win(record), win(drecord), loss, param_direction=dtheta, wrt_params=True)
    for k in dtheta:
        assert O.max_abs_normalised(ga[2][k].cpu(), gb[2][k].cpu()) < 1e-5, k
        assert O.max_abs_normalised(ha[2][k].cpu(), hb[2][k].cpu()) < 1e-5, k


def test_refusals():
    B, T, C, H, W, hidden = 2, 3, 5, 12, 16, [16]
    net, params = _net(C, hidden, [3], "bf16")
    x = torch.randn(B, T, C, H, W, device="cuda")
    u = torch.randn(B, 1, H, W, device="cuda")
    d = net.param_direction({k: torch.randn_like(v) for k, v in net.named_parameters()})
    sp = net.plan_for(x, True, second_order=True)                           # no NINT_FLAG_PARAM_TANGENT
    sp.forward(x)
    sp.forward_tangent(torch.randn_like(x))
    sp.backward_second_order(u, u)
    with pytest.raises(RuntimeError, match="NINT_FLAG_PARAM_TANGENT"):
        sp.backward_second_order_params()
    pp = net.plan_for(x, True, second_order=True, param_tangent=True)
    pp.forward(x)
    with pytest.raises(RuntimeError, match="before nint_backward_second_order"):
        pp.backward_second_order_params()
    pp.set_param_tangent(*d)
    pp.forward_tangent(None)
    with pytest.raises(RuntimeError, match="before nint_backward_second_order"):
        pp.backward_second_order_params()
    pp.backward_second_order(u, u)
    pp.backward_second_order_params()
    pp.clear_param_tangent()                                                # the direction changed: stale
    with pytest.raises(RuntimeError, match="before nint_backward_second_order"):
        pp.backward_second_order_params()
    with pytest.raises(RuntimeError, match="before nint_forward_tangent"):
        pp.backward_second_order(u, u)
    tp = net.plan_for(x, True, param_tangent=True)                          # no NINT_FLAG_SECOND_ORDER
    tp.forward(x)
    tp.set_param_tangent(*d)
    tp.forward_tangent(None)
    with pytest.raises(RuntimeError, match="NINT_FLAG_SECOND_ORDER"):
        tp.backward_second_order(u, u)
    torch.cuda.synchronize()
