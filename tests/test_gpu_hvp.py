"""GPU (B200): the second-order adjoint -- ConvLSTM.hvp / hvp_windows, Plan.backward_second_order[_bank] and
utils.emission_hvp.

References: torch.func.jvp(torch.func.grad(L o f)) of the fp32 oracle (convlstm_forward_state, run on the device with
TF32 off), with the bars of the parity tests (max|a-b| / max|b| <= 2e-2 in bf16, <= 1e-3 in tf32); bit-for-bit
identities wherever the arithmetic is the same (linearity in the direction, explicit vs frame-bank windows, several
directions on one forward, a backward untouched by the pass)."""
import pytest
import torch

from oracle import convlstm_oracle as O
from oracle.adjoint_oracle import fuse_inputs_torch
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
    """(net on the GPU, device copies of its parameters for the fp32 oracle)"""
    from nasa_niswan_b200 import ConvLSTM
    torch.manual_seed(seed)
    net = ConvLSTM(C, hidden, ks, len(hidden), precision=precision, return_sequence=return_sequence).cuda()
    params = {k: v.detach().clone() for k, v in net.state_dict().items()}
    return net, params


def _rand(g, *shape, scale=1.0):
    return (torch.randn(*shape, generator=g) * scale).cuda()


def _mse_l1(B, T, H, W, crop, seed=3, at=None):
    """the training loss (MSE + L1 on a crop) on pred and on the sequence: curvature from the MSE.  at: outputs (pred,
    seq) whose L1 piece to keep -- |d| becomes sign(d_at) d, the same loss, gradient and curvature at `at`"""
    g = torch.Generator().manual_seed(seed)
    y, ys = _rand(g, B, 1, H, W), _rand(g, B, T, H, W)
    y0, y1, x0, x1 = crop
    cut = lambda p, t: (p - t)[..., y0:y1, x0:x1]
    signs = None if at is None else (torch.sign(cut(at[0], y)), torch.sign(cut(at[1], ys)))

    def term(p, t, j):
        d = cut(p, t)
        return (d * d).mean() + (d.abs().mean() if signs is None else (signs[j] * d).mean())
    return lambda out: term(out[0], y, 0) + 0.5 * term(out[1], ys, 1)


def _oracle_hvp(params, L, loss_fn, x, state, dx, dstate):
    """(grad, hvp), each (x part, [h0 parts], [c0 parts]), of the fp32 oracle by torch.func"""
    def lf(x, hs, cs):
        out, _ = convlstm_forward_state(x, params, L, list(zip(hs, cs)), return_sequence=True)
        return loss_fn(out)
    primals = (x, tuple(h for h, _ in state), tuple(c for _, c in state))
    tangents = (dx, tuple(h for h, _ in dstate), tuple(c for _, c in dstate))
    with torch.no_grad():
        return torch.func.jvp(torch.func.grad(lf, argnums=(0, 1, 2)), primals, tangents)


# (B, T, C, H, W, hidden, ks, precisions): the case list of the tangent tests
CASES = {
    "one_layer_90x144": (2, 4, 7, 90, 144, [32], [3], PRECISIONS),
    "edge_h20_k5": (2, 4, 5, 18, 22, [20], [5], PRECISIONS),
    "edge_two_layers_padded": (3, 3, 5, 20, 26, [20, 48], [5, 3], PRECISIONS),
    "shipped_3layer": (2, 6, 5, 100, 154, [64, 32, 16], [5, 3, 3], PRECISIONS),
    "cfg2": (32, 12, 21, 90, 144, [64], [3], ["bf16"]),
}


def _case_inputs(name, with_state):
    B, T, C, H, W, hidden, ks, _ = CASES[name]
    g = torch.Generator().manual_seed(31)
    x, dx = _rand(g, B, T, C, H, W), _rand(g, B, T, C, H, W)
    zero = [(torch.zeros(B, hc, H, W, device="cuda"), torch.zeros(B, hc, H, W, device="cuda")) for hc in hidden]
    if not with_state:
        return x, dx, zero, zero, None, None
    state = [(_rand(g, B, hc, H, W, scale=0.5), _rand(g, B, hc, H, W, scale=0.5)) for hc in hidden]
    dstate = [(_rand(g, B, hc, H, W), _rand(g, B, hc, H, W)) for hc in hidden]
    return x, dx, state, dstate, state, dstate


def _errs(got, ref, with_state):
    (gx, gs), (hx, hs) = got
    e = {"grad_x": O.max_abs_normalised(gx, ref[0][0]), "hvp_x": O.max_abs_normalised(hx, ref[1][0])}
    if with_state:
        for l in range(len(gs)):
            e[f"grad_h0[{l}]"] = O.max_abs_normalised(gs[l][0], ref[0][1][l])
            e[f"grad_c0[{l}]"] = O.max_abs_normalised(gs[l][1], ref[0][2][l])
            e[f"hvp_h0[{l}]"] = O.max_abs_normalised(hs[l][0], ref[1][1][l])
            e[f"hvp_c0[{l}]"] = O.max_abs_normalised(hs[l][1], ref[1][2][l])
    return e


@pytest.mark.parametrize("with_state", [False, True], ids=["input_direction", "input_and_state_directions"])
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", list(CASES))
def test_hvp_matches_the_oracle(name, precision, with_state):
    """loss, gradient and H v w.r.t. x (and the initial state) against torch.func of the fp32 oracle, MSE + L1 loss"""
    B, T, C, H, W, hidden, ks, precisions = CASES[name]
    if precision not in precisions:
        pytest.skip(f"{name} runs in {precisions} only")
    net, params = _net(C, hidden, ks, precision)
    x, dx, state, dstate, hs, ds = _case_inputs(name, with_state)
    crop = (2, H - 2, 3, W - 3)
    loss_fn = _mse_l1(B, T, H, W, crop)
    loss, grad, hv = net.hvp(x, dx, loss_fn, hidden_state=hs, state_tangent=ds)
    # L1's derivative jumps where the prediction crosses the target: where the bf16 / tf32 prediction and the fp32 one
    # sit on different sides, their seeds u differ by 2/n.  The oracle is therefore differentiated on the L1 piece of the
    # device's prediction -- the same loss at that point -- and the unpinned comparison is reported for the record.
    at = net.plan_for(x, True, second_order=True).forward(x, hs)
    ref = _oracle_hvp(params, len(hidden), _mse_l1(B, T, H, W, crop, at=at), x, state, dx, dstate)
    errs = _errs((grad, hv), ref, with_state)
    free = _errs((grad, hv), _oracle_hvp(params, len(hidden), loss_fn, x, state, dx, dstate), with_state)
    print(f"{name} {precision} state={with_state}: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()) +
          f" | L1 piece of the fp32 prediction: worst {max(free.values()):.2e}")
    bad = {k: e for k, e in errs.items() if not e < TOL[precision]}
    assert not bad, bad
    assert (grad[1] is None) == (not with_state)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_linear_loss_gives_the_pure_model_curvature(precision):
    """L = <r, pred> has L'' = 0: the jvp + backward (Gauss-Newton) composition is exactly zero, the HVP is the
    curvature of the recurrence alone, and it matches the oracle"""
    from nasa_niswan_b200.engine import Plan
    B, T, C, H, W, hidden, ks = 2, 5, 5, 20, 26, [32, 16], [3, 5]
    net, params = _net(C, hidden, ks, precision)
    g = torch.Generator().manual_seed(4)
    x, dx, r = _rand(g, B, T, C, H, W), _rand(g, B, T, C, H, W), _rand(g, B, 1, H, W)
    loss_fn = lambda out: (out[0] * r).sum()
    zero = [(torch.zeros(B, hc, H, W, device="cuda"),) * 2 for hc in hidden]
    ref = _oracle_hvp(params, len(hidden), loss_fn, x, zero, dx, zero)
    _, (gx, _), (hx, _) = net.hvp(x, dx, loss_fn)
    assert torch.count_nonzero(hx) > 0
    e = O.max_abs_normalised(hx, ref[1][0]), O.max_abs_normalised(gx, ref[0][0])
    print(f"linear loss {precision}: hvp {e[0]:.2e} grad {e[1]:.2e}")
    assert max(e) < TOL[precision]
    plan = Plan(B, T, H, W, C, hidden, ks, precision=precision, training=True, return_sequence=True, input_grad=True,
                tangent=True)
    for l, cell in enumerate(net.layers):
        plan.set_weights(l, cell.conv.weight, cell.conv.bias)
    plan.set_head(net.conv.weight, net.conv.bias)
    plan.forward(x)
    plan.forward_tangent(dx)
    plan.backward(torch.zeros(B, 1, H, W, device="cuda"))       # L'' J v = 0
    assert torch.count_nonzero(plan.backward_input()) == 0


def _plan(net, B, T, H, W, C, hidden, ks, precision, **kw):
    from nasa_niswan_b200.engine import Plan
    plan = Plan(B, T, H, W, C, hidden, ks, precision=precision, training=True, return_sequence=True, **kw)
    for l, cell in enumerate(net.layers):
        plan.set_weights(l, cell.conv.weight, cell.conv.bias)
    plan.set_head(net.conv.weight, net.conv.bias)
    return plan


@pytest.mark.parametrize("precision", PRECISIONS)
def test_exact_identities(precision):
    """H(2v) = 2 H v and H 0 = 0 bit for bit; two directions on one forward equal two separate forwards"""
    B, T, C, H, W, hidden, ks = 2, 4, 5, 20, 24, [20, 32], [5, 3]
    net, _ = _net(C, hidden, ks, precision)
    g = torch.Generator().manual_seed(6)
    x, v, w = _rand(g, B, T, C, H, W), _rand(g, B, T, C, H, W), _rand(g, B, T, C, H, W)
    state = [(_rand(g, B, hc, H, W), _rand(g, B, hc, H, W)) for hc in hidden]
    dv = [(_rand(g, B, hc, H, W), _rand(g, B, hc, H, W)) for hc in hidden]
    loss_fn = _mse_l1(B, T, H, W, (1, H - 1, 1, W - 1))
    flat = lambda r: [r[2][0]] + [t for p in (r[2][1] or []) for t in p]
    one = flat(net.hvp(x, v, loss_fn, hidden_state=state, state_tangent=dv))
    two = flat(net.hvp(x, 2 * v, loss_fn, hidden_state=state, state_tangent=[(2 * h, 2 * c) for h, c in dv]))
    assert all(torch.equal(2 * a, b) for a, b in zip(one, two))
    for t in flat(net.hvp(x, torch.zeros_like(v), loss_fn, hidden_state=state)) + flat(net.hvp(x, None, loss_fn)):
        assert torch.count_nonzero(t) == 0
    # several directions on one forward (the plan API) equal one forward per direction
    seeds = lambda pred, seq, dpred, dseq: net._loss_seeds(loss_fn, pred, seq, dpred, dseq)[1:]
    plan = net.plan_for(x, True, second_order=True)
    pred, seq = plan.forward(x, state)
    together = []
    for d in (v, w):
        dpred, dseq, _ = plan.forward_tangent(d)
        u, du = seeds(pred, seq, dpred, dseq)
        together.append([t.clone() for t in plan.backward_second_order(u, du)[:2]])
    for d, got in zip((v, w), together):
        _, (gx, _), (hx, _) = net.hvp(x, d, loss_fn, hidden_state=state)
        assert torch.equal(got[0], gx) and torch.equal(got[1], hx)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_backward_after_a_second_order_pass_is_bitwise_unchanged(precision):
    """deterministic plan: a backward (parameter, x, h0 and c0 gradients) after two (tangent, second-order) pairs of the
    same forward equals the backward of a forward without them"""
    B, T, C, H, W, hidden, ks = 2, 5, 5, 20, 24, [32, 16], [3, 5]
    net, _ = _net(C, hidden, ks, precision)
    plan = _plan(net, B, T, H, W, C, hidden, ks, precision, deterministic=True, input_grad=True, state_grad=True,
                 second_order=True)
    g = torch.Generator().manual_seed(5)
    x, dx = _rand(g, B, T, C, H, W), _rand(g, B, T, C, H, W)
    state = [(_rand(g, B, hc, H, W), _rand(g, B, hc, H, W)) for hc in hidden]
    dseq, dh_T, dc_T = _rand(g, B, T, H, W), [_rand(g, B, hc, H, W) for hc in hidden], [_rand(g, B, hc, H, W) for hc in hidden]

    def step(pairs):
        plan.forward(x, state)
        for _ in range(pairs):
            plan.forward_tangent(dx, [s[0] for s in state], [s[1] for s in state])
            plan.backward_second_order((None, dseq), (None, 0.5 * dseq), state=True)
        gw, gb, ghw, ghb = plan.backward(None, dseq, dh_T=dh_T, dc_T=dc_T)
        dh0, dc0 = plan.backward_initial_state()
        return [t.clone() for t in (*gw, *gb, ghw, ghb, plan.backward_input(), *dh0, *dc0)]

    for a, b in zip(step(0), step(2)):
        assert torch.equal(a, b)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_frame_bank_windows_equal_explicit_windows_scattered(precision):
    """hvp_windows (repeated window starts included) equals hvp over the same windows cut out explicitly, its per-window
    results added into the frames in decreasing t, then increasing b -- bit for bit"""
    from nasa_niswan_b200.preprocess import FrameBank
    T, C, H, W, N, hidden, ks = 4, 5, 20, 24, 9, [32, 16], [5, 3]
    net, _ = _net(C, hidden, ks, precision)
    g = torch.Generator().manual_seed(10)
    record, drecord = _rand(g, N, C, H, W), _rand(g, N, C, H, W)
    if precision == "bf16":     # the bank holds bf16 frames: explicit windows of the same values
        record, drecord = record.bfloat16().float(), drecord.bfloat16().float()
    bank = FrameBank.from_frames(record, precision)
    starts = torch.tensor([3, 0, 3, 5])
    state = [(_rand(g, 4, hc, H, W), _rand(g, 4, hc, H, W)) for hc in hidden]
    dstate = [(_rand(g, 4, hc, H, W), _rand(g, 4, hc, H, W)) for hc in hidden]
    loss_fn = _mse_l1(4, T, H, W, (1, H - 1, 1, W - 1))
    la, (ga, gsa), (ha, hsa) = net.hvp_windows(bank, starts, T, bank.tangent(drecord), loss_fn, hidden_state=state,
                                               state_tangent=dstate)
    win = lambda r: torch.stack([r[s:s + T] for s in starts.tolist()])
    lb, (gb, gsb), (hb, hsb) = net.hvp(win(record), win(drecord), loss_fn, hidden_state=state, state_tangent=dstate)
    assert torch.equal(la, lb)

    def scatter(d):             # frame f sums its terms in decreasing t (the pass runs backwards in time), then b
        out = torch.zeros(N, C, H, W)
        for t in reversed(range(T)):
            for b, s in enumerate(starts.tolist()):
                out[s + t] += d[b, t].cpu()
        return out
    assert torch.equal(ga.cpu(), scatter(gb)) and torch.equal(ha.cpu(), scatter(hb))
    assert all(torch.equal(p, q) for a, b in ((gsa, gsb), (hsa, hsb)) for pa, pb in zip(a, b) for p, q in zip(pa, pb))
    assert bank.grad is None


@pytest.mark.parametrize("precision", PRECISIONS)
def test_emission_hvp_matches_the_oracle_pipeline(precision):
    """utils.emission_hvp against torch.func of the fusion restatement followed by the oracle over the same windows"""
    from nasa_niswan_b200 import utils
    from nasa_niswan_b200.preprocess import FrameBank
    g = torch.Generator().manual_seed(14)
    N, Lv, H, W, S = 9, 2, 18, 24, 2
    lev, emis = _rand(g, N, Lv, H, W) * 3 + 1, _rand(g, N, H, W).abs() * 5
    mean, std, statics = _rand(g, Lv + 1), _rand(g, Lv + 1).abs() + 0.5, _rand(g, S, H, W)
    target, mode, T = (22, 30), "reference_rnn", 4
    C = Lv + 1 + S
    net, params = _net(C, [32, 16], [5, 3], precision)
    bank = FrameBank.from_fields(lev, emis, mean, std, target, mode, statics, precision)
    d_emis = torch.zeros_like(emis)
    d_emis[2:5, 4:11, 6:15] = 0.1 * emis[2:5, 4:11, 6:15]
    starts = torch.tensor([0, 2, 5, 2])
    loss_fn = _mse_l1(4, T, *target, (2, 20, 3, 27))
    got = utils.emission_hvp(net, bank, starts, T, d_emis, loss_fn)

    def lf(lev_, e, st):
        frames = fuse_inputs_torch(lev_, e, mean, std, target, mode, st)
        x = torch.stack([frames[s:s + T] for s in starts.tolist()])
        out, _ = convlstm_forward_state(x, params, 2, [(torch.zeros(4, hc, *target, device="cuda"),) * 2
                                                       for hc in (32, 16)], return_sequence=True)
        return loss_fn(out)
    with torch.no_grad():
        _, ref = torch.func.jvp(torch.func.grad(lf, argnums=(0, 1, 2)), (lev, emis, statics),
                                (torch.zeros_like(lev), d_emis, torch.zeros_like(statics)))
    errs = {k: O.max_abs_normalised(got[k], r) for k, r in zip(("levels3d", "emis2d", "statics"), ref)}
    print(f"emission hvp {precision}: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert max(errs.values()) < TOL[precision]


def test_flagless_launch_sequences_are_unchanged():
    """the flag adds launches only in its own pass: forward, tangent and backward issue the same launches per kernel
    class on a tangent-only plan and on a second-order plan, and forward + backward the same on a plan without either"""
    from nasa_niswan_b200 import _lib
    B, T, C, H, W, hidden, ks = 2, 4, 5, 20, 24, [32, 16], [3, 5]
    net, _ = _net(C, hidden, ks, "bf16")
    lib = _lib.load()
    g = torch.Generator().manual_seed(7)
    x, dx, dseq = _rand(g, B, T, C, H, W), _rand(g, B, T, C, H, W), _rand(g, B, T, H, W)

    def counts(plan, tangent):
        before = [lib.nint_launch_count(c) for c in range(4)]
        plan.forward(x)
        if tangent:
            plan.forward_tangent(dx)
        plan.backward(None, dseq)
        torch.cuda.synchronize()
        return [lib.nint_launch_count(c) - b for c, b in zip(range(4), before)]
    plain = _plan(net, B, T, H, W, C, hidden, ks, "bf16")
    tan = _plan(net, B, T, H, W, C, hidden, ks, "bf16", tangent=True)
    soa = _plan(net, B, T, H, W, C, hidden, ks, "bf16", second_order=True)
    assert counts(tan, True) == counts(soa, True)
    assert counts(plain, False) == counts(soa, False)


def test_refusals():
    from nasa_niswan_b200 import _lib
    from nasa_niswan_b200.engine import Plan
    from nasa_niswan_b200.preprocess import FrameBank
    B, T, C, H, W, hidden = 2, 3, 5, 12, 16, [16]
    net, _ = _net(C, hidden, [3], "bf16", return_sequence=False)
    x = torch.randn(B, T, C, H, W, device="cuda")
    dx, u = torch.randn_like(x), torch.randn(B, 1, H, W, device="cuda")
    tp = net.plan_for(x, True, tangent=True)                    # a tangent plan without NINT_FLAG_SECOND_ORDER
    tp.forward(x)
    tp.forward_tangent(dx)
    with pytest.raises(RuntimeError, match="NINT_FLAG_SECOND_ORDER"):
        tp.backward_second_order(u, u)
    inf = Plan(B, T, H, W, C, hidden, [3], training=False, second_order=True)
    inf.set_weights(0, net.layers[0].conv.weight, net.layers[0].conv.bias)
    inf.set_head(net.conv.weight, net.conv.bias)
    inf.forward(x)
    with pytest.raises(RuntimeError, match="training plan"):
        inf.backward_second_order(u, u)
    sp = net.plan_for(x, True, second_order=True)
    with pytest.raises(RuntimeError, match="before nint_forward"):
        sp.backward_second_order(u, u)
    sp.forward(x)
    with pytest.raises(RuntimeError, match="before nint_forward_tangent"):
        sp.backward_second_order(u, u)
    sp.forward_tangent(dx)
    sp.backward_second_order(u, u)
    sp.forward(x)                                               # a new forward: the old tangent history is stale
    with pytest.raises(RuntimeError, match="before nint_forward_tangent"):
        sp.backward_second_order(u, u)
    sp.forward_tangent(dx)
    sp.backward(u)
    with pytest.raises(RuntimeError, match="consumed"):
        sp.backward_second_order(u, u)
    bank = FrameBank.from_frames(torch.randn(T + 2, C, H, W, device="cuda"), "bf16")
    frames = torch.zeros(T + 2, C, H, W, device="cuda")
    sp.forward_bank(bank.frames, torch.tensor([0, 2], dtype=torch.int32, device="cuda"))
    sp.forward_tangent_bank(bank.tangent(frames))
    with pytest.raises(RuntimeError, match="frame bank"):
        sp.backward_second_order(u, u)
    sp.forward(x)
    sp.forward_tangent(dx)
    with pytest.raises(RuntimeError, match="did not read a frame bank"):
        sp.backward_second_order_bank(u, u, frames, frames.clone())
    with pytest.raises(ValueError, match="shape"):
        sp.backward_second_order(u[:, :, :4], u)
    # a per-step seed on a plan without return_sequence
    seq = torch.zeros(B, T, H, W, device="cuda")
    rc = sp.lib.nint_backward_second_order(sp._h, _lib.ptr(u), None, None, _lib.ptr(seq), None, None, None, None, None,
                                           None, sp._stream())
    assert rc != 0 and "return_sequence" in sp.lib.nint_last_error().decode()
