"""GPU (B200): the tangent-linear model -- ConvLSTM.jvp / jvp_windows, Plan.forward_tangent[_bank] and the fused
preprocessing's tangent.

References: torch.func.jvp of the fp32 oracle (convlstm_forward_state), with the bars of the parity tests (max|a-b| /
max|b| <= 2e-2 in bf16, <= 1e-3 in tf32); the existing adjoint of the same forward for the dot-product identity; and
bit-for-bit identities wherever the arithmetic is the same (linearity in the direction, explicit vs frame-bank windows,
a window split in two, the primal and a backward untouched by a tangent pass)."""
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
    """(net on the GPU, CPU copies of its parameters)"""
    from nasa_niswan_b200 import ConvLSTM
    torch.manual_seed(seed)
    net = ConvLSTM(C, hidden, ks, len(hidden), precision=precision, return_sequence=return_sequence)
    params = {k: v.detach().clone() for k, v in net.state_dict().items()}
    return net.cuda(), params


def _rand(g, *shape, scale=1.0):
    return torch.randn(*shape, generator=g) * scale


def _oracle_jvp(params, L, x, state, dx, dstate):
    """torch.func.jvp of the fp32 oracle: (pred, seq, [h_T], [c_T]) and their tangents"""
    def f(x, hs, cs):
        (pred, seq), final = convlstm_forward_state(x, params, L, list(zip(hs, cs)), return_sequence=True)
        return pred, seq, tuple(h for h, _ in final), tuple(c for _, c in final)
    primals = (x, tuple(h for h, _ in state), tuple(c for _, c in state))
    tangents = (dx, tuple(h for h, _ in dstate), tuple(c for _, c in dstate))
    with torch.no_grad():
        return torch.func.jvp(f, primals, tangents)


# (B, T, C, H, W, hidden, ks): one layer on the 90x144 grid, ragged tiles with padded hidden sizes, C = 5 and k = 5, the
# shipped three-layer model (5 -> 64/32/16, k 5/3/3) on its 100x154 halo grid, BASELINE cfg 2 at B = 32
CASES = {
    "one_layer_90x144": (2, 4, 7, 90, 144, [32], [3], PRECISIONS),
    "edge_h20_k5": (2, 4, 5, 18, 22, [20], [5], PRECISIONS),
    "edge_two_layers_padded": (3, 3, 5, 20, 26, [20, 48], [5, 3], PRECISIONS),
    "shipped_3layer": (2, 6, 5, 100, 154, [64, 32, 16], [5, 3, 3], PRECISIONS),
    "cfg2": (32, 12, 21, 90, 144, [64], [3], ["bf16"]),
}
_ORACLE = {}


def _case_inputs(name, with_state):
    B, T, C, H, W, hidden, ks, _ = CASES[name]
    g = torch.Generator().manual_seed(31)
    x = _rand(g, B, T, C, H, W)
    dx = _rand(g, B, T, C, H, W)
    zero = [(torch.zeros(B, hc, H, W), torch.zeros(B, hc, H, W)) for hc in hidden]
    if not with_state:
        return x, dx, zero, zero, None, None
    state = [(_rand(g, B, hc, H, W, scale=0.5), _rand(g, B, hc, H, W, scale=0.5)) for hc in hidden]
    dstate = [(_rand(g, B, hc, H, W), _rand(g, B, hc, H, W)) for hc in hidden]
    return x, dx, state, dstate, state, dstate


def _oracle(name, with_state, params):
    key = (name, with_state)
    if key not in _ORACLE:
        x, dx, state, dstate, _, _ = _case_inputs(name, with_state)
        _ORACLE[key] = _oracle_jvp(params, len(CASES[name][5]), x, state, dx, dstate)[1]
    return _ORACLE[key]


def _cuda_pairs(pairs):
    return None if pairs is None else [(h.cuda(), c.cuda()) for h, c in pairs]


@pytest.mark.parametrize("with_state", [False, True], ids=["input_tangent", "input_and_state_tangents"])
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", list(CASES))
def test_tangent_matches_the_oracle_jvp(name, precision, with_state):
    """dpred, dseq, dh_T and dc_T against torch.func.jvp of the fp32 oracle"""
    B, T, C, H, W, hidden, ks, precisions = CASES[name]
    if precision not in precisions:
        pytest.skip(f"{name} runs in {precisions} only")
    net, params = _net(C, hidden, ks, precision)
    ref = _oracle(name, with_state, params)
    x, dx, _, _, state, dstate = _case_inputs(name, with_state)
    (_, final), ((dpred, dseq), dfinal) = net.jvp(x.cuda(), dx.cuda(), hidden_state=_cuda_pairs(state),
                                                  state_tangent=_cuda_pairs(dstate), return_state=True)
    errs = {"dpred": O.max_abs_normalised(dpred.cpu(), ref[0]), "dseq": O.max_abs_normalised(dseq.cpu(), ref[1])}
    for l, (dh, dc) in enumerate(dfinal):
        errs[f"dh_T[{l}]"] = O.max_abs_normalised(dh.cpu(), ref[2][l])
        errs[f"dc_T[{l}]"] = O.max_abs_normalised(dc.cpu(), ref[3][l])
    print(f"{name} {precision} state={with_state}: worst {max(errs.values()):.2e}")
    bad = {k: e for k, e in errs.items() if not e < TOL[precision]}
    assert not bad, bad


# ------------------------------------------------------------------------------------------------ primal untouched
@pytest.mark.parametrize("precision", PRECISIONS)
def test_primal_outputs_equal_forward_bitwise(precision):
    B, T, C, H, W, hidden, ks = 2, 4, 5, 20, 24, [32, 16], [3, 5]
    net, _ = _net(C, hidden, ks, precision)
    g = torch.Generator().manual_seed(2)
    x = _rand(g, B, T, C, H, W).cuda()
    state = _cuda_pairs([(_rand(g, B, hc, H, W), _rand(g, B, hc, H, W)) for hc in hidden])
    ((pred, seq), final), _ = net.jvp(x, torch.randn_like(x), hidden_state=state, return_state=True)
    (pred2, seq2), final2 = net(x, hidden_state=state, return_state=True)
    assert torch.equal(pred, pred2.detach()) and torch.equal(seq, seq2.detach())
    assert all(torch.equal(a, b.detach()) and torch.equal(c, d.detach()) for (a, c), (b, d) in zip(final, final2))
    assert not pred.requires_grad


@pytest.mark.parametrize("precision", PRECISIONS)
def test_backward_after_a_tangent_pass_is_bitwise_unchanged(precision):
    """deterministic plan: a backward (parameter, x, h0 and c0 gradients) that follows two tangent passes of the same
    forward equals the backward of a forward without them"""
    from nasa_niswan_b200.engine import Plan
    B, T, C, H, W, hidden, ks = 2, 5, 5, 20, 24, [32, 16], [3, 5]
    net, _ = _net(C, hidden, ks, precision)
    plan = Plan(B, T, H, W, C, hidden, ks, precision=precision, training=True, return_sequence=True, deterministic=True,
                input_grad=True, state_grad=True, tangent=True)
    for l, cell in enumerate(net.layers):
        plan.set_weights(l, cell.conv.weight, cell.conv.bias)
    plan.set_head(net.conv.weight, net.conv.bias)
    g = torch.Generator().manual_seed(5)
    r = lambda *s: _rand(g, *s).cuda()
    x, dx = r(B, T, C, H, W), r(B, T, C, H, W)
    state = [(r(B, hc, H, W), r(B, hc, H, W)) for hc in hidden]
    dseq, dh_T, dc_T = r(B, T, H, W), [r(B, hc, H, W) for hc in hidden], [r(B, hc, H, W) for hc in hidden]

    def step(tangents):
        plan.forward(x, state)
        for _ in range(tangents):
            plan.forward_tangent(dx, [s[0] for s in state], [s[1] for s in state])
        gw, gb, ghw, ghb = plan.backward(None, dseq, dh_T=dh_T, dc_T=dc_T)
        dh0, dc0 = plan.backward_initial_state()
        return [t.clone() for t in (*gw, *gb, ghw, ghb, plan.backward_input(), *dh0, *dc0)]

    for a, b in zip(step(0), step(2)):
        assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ exact linearity
@pytest.mark.parametrize("precision", PRECISIONS)
def test_exact_linearity(precision):
    """a zero direction gives exactly zero (no bias or constant-1 lane leaks into the tangent); scaling the direction by
    2 scales every output by 2 bit for bit; the state-only and input-only tangents add up to the joint one"""
    B, T, C, H, W, hidden, ks = 2, 4, 5, 20, 24, [20, 32], [5, 3]
    net, _ = _net(C, hidden, ks, precision)
    g = torch.Generator().manual_seed(6)
    x, dx = _rand(g, B, T, C, H, W).cuda(), _rand(g, B, T, C, H, W).cuda()
    state = _cuda_pairs([(_rand(g, B, hc, H, W), _rand(g, B, hc, H, W)) for hc in hidden])
    dstate = _cuda_pairs([(_rand(g, B, hc, H, W), _rand(g, B, hc, H, W)) for hc in hidden])
    flat = lambda r: [r[1][0][0], r[1][0][1]] + [t for pair in r[1][1] for t in pair]
    jvp = lambda d, ds: flat(net.jvp(x, d, hidden_state=state, state_tangent=ds, return_state=True))
    for t in jvp(torch.zeros_like(dx), None) + jvp(None, None):
        assert torch.count_nonzero(t) == 0
    double = [(2 * h, 2 * c) for h, c in dstate]
    for a, b in zip(jvp(dx, dstate), jvp(2 * dx, double)):
        assert torch.equal(2 * a, b)
    joint, inp, st = jvp(dx, dstate), jvp(dx, None), jvp(None, dstate)
    for j, a, b in zip(joint, inp, st):
        assert O.max_abs_normalised((a + b).cpu(), j.cpu()) < TOL[precision]


# ------------------------------------------------------------------------------------------------ dot-product test
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("hidden,ks", [([32], [3]), ([20, 48, 16], [5, 3, 3])], ids=["one_layer", "three_layers"])
def test_dot_product_identity_with_the_adjoint(precision, hidden, ks):
    """<u, J v> from the tangent pass against <J^T u, v> from the backward of the same forward (x.grad, dh0, dc0)"""
    from nasa_niswan_b200.engine import Plan
    B, T, C, H, W = 2, 5, 5, 20, 26
    net, _ = _net(C, hidden, ks, precision)
    plan = Plan(B, T, H, W, C, hidden, ks, precision=precision, training=True, return_sequence=True, input_grad=True,
                state_grad=True, tangent=True)
    for l, cell in enumerate(net.layers):
        plan.set_weights(l, cell.conv.weight, cell.conv.bias)
    plan.set_head(net.conv.weight, net.conv.bias)
    g = torch.Generator().manual_seed(8)
    r = lambda *s: _rand(g, *s).cuda()
    x, state = r(B, T, C, H, W), [(r(B, hc, H, W) * 0.5, r(B, hc, H, W) * 0.5) for hc in hidden]
    v = (r(B, T, C, H, W), [r(B, hc, H, W) for hc in hidden], [r(B, hc, H, W) for hc in hidden])
    u = (r(B, 1, H, W), r(B, T, H, W), [r(B, hc, H, W) for hc in hidden], [r(B, hc, H, W) for hc in hidden])
    plan.forward(x, state)
    dpred, dseq, dfinal = plan.forward_tangent(*v)
    plan.backward(u[0], u[1], dh_T=u[2], dc_T=u[3])
    dx = plan.backward_input()
    dh0, dc0 = plan.backward_initial_state()
    dot = lambda a, b: sum(float((p.double() * q.double()).sum()) for p, q in zip(a, b))
    lhs = dot([u[0], u[1], *u[2], *u[3]], [dpred, dseq, *[h for h, _ in dfinal], *[c for _, c in dfinal]])
    rhs = dot([dx, *dh0, *dc0], [v[0], *v[1], *v[2]])
    print(f"dot product {precision} {hidden}: {lhs:.6e} vs {rhs:.6e}")
    assert abs(lhs - rhs) <= TOL[precision] * max(abs(lhs), abs(rhs))


# ------------------------------------------------------------------------------------------------ paths agree
@pytest.mark.parametrize("precision", PRECISIONS)
def test_frame_bank_windows_equal_explicit_windows_bitwise(precision):
    """jvp_windows over a bank and its tangent bank (repeated window starts included) equals jvp over the same windows
    cut out explicitly"""
    from nasa_niswan_b200.preprocess import FrameBank
    T, C, H, W, N, hidden, ks = 4, 5, 20, 24, 9, [32, 16], [5, 3]
    net, _ = _net(C, hidden, ks, precision)
    g = torch.Generator().manual_seed(10)
    record, drecord = _rand(g, N, C, H, W).cuda(), _rand(g, N, C, H, W).cuda()
    if precision == "bf16":     # the bank holds bf16 frames: explicit windows of the same values
        record, drecord = record.bfloat16().float(), drecord.bfloat16().float()
    bank = FrameBank.from_frames(record, precision)
    dbank = bank.tangent(drecord)
    starts = torch.tensor([3, 0, 3, 5])
    state = _cuda_pairs([(_rand(g, 4, hc, H, W), _rand(g, 4, hc, H, W)) for hc in hidden])
    dstate = _cuda_pairs([(_rand(g, 4, hc, H, W), _rand(g, 4, hc, H, W)) for hc in hidden])
    win = lambda r: torch.stack([r[s:s + T] for s in starts.tolist()])
    a = net.jvp_windows(bank, starts, T, dbank, hidden_state=state, state_tangent=dstate, return_state=True)
    b = net.jvp(win(record), win(drecord), hidden_state=state, state_tangent=dstate, return_state=True)
    (da, dsa), dfa = a[1]
    (db, dsb), dfb = b[1]
    assert torch.equal(da, db) and torch.equal(dsa, dsb)
    assert all(torch.equal(p, q) and torch.equal(s, t) for (p, s), (q, t) in zip(dfa, dfb))
    assert torch.equal(a[0][0][0], b[0][0][0])


@pytest.mark.parametrize("precision", PRECISIONS)
def test_split_window_with_carried_state_tangent_equals_whole_window_bitwise(precision):
    B, T, T1, C, H, W, hidden, ks = 2, 6, 2, 5, 20, 24, [20, 48, 64], [5, 3, 3]
    net, _ = _net(C, hidden, ks, precision)
    g = torch.Generator().manual_seed(11)
    x, dx = _rand(g, B, T, C, H, W).cuda(), _rand(g, B, T, C, H, W).cuda()
    (_, _), ((dpred, dseq), dfin) = net.jvp(x, dx, return_state=True)
    (_, mid), ((_, dseq1), dmid) = net.jvp(x[:, :T1], dx[:, :T1], return_state=True)
    (_, _), ((dpred2, dseq2), dfin2) = net.jvp(x[:, T1:], dx[:, T1:], hidden_state=mid, state_tangent=dmid,
                                               return_state=True)
    assert torch.equal(dpred, dpred2) and torch.equal(dseq, torch.cat([dseq1, dseq2], 1))
    assert all(torch.equal(p, q) and torch.equal(s, t) for (p, s), (q, t) in zip(dfin, dfin2))


# ------------------------------------------------------------------------------------------------ preprocessing
def _round_like_bank(t, precision):
    if precision == "bf16":
        return t.bfloat16().float()
    u = t.view(torch.int32)      # cvt.rna.tf32.f32: round to nearest, ties away from zero, on the magnitude bits
    return ((u + 0x1000) & ~0x1FFF).view(torch.float32)


def _fields(seed, N=10, L=2, H=18, W=24, S=2):
    g = torch.Generator().manual_seed(seed)
    lev, emis = _rand(g, N, L, H, W) * 3 + 1, _rand(g, N, H, W).abs() * 5
    mean, std = _rand(g, L + 1), _rand(g, L + 1).abs() + 0.5
    statics = _rand(g, S, H, W)
    return lev, emis, mean, std, statics


@pytest.mark.parametrize("mode", ["reflect", "reference_rnn"])
@pytest.mark.parametrize("precision", PRECISIONS)
def test_tangent_from_fields_equals_the_restatement_bitwise(precision, mode):
    from nasa_niswan_b200.preprocess import FrameBank
    lev, emis, mean, std, statics = _fields(12)
    g = torch.Generator().manual_seed(13)
    dlev, demis, dstat = _rand(g, *lev.shape), _rand(g, *emis.shape), _rand(g, *statics.shape)
    target = (22, 30)
    bank = FrameBank.from_fields(lev.cuda(), emis.cuda(), mean.cuda(), std.cuda(), target, mode, statics.cuda(), precision)
    C = lev.shape[1] + 1 + statics.shape[0]
    for d in ((dlev, demis, dstat), (None, demis, None), (dlev, None, None)):
        got = bank.tangent_from_fields(*[None if t is None else t.cuda() for t in d])
        z = lambda t, ref: torch.zeros_like(ref) if t is None else t
        ref = fuse_inputs_torch(z(d[0], lev), z(d[1], emis), torch.zeros_like(mean), std, target, mode, z(d[2], statics))
        assert torch.equal(got[..., :C].float().permute(0, 3, 1, 2).cpu(), _round_like_bank(ref, precision))
        assert torch.count_nonzero(got[..., C:]) == 0          # the constant-1 lane and the padding lanes are 0


@pytest.mark.parametrize("precision", PRECISIONS)
def test_emission_response_matches_the_oracle_pipeline(precision):
    """utils.emission_response (a regional emission perturbation over a few frames) against torch.func.jvp of the
    fusion restatement followed by the oracle over the same windows"""
    from nasa_niswan_b200 import utils
    from nasa_niswan_b200.preprocess import FrameBank
    lev, emis, mean, std, statics = _fields(14, N=9)
    target, mode, T = (22, 30), "reference_rnn", 4
    C = lev.shape[1] + 1 + statics.shape[0]
    net, params = _net(C, [32, 16], [5, 3], precision, return_sequence=False)
    bank = FrameBank.from_fields(lev.cuda(), emis.cuda(), mean.cuda(), std.cuda(), target, mode, statics.cuda(), precision)
    d_emis = torch.zeros_like(emis)
    d_emis[2:5, 4:11, 6:15] = 0.1 * emis[2:5, 4:11, 6:15]      # +10 % over a region during three frames
    starts = torch.tensor([0, 2, 5, 2])
    got = utils.emission_response(net, bank, starts, T, d_emis.cuda(), crop=(1, 20, 2, 28), y_std=2.5)

    def pipeline(e):
        frames = fuse_inputs_torch(lev, e, mean, std, target, mode, statics)
        x = torch.stack([frames[s:s + T] for s in starts.tolist()])
        (pred, _), _ = convlstm_forward_state(x, params, 2, return_sequence=True)
        return pred[:, 0, 1:20, 2:28] * 2.5
    with torch.no_grad():
        _, ref = torch.func.jvp(pipeline, (emis,), (d_emis,))
    err = O.max_abs_normalised(got.cpu(), ref)
    print(f"emission response {precision}: {err:.2e}")
    assert err < TOL[precision]


# ------------------------------------------------------------------------------------------------ sweep
@pytest.mark.parametrize("precision", PRECISIONS)
def test_tangent_sweep_matches_the_oracle_jvp_per_feature(precision):
    """utils.tangent_sweep over a two-batch loader against torch.func.jvp of the fp32 oracle in each direction
    perturbation * x restricted to one feature, cropped and de-normalised; the same shape as sensitivity_sweep"""
    from nasa_niswan_b200 import utils
    B, T, C, H, W = 3, 4, 5, 24, 30
    net, params = _net(C, [32, 16], [3, 5], precision, return_sequence=False)
    g = torch.Generator().manual_seed(15)
    X = _rand(g, 2 * B, T, C, H, W)
    loader = [(X[:B], None), (X[B:], None)]
    crop = (2, 20, 3, 27)
    lin = utils.tangent_sweep(loader, net, C, perturbation=0.05, crop=crop, y_std=2.0)
    assert lin.shape == utils.sensitivity_sweep(loader, net, C, crop=crop, y_std=2.0).shape == (C, 2 * B, 18, 24)
    f = lambda x: convlstm_forward_state(x, params, 2)[0][:, 0, crop[0]:crop[1], crop[2]:crop[3]] * 2.0
    for i in range(C):
        v = torch.zeros_like(X)
        v[:, :, i] = X[:, :, i] * 0.05
        with torch.no_grad():
            ref = torch.func.jvp(f, (X,), (v,))[1]
        assert O.max_abs_normalised(lin[i], ref) < TOL[precision]


# ------------------------------------------------------------------------------------------------ refusals
def test_refusals():
    from nasa_niswan_b200 import _lib
    from nasa_niswan_b200.engine import Plan
    from nasa_niswan_b200.preprocess import FrameBank
    B, T, C, H, W, hidden = 2, 3, 5, 12, 16, [16]
    net, _ = _net(C, hidden, [3], "bf16", return_sequence=False)
    x = torch.randn(B, T, C, H, W, device="cuda")
    dx = torch.randn_like(x)
    plan = net.plan_for(x, True)                               # a training plan without NINT_FLAG_TANGENT
    plan.forward(x)
    with pytest.raises(RuntimeError, match="NINT_FLAG_TANGENT"):
        plan.forward_tangent(dx)
    inf = Plan(B, T, H, W, C, hidden, [3], training=False, tangent=True)
    inf.set_weights(0, net.layers[0].conv.weight, net.layers[0].conv.bias)
    inf.set_head(net.conv.weight, net.conv.bias)
    inf.forward(x)
    with pytest.raises(RuntimeError, match="training plan"):
        inf.forward_tangent(dx)
    tp = net.plan_for(x, True, tangent=True)
    with pytest.raises(RuntimeError, match="before nint_forward"):
        tp.forward_tangent(dx)
    tp.forward(x)
    tp.forward_tangent(dx)
    tp.backward(torch.ones(B, 1, H, W, device="cuda"))
    with pytest.raises(RuntimeError, match="consumed"):
        tp.forward_tangent(dx)
    bank = FrameBank.from_frames(torch.randn(T + 2, C, H, W, device="cuda"), "bf16")
    tp.forward_bank(bank.frames, torch.tensor([0, 2], dtype=torch.int32, device="cuda"))
    with pytest.raises(RuntimeError, match="frame bank"):
        tp.forward_tangent(dx)
    tp.forward(x)
    with pytest.raises(RuntimeError, match="did not read a frame bank"):
        tp.forward_tangent_bank(bank.tangent(torch.zeros(T + 2, C, H, W, device="cuda")))
    with pytest.raises(ValueError, match="shape"):
        tp.forward_tangent(dx[:, :2])
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        tp.forward_tangent(dx.cpu())
    with pytest.raises(TypeError, match="float32"):
        tp.forward_tangent(dx.double())
    with pytest.raises(ValueError, match="shape"):
        tp.forward_tangent(dx, dh0=[torch.zeros(B, 8, H, W, device="cuda")])
    with pytest.raises(ValueError, match="shape"):
        net.jvp(x, dx, state_tangent=[(torch.zeros(B, 8, H, W, device="cuda"), None)])
    # a per-step output on a plan without return_sequence
    seq = torch.empty(B, T, H, W, device="cuda")
    rc = tp.lib.nint_forward_tangent(tp._h, _lib.ptr(dx), _lib.X_FP32, None, None, None, _lib.ptr(seq), None, None,
                                     tp._stream())
    assert rc != 0 and "return_sequence" in tp.lib.nint_last_error().decode()
