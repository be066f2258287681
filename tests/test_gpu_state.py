"""GPU (B200): ConvLSTM from an explicit initial state, returning the final state, with gradients through both.

Every case runs in bf16 and tf32, and with one launch per step (NINT_FUSE_STEPS=0) as well as with time-fused forward
and BPTT launches (NINT_FUSE_STEPS=3), so both launch schedules start the forward at t=0 from a real state and end the
BPTT at t=0 against a real c_{-1}.  Metric and bars as in test_gpu_parity.py: max|a-b| / max|b| vs the fp32 oracle,
<= 1e-3 (tf32) / <= 2e-2 (bf16)."""
import pytest
import torch

from oracle import convlstm_oracle as O
from oracle.state_oracle import convlstm_forward_state

pytestmark = pytest.mark.gpu

TOL = {"tf32": 1e-3, "bf16": 2e-2}
PRECISIONS = ["bf16", "tf32"]
FUSE = ["0", "3"]


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists)")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.deterministic = False


def _net(C, hidden, ks, precision, seed=0, **kw):
    """(net on the GPU, CPU copies of its parameters)"""
    from nasa_niswan_b200 import ConvLSTM
    torch.manual_seed(seed)
    net = ConvLSTM(C, hidden, ks, len(hidden), precision=precision, **kw)
    params = {k: v.detach().clone() for k, v in net.state_dict().items()}
    return net.cuda(), params


def _random_state(B, hidden, H, W, seed, scale=0.5):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(B, hc, H, W, generator=g) * scale, torch.randn(B, hc, H, W, generator=g) * scale)
            for hc in hidden]


def _equal_states(a, b):
    return len(a) == len(b) and all(torch.equal(h, h2) and torch.equal(c, c2) for (h, c), (h2, c2) in zip(a, b))


# ------------------------------------------------------------------------------------------------ split equivalence
SPLIT_GEOMS = [([64], [3]), ([20, 48, 64], [5, 3, 3])]


@pytest.mark.parametrize("fuse", FUSE)
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("hidden,ks", SPLIT_GEOMS, ids=["one_layer_k3", "three_layers_padded_k533"])
def test_split_window_equals_whole_window_bitwise(monkeypatch, hidden, ks, precision, fuse):
    """forward(x[:, :T1]) then forward(x[:, T1:], hidden_state=its final state) gives the pred, seq and final state of
    forward(x) bit for bit: per-tile arithmetic does not depend on the launch schedule, h round-trips exactly through
    get_state / set_state (a stored bf16 h is exact in fp32; tf32 rounding is idempotent) and c stays fp32.  Training
    plans (every h_t kept) and inference plans (2-slot h ring, c updated in place) both."""
    monkeypatch.setenv("NINT_FUSE_STEPS", fuse)
    B, T, T1, C, H, W = 3, 6, 2, 5, 20, 24
    torch.manual_seed(4)
    x = torch.randn(B, T, C, H, W, device="cuda")
    net_tr, _ = _net(C, hidden, ks, precision, return_sequence=True)
    (pred, seq), fin = net_tr(x, return_state=True)
    (_, seq1), mid = net_tr(x[:, :T1], return_state=True)
    (pred2, seq2), fin2 = net_tr(x[:, T1:], hidden_state=mid, return_state=True)
    assert torch.equal(pred, pred2) and torch.equal(seq, torch.cat([seq1, seq2], 1))
    assert _equal_states(fin, fin2)
    net_inf, _ = _net(C, hidden, ks, precision)
    with torch.no_grad():
        pred, fin = net_inf(x, return_state=True)
        _, mid = net_inf(x[:, :T1], return_state=True)
        pred2, fin2 = net_inf(x[:, T1:], hidden_state=mid, return_state=True)
    assert torch.equal(pred, pred2) and _equal_states(fin, fin2)


@pytest.mark.parametrize("fuse", FUSE)
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("hidden,ks", SPLIT_GEOMS, ids=["one_layer_k3", "three_layers_padded_k533"])
def test_split_frame_bank_windows_equal_the_whole_window_bitwise(monkeypatch, hidden, ks, precision, fuse):
    """the same through forward_windows: the second call reads frames win_start + T1 .. win_start + T - 1"""
    from nasa_niswan_b200.preprocess import FrameBank
    monkeypatch.setenv("NINT_FUSE_STEPS", fuse)
    T, T1, C, H, W, N = 6, 2, 5, 20, 24, 11
    torch.manual_seed(5)
    record = torch.randn(N, C, H, W, device="cuda")
    bank = FrameBank.from_frames(record, precision)
    starts = torch.tensor([4, 0, 5], dtype=torch.int32)
    net, _ = _net(C, hidden, ks, precision, return_sequence=True)
    (pred, seq), fin = net.forward_windows(bank, starts, T, return_state=True)
    (_, seq1), mid = net.forward_windows(bank, starts, T1, return_state=True)
    (pred2, seq2), fin2 = net.forward_windows(bank, starts + T1, T - T1, hidden_state=mid, return_state=True)
    assert torch.equal(pred, pred2) and torch.equal(seq, torch.cat([seq1, seq2], 1))
    assert _equal_states(fin, fin2)


# ------------------------------------------------------------------------------------------------ oracle parity
# (B, T, C, H, W, hidden, ks): small padded cases, BASELINE cfg 2 (B=32, T=12, 21 -> 64, 90x144) and the shipped
# three-layer model (64/32/16, k 5/3/3) on its 100x154 halo grid
PARITY_CASES = {
    "one_layer_h20_k5": (2, 4, 7, 18, 22, [20], [5]),
    "three_layers_padded": (2, 4, 5, 20, 24, [20, 48, 64], [5, 3, 3]),
    "cfg2": (32, 12, 21, 90, 144, [64], [3]),
    "shipped_3layer": (2, 6, 5, 100, 154, [64, 32, 16], [5, 3, 3]),
}
_ORACLE = {}


def _parity_inputs(name):
    B, T, C, H, W, hidden, ks = PARITY_CASES[name]
    g = torch.Generator().manual_seed(21)
    x = torch.randn(B, T, C, H, W, generator=g)
    state = _random_state(B, hidden, H, W, seed=22)
    # a linear loss on every output: both sides back-propagate the same upstream gradients (the top layer's dL/dh_T
    # joins the head's dpred term in the same epilogue)
    w = dict(pred=torch.randn(B, 1, H, W, generator=g), seq=torch.randn(B, T, H, W, generator=g),
             h=[torch.randn(B, hc, H, W, generator=g) for hc in hidden],
             c=[torch.randn(B, hc, H, W, generator=g) for hc in hidden])
    return x, state, w


def _loss(pred, seq, final, w):
    loss = (pred * w["pred"]).sum() + (seq * w["seq"]).sum()
    for (h, c), wh, wc in zip(final, w["h"], w["c"]):
        loss = loss + (h * wh).sum() + (c * wc).sum()
    return loss


def _oracle(name, params):
    if name not in _ORACLE:
        x, state, w = _parity_inputs(name)
        L = len(PARITY_CASES[name][5])
        leaf = {k: v.clone().requires_grad_(True) for k, v in params.items()}
        xl = x.clone().requires_grad_(True)
        st = [(h.clone().requires_grad_(True), c.clone().requires_grad_(True)) for h, c in state]
        (pred, seq), final = convlstm_forward_state(xl, leaf, L, st, return_sequence=True)
        _loss(pred, seq, final, w).backward()
        _ORACLE[name] = dict(pred=pred.detach(), seq=seq.detach(), final=[(h.detach(), c.detach()) for h, c in final],
                             grads={k: v.grad for k, v in leaf.items()}, dx=xl.grad,
                             dh0=[h.grad for h, _ in st], dc0=[c.grad for _, c in st])
    return _ORACLE[name]


@pytest.mark.parametrize("fuse", FUSE)
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", list(PARITY_CASES))
def test_explicit_state_matches_the_oracle(monkeypatch, name, precision, fuse):
    """random nonzero (h0, c0) per layer requiring grad, a loss on pred, seq, h_T and c_T: outputs, every parameter
    gradient, x.grad, h0.grad and c0.grad against the fp32 oracle's autograd"""
    monkeypatch.setenv("NINT_FUSE_STEPS", fuse)
    B, T, C, H, W, hidden, ks = PARITY_CASES[name]
    net, params = _net(C, hidden, ks, precision, return_sequence=True)
    ref = _oracle(name, params)
    x, state, w = _parity_inputs(name)
    cu = lambda t: t.cuda()
    xd = x.cuda().requires_grad_(True)
    st = [(h.cuda().requires_grad_(True), c.cuda().requires_grad_(True)) for h, c in state]
    (pred, seq), final = net(xd, hidden_state=st, return_state=True)
    _loss(pred, seq, final, {"pred": cu(w["pred"]), "seq": cu(w["seq"]), "h": [cu(t) for t in w["h"]],
                             "c": [cu(t) for t in w["c"]]}).backward()
    tol = TOL[precision]
    errs = {"pred": O.max_abs_normalised(pred.detach().cpu(), ref["pred"]),
            "seq": O.max_abs_normalised(seq.detach().cpu(), ref["seq"]),
            "x.grad": O.max_abs_normalised(xd.grad.cpu(), ref["dx"])}
    for l, ((h, c), (rh, rc)) in enumerate(zip(final, ref["final"])):
        errs[f"h_T[{l}]"] = O.max_abs_normalised(h.detach().cpu(), rh)
        errs[f"c_T[{l}]"] = O.max_abs_normalised(c.detach().cpu(), rc)
    for l, (h, c) in enumerate(st):
        errs[f"h0.grad[{l}]"] = O.max_abs_normalised(h.grad.cpu(), ref["dh0"][l])
        errs[f"c0.grad[{l}]"] = O.max_abs_normalised(c.grad.cpu(), ref["dc0"][l])
    for k, p in net.named_parameters():
        errs[k] = O.max_abs_normalised(p.grad.cpu(), ref["grads"][k])
    bad = {k: e for k, e in errs.items() if not e < tol}
    print(f"{name} {precision} fuse={fuse}: worst {max(errs.values()):.2e}")
    assert not bad, bad


# ------------------------------------------------------------------------------------------------ truncated BPTT
@pytest.mark.parametrize("fuse", FUSE)
@pytest.mark.parametrize("precision", PRECISIONS)
def test_chained_windows_differentiate_like_the_whole_window(monkeypatch, precision, fuse):
    """two chained calls with the state NOT detached: the gradients (parameters, x, initial state) equal those of one
    call over the whole window; the first window's backward gets dL/dh_T and dL/dc_T from the second one's dh0 and
    dc0 next to its own head gradient.  In deterministic mode two identical stateful runs are bit-identical."""
    monkeypatch.setenv("NINT_FUSE_STEPS", fuse)
    B, T, T1, C, H, W, hidden, ks = 2, 7, 3, 5, 20, 24, [32, 16], [3, 5]
    torch.manual_seed(8)
    x0 = torch.randn(B, T, C, H, W, device="cuda")
    s0 = [(h.cuda(), c.cuda()) for h, c in _random_state(B, hidden, H, W, seed=9)]
    wp1, wp2 = torch.randn(B, 1, H, W, device="cuda"), torch.randn(B, 1, H, W, device="cuda")

    def run(chained):
        net, _ = _net(C, hidden, ks, precision, seed=3)
        x = x0.clone().requires_grad_(True)
        st = [(h.clone().requires_grad_(True), c.clone().requires_grad_(True)) for h, c in s0]
        if chained:
            p1, mid = net(x[:, :T1], hidden_state=st, return_state=True)
            p2, fin = net(x[:, T1:], hidden_state=mid, return_state=True)
        else:
            p2, fin = net(x, hidden_state=st, return_state=True)
            p1 = net(x[:, :T1], hidden_state=st)           # the first window's pred, on a plan of its own
        loss = (p1 * wp1).sum() + (p2 * wp2).sum() + fin[-1][0].square().sum()
        loss.backward()
        return [p.grad for p in net.parameters()] + [x.grad] + [t.grad for pair in st for t in pair]

    whole, chain = run(False), run(True)
    for a, b in zip(whole, chain):
        assert O.max_abs_normalised(b.cpu(), a.cpu()) < TOL[precision]
    prev = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        again, again2 = run(True), run(True)
    finally:
        torch.backends.cudnn.deterministic = prev
    for a, b in zip(again, again2):
        assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ state hygiene
@pytest.mark.parametrize("fuse", FUSE)
@pytest.mark.parametrize("precision", PRECISIONS)
def test_no_state_leaks_into_a_later_stateless_forward(monkeypatch, precision, fuse):
    """plans are cached and shared: a stateless forward right after a stateful one on the same module (same plan)
    equals a fresh stateless forward bit for bit, in inference and in training"""
    monkeypatch.setenv("NINT_FUSE_STEPS", fuse)
    B, T, C, H, W, hidden, ks = 2, 5, 5, 20, 24, [32, 16], [3, 3]
    torch.manual_seed(12)
    x = torch.randn(B, T, C, H, W, device="cuda")
    state = [(h.cuda(), c.cuda()) for h, c in _random_state(B, hidden, H, W, seed=13)]
    for grad in (False, True):
        with torch.set_grad_enabled(grad):
            fresh, _ = _net(C, hidden, ks, precision, seed=1)
            want = fresh(x).detach()
            net, _ = _net(C, hidden, ks, precision, seed=1)
            stateful = net(x, hidden_state=state).detach()
            got = net(x).detach()
            assert len(net._plans._plans) == 1          # the stateful and the stateless call shared one plan
        assert not torch.equal(stateful, want)
        assert torch.equal(got, want)


def test_a_pair_of_nones_is_the_zero_state_of_that_layer():
    B, T, C, H, W, hidden = 2, 4, 5, 20, 24, [32, 16]
    net, _ = _net(C, hidden, [3, 3], "bf16")
    x = torch.randn(B, T, C, H, W, device="cuda")
    h1, c1 = (t.cuda() for t in _random_state(B, hidden, H, W, seed=3)[1])
    with torch.no_grad():
        a = net(x, hidden_state=[(None, None), (h1, c1)])
        z = torch.zeros(B, hidden[0], H, W, device="cuda")
        b = net(x, hidden_state=[(z, z), (h1, c1)])
        assert torch.equal(a, b)
        assert torch.equal(net(x, hidden_state=[(None, None), (None, None)]), net(x))


# ------------------------------------------------------------------------------------------------ refusals
def test_refusals():
    """a second backward of one stateful forward, a state of the wrong shape, device or dtype, and state gradients on
    a plan made without room for them"""
    B, T, C, H, W, hidden = 2, 3, 5, 12, 16, [16]
    net, _ = _net(C, hidden, [3], "bf16")
    x = torch.randn(B, T, C, H, W, device="cuda")
    h0 = torch.randn(B, 16, H, W, device="cuda", requires_grad=True)
    c0 = torch.randn(B, 16, H, W, device="cuda")
    pred, fin = net(x, hidden_state=[(h0, c0)], return_state=True)
    loss = pred.sum() + fin[0][1].sum()
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="already back-propagated|consumed"):
        loss.backward()
    with pytest.raises(ValueError, match="shape"):
        net(x, hidden_state=[(h0[:, :8], c0)])
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        net(x, hidden_state=[(h0.detach().cpu(), c0)])
    with pytest.raises(TypeError, match="float32"):
        net(x, hidden_state=[(h0.detach().to(torch.bfloat16), c0)])
    with pytest.raises(ValueError, match="pairs"):
        net(x, hidden_state=[(h0, c0), (h0, c0)])
    plan = net.plan_for(x, True)                         # a training plan without NINT_FLAG_STATE_GRAD
    plan.forward(x)
    with pytest.raises(RuntimeError, match="NINT_FLAG_STATE_GRAD"):
        plan.backward(torch.ones(B, 1, H, W, device="cuda"), dh_T=[torch.ones(B, 16, H, W, device="cuda")])
    plan.backward(torch.ones(B, 1, H, W, device="cuda"))
    with pytest.raises(RuntimeError, match="NINT_FLAG_STATE_GRAD"):
        plan.backward_initial_state()
