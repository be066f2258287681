"""GPU (B200): input gradients of frame-bank windows (FrameBank.requires_grad_ -> bank.grad) and the adjoint of the fused
preprocessing (nint_fuse_inputs_adjoint -> FrameBank.field_grads, differentiable preprocess.fuse_inputs).

bank.grad must equal, bit for bit, the (t, b)-ordered scatter of x.grad of the same windows cut out as an explicit
tensor: both come from the same dgrad dumps, and the accumulation kernel adds them in that order.  The adjoint kernel must
equal the CPU reference of oracle/adjoint_oracle.py bit for bit.  The whole pipeline (raw fields -> bank -> model ->
field gradients) is compared with autograd of the torch restatement of the preprocessing followed by the fp32 oracle,
at the project's bars: max|a-b| / max|b| <= 1e-3 (tf32) / <= 2e-2 (bf16)."""
import functools

import numpy as np
import pytest
import torch

from oracle import convlstm_oracle as O
from oracle import lattice as Lt
from oracle.adjoint_oracle import fuse_adjoint_reference, fuse_inputs_torch, scatter_windows

pytestmark = pytest.mark.gpu

TOL = {"tf32": 1e-3, "bf16": 2e-2}
PRECISIONS = ["bf16", "tf32"]


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists)")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    prev = torch.backends.cudnn.deterministic
    yield
    torch.backends.cudnn.deterministic = prev


def _net(C, hidden, ks, precision, seed=0, **kw):
    from nasa_niswan_b200 import ConvLSTM
    torch.manual_seed(seed)
    net = ConvLSTM(C, hidden, ks, len(hidden), precision=precision, **kw)
    params = {k: v.detach().clone() for k, v in net.state_dict().items()}
    return net.cuda(), params


def _bank(frames, precision):
    from nasa_niswan_b200.preprocess import FrameBank
    return FrameBank.from_frames(frames, precision).requires_grad_()


def _upstream(out, seed=5):
    g = torch.Generator(device="cuda").manual_seed(seed)
    outs = list(out) if isinstance(out, tuple) else [out]
    return outs, [torch.randn(o.shape, generator=g, device="cuda") for o in outs]


# ------------------------------------------------------------------------------------------------ bank.grad == scatter
# (C, hidden, ks, B, T, H, W, starts, n_frames, return_sequence, stateful)
SCATTER_CASES = {
    "overlap_repeated_start": (21, [64], [3], 4, 4, 17, 20, [0, 2, 2, 5], 10, False, False),
    "return_sequence_two_layers": (9, [32, 16], [3, 5], 3, 3, 13, 16, [1, 0, 3], 7, True, False),
    "padded_hidden": (5, [20], [3], 2, 3, 12, 20, [0, 1], 5, False, False),
    "shipped_geometry_small": (5, [64, 32, 16], [5, 3, 3], 2, 6, 20, 24, [0, 2], 9, False, False),
    "stateful": (7, [32], [3], 2, 4, 16, 16, [3, 1], 8, False, True),
}


def _bank_vs_explicit(case, precision, deterministic):
    C, hidden, ks, B, T, H, W, starts, N, seq, stateful = case
    torch.backends.cudnn.deterministic = deterministic
    try:
        net, _ = _net(C, hidden, ks, precision, return_sequence=seq)
        torch.manual_seed(9)
        frames = torch.randn(N, C, H, W, device="cuda")
        state = None
        if stateful:
            g = torch.Generator().manual_seed(3)
            state = [(torch.randn(B, hc, H, W, generator=g).cuda() * 0.5, torch.randn(B, hc, H, W, generator=g).cuda() * 0.5)
                     for hc in hidden]
        bank = _bank(frames, precision)
        kw = dict(hidden_state=state, return_state=True) if stateful else {}
        out = net.forward_windows(bank, torch.tensor(starts), T, **kw)
        outs, gs = _upstream(out[0] if stateful else out)
        torch.autograd.backward(outs, gs)
        x = torch.stack([frames[s:s + T] for s in starts]).requires_grad_()
        out = net(x, **kw)
        outs2, _ = _upstream(out[0] if stateful else out)
        for a, b in zip(outs, outs2):
            assert torch.equal(a, b)
        torch.autograd.backward(outs2, gs)
        torch.cuda.synchronize()
    finally:
        torch.backends.cudnn.deterministic = False
    return bank.grad.cpu(), scatter_windows(x.grad.cpu(), starts, N)


@pytest.mark.parametrize("fuse", ["0", "3"])
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", list(SCATTER_CASES))
def test_bank_grad_is_the_ordered_scatter_of_x_grad(monkeypatch, name, precision, fuse):
    """overlapping windows with a repeated start, return_sequence, a padded hidden size, the shipped 3-layer geometry at a
    small size and a stateful call: deterministic reductions first, then atomic ones (no atomics feed dgates or dx)"""
    monkeypatch.setenv("NINT_FUSE_STEPS", fuse)
    for det in (True, False):
        got, ref = _bank_vs_explicit(SCATTER_CASES[name], precision, det)
        assert torch.equal(got, ref), f"deterministic={det}: {int((got != ref).sum())} elements differ"


@pytest.mark.parametrize("precision", PRECISIONS)
def test_bank_grad_is_exact_on_the_lattice_case(precision):
    """the frame-bank lattice case (overlapping windows of one record): bank.grad equals the fp64 scatter of the exact dx"""
    cid = f"C-{precision}-h64_k3_33x9_T4"
    case = dict(Lt.suite_cases())[cid]
    ref = Lt.reference(case)
    net, _ = _net(case["C"], case["hidden"], case["ks"], precision)
    with torch.no_grad():
        net.layers[0].conv.weight.copy_(case["ws"][0].float())
        net.layers[0].conv.bias.copy_(case["bs"][0].float())
        net.conv.weight.copy_(case["hw"].float())
        net.conv.bias.copy_(case["hb"].float())
    bank = _bank(case["frames"].float().cuda(), precision)
    pred = net.forward_windows(bank, case["starts"], case["T"])
    pred.backward(case["dpred"].float().cuda())
    want = scatter_windows(ref["dx"], case["starts"].tolist(), case["frames"].shape[0])
    assert torch.equal(bank.grad.cpu().double(), want)


# ------------------------------------------------------------------------------------------------ adjoint kernel
ADJ_SHAPES = [(3, 2, 0, 7, 9, 7, 9), (2, 1, 0, 8, 10, 12, 16), (3, 2, 2, 9, 11, 12, 14), (2, 1, 1, 5, 5, 13, 13),
              (2, 0, 3, 6, 8, 9, 11), (4, 4, 0, 90, 144, 100, 154)]


@pytest.mark.parametrize("mode", ["reflect", "reference_rnn"])
@pytest.mark.parametrize("shape", ADJ_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_adjoint_kernel_equals_the_ordered_reference(shape, mode):
    from nasa_niswan_b200.preprocess import fuse_inputs_adjoint
    N, L, S, H, W, Hp, Wp = shape
    g = torch.Generator().manual_seed(2)
    d = torch.randn(N, L + 1 + S, Hp, Wp, generator=g)
    std = torch.rand(L + 1, generator=g) + 0.3
    got = fuse_inputs_adjoint(d.cuda(), std.cuda(), L, S, H, W, mode)
    ref = fuse_adjoint_reference(d, std, L, S, H, W, mode)
    for k in ("levels3d", "emis2d", "statics"):
        if ref[k] is None:
            assert got[k] is None
        else:
            assert torch.equal(got[k].cpu(), ref[k]), k
    part = fuse_inputs_adjoint(d.cuda(), std.cuda(), L, S, H, W, mode, want=(False, True, False))
    assert part["levels3d"] is None and part["statics"] is None and torch.equal(part["emis2d"].cpu(), ref["emis2d"])


# ------------------------------------------------------------------------------------------------ whole pipeline
def _raw_fields(N, L, H, W, seed):
    rng = np.random.default_rng(seed)
    lev = rng.standard_normal((N, L, H, W)).astype(np.float32) * 2 + 0.5
    emis = np.abs(rng.standard_normal((N, H, W))).astype(np.float32)
    mean, std = rng.standard_normal(L + 1).astype(np.float32), (rng.random(L + 1) + 0.5).astype(np.float32)
    return lev, emis, mean, std


# name: (L, H, W, Hp, Wp, N, T, starts, hidden, ks, mode)
PIPELINES = {
    "shipped_reference_rnn": (4, 90, 144, 100, 154, 50, 48, [0, 2], [64, 32, 16], [5, 3, 3], "reference_rnn"),
    "cfg2_reflect": (20, 80, 134, 90, 144, 8, 4, [0, 3], [64], [3], "reflect"),
}


@functools.lru_cache(maxsize=None)
def _oracle_field_grads(name):
    L, H, W, Hp, Wp, N, T, starts, hidden, ks, mode = PIPELINES[name]
    lev, emis, mean, std = _raw_fields(N, L, H, W, 3)
    _, params = _net(L + 1, hidden, ks, "tf32")
    lev_t, emis_t = torch.from_numpy(lev).requires_grad_(), torch.from_numpy(emis).requires_grad_()
    frames = fuse_inputs_torch(lev_t, emis_t, torch.from_numpy(mean), torch.from_numpy(std), (Hp, Wp), mode)
    assert torch.equal(frames.detach(), torch.from_numpy(O.fuse_inputs(lev, emis, mean, std, (Hp, Wp), mode)))
    x = torch.stack([frames[s:s + T] for s in starts])
    pred = O.convlstm_forward(x, params, len(hidden))
    dpred = torch.randn(pred.shape, generator=torch.Generator().manual_seed(8))
    pred.backward(dpred)
    return (lev, emis, mean, std), dpred, lev_t.grad, emis_t.grad


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", list(PIPELINES))
def test_field_grads_against_the_oracle(name, precision):
    """raw fields -> FrameBank.from_fields -> forward_windows -> a fixed upstream gradient -> field_grads(), against
    autograd of the torch restatement of the preprocessing followed by the fp32 oracle ConvLSTM"""
    from nasa_niswan_b200.preprocess import FrameBank
    L, H, W, Hp, Wp, N, T, starts, hidden, ks, mode = PIPELINES[name]
    (lev, emis, mean, std), dpred, ref_lev, ref_emis = _oracle_field_grads(name)
    net, _ = _net(L + 1, hidden, ks, precision)
    for p in net.parameters():
        p.requires_grad_(False)
    cu = lambda a: torch.from_numpy(a).cuda()
    bank = FrameBank.from_fields(cu(lev), cu(emis), cu(mean), cu(std), (Hp, Wp), mode, None, precision).requires_grad_()
    net.forward_windows(bank, torch.tensor(starts), T).backward(dpred.cuda())
    got = bank.field_grads()
    e_lev = O.max_abs_normalised(got["levels3d"].cpu(), ref_lev)
    e_emis = O.max_abs_normalised(got["emis2d"].cpu(), ref_emis)
    print(f"{name} {precision}: levels3d {e_lev:.2e}, emis2d {e_emis:.2e}")
    assert e_lev < TOL[precision] and e_emis < TOL[precision] and got["statics"] is None


@pytest.mark.parametrize("precision", PRECISIONS)
def test_explicit_route_matches_field_grads(precision):
    """fuse_inputs (differentiable) -> windows as a tensor -> model(x) -> levels3d.grad equals field_grads() of the bank
    route up to the order in which the frames' window terms are summed"""
    from nasa_niswan_b200.preprocess import FrameBank, fuse_inputs
    L, H, W, Hp, Wp, N, T, starts, mode = 3, 20, 30, 26, 36, 9, 4, [0, 2, 2, 5], "reference_rnn"
    lev, emis, mean, std = (torch.from_numpy(a).cuda() for a in _raw_fields(N, L, H, W, 4))
    g = torch.Generator().manual_seed(6)
    statics = torch.randn(2, H, W, generator=g).cuda()
    net, _ = _net(L + 3, [32], [3], precision)
    bank = FrameBank.from_fields(lev, emis, mean, std, (Hp, Wp), mode, statics, precision).requires_grad_()
    dpred = torch.randn(len(starts), 1, Hp, Wp, generator=g).cuda()
    net.forward_windows(bank, torch.tensor(starts), T).backward(dpred)
    want = bank.field_grads()
    lev_g, emis_g, st_g = (t.clone().requires_grad_() for t in (lev, emis, statics))
    frames = fuse_inputs(lev_g, emis_g, mean, std, (Hp, Wp), mode, st_g)
    with torch.no_grad():
        assert torch.equal(frames, fuse_inputs(lev, emis, mean, std, (Hp, Wp), mode, statics))
    net(torch.stack([frames[s:s + T] for s in starts])).backward(dpred)
    for k, t in (("levels3d", lev_g), ("emis2d", emis_g), ("statics", st_g)):
        err = float((t.grad - want[k]).abs().max()) / float(want[k].abs().max())
        assert err <= 1e-5, f"{k}: {err:.2e}"


# ------------------------------------------------------------------------------------------------ semantics
def _setup(precision="bf16", frozen=False, starts=(0, 4, 8), N=16, T=4):
    net, _ = _net(8, [32], [3], precision)
    if frozen:
        for p in net.parameters():
            p.requires_grad_(False)
    torch.manual_seed(1)
    frames = torch.randn(N, 8, 16, 24, device="cuda")
    return net, _bank(frames, precision), torch.tensor(list(starts)), T


def _step(net, bank, starts, T, seed=5):
    pred = net.forward_windows(bank, starts, T)
    pred.backward(_upstream(pred, seed)[1][0])


def test_accumulation_zeroing_coverage_and_determinism():
    """windows that do not overlap, so every frame gets one term per backward: two backwards give exactly twice one;
    zero_grad clears; frames no window covers stay 0; two identical runs are bit-identical"""
    net, bank, starts, T = _setup()
    _step(net, bank, starts, T)
    one = bank.grad.clone()
    assert bool(one[:12].abs().amax((1, 2, 3)).gt(0).all()) and bool((one[12:] == 0).all())
    _step(net, bank, starts, T)
    assert torch.equal(bank.grad, 2 * one)
    bank.zero_grad()
    assert bool((bank.grad == 0).all())
    _step(net, bank, starts, T)
    assert torch.equal(bank.grad, one)


def test_frozen_model_still_fills_the_bank_gradient_and_no_grad_collects_nothing():
    net, bank, starts, T = _setup(frozen=True)
    _step(net, bank, starts, T)
    assert float(bank.grad.abs().max()) > 0
    assert all(p.grad is None for p in net.parameters())
    before = bank.grad.clone()
    with torch.no_grad():
        pred = net.forward_windows(bank, starts, T)
    assert not pred.requires_grad and torch.equal(bank.grad, before)
    bank.requires_grad_(False)         # a bank without gradients takes the existing op
    assert not net.forward_windows(bank, starts, T).requires_grad and bank.grad is None


def test_input_sensitivity_restores_the_bank_state():
    from nasa_niswan_b200.preprocess import FrameBank
    from nasa_niswan_b200.utils import input_sensitivity
    L, H, W, Hp, Wp, N, T = 4, 90, 144, 100, 154, 12, 4
    lev, emis, mean, std = (torch.from_numpy(a).cuda() for a in _raw_fields(N, L, H, W, 7))
    net, _ = _net(L + 1, [16], [3], "bf16")
    bank = FrameBank.from_fields(lev, emis, mean, std, (Hp, Wp), "reference_rnn")
    sens = input_sensitivity(net, bank, torch.tensor([0, 4]), T, y_std=2.0)
    assert not bank.requires_grad and all(p.grad is None for p in net.parameters())
    assert sens["levels3d"].shape == (N, L, H, W) and float(sens["emis2d"][:8].abs().max()) > 0
    assert bool((sens["emis2d"][8:] == 0).all())
    half = input_sensitivity(net, bank, torch.tensor([0, 4]), T, y_std=1.0)
    assert torch.equal(half["emis2d"] * 2, sens["emis2d"])


def test_cuda_graph_replays_accumulate():
    """forward + backward with bank gradients captured in one CUDA graph: two replays give twice one replay (no host
    synchronisation on the path)"""
    net, bank, starts, T = _setup(frozen=True)
    starts = starts.to("cuda", torch.int32)
    gpred = torch.randn(3, 1, 16, 24, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            net.forward_windows(bank, starts, T).backward(gpred)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        net.forward_windows(bank, starts, T).backward(gpred)
    bank.zero_grad()
    graph.replay()
    torch.cuda.synchronize()
    one = bank.grad.clone()
    assert float(one.abs().max()) > 0
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(bank.grad, 2 * one)
    bank.zero_grad()
    net.forward_windows(bank, starts, T).backward(gpred)     # eager: the same as one replay
    assert torch.equal(bank.grad, one)


# ------------------------------------------------------------------------------------------------ refusals
def test_refusals():
    from nasa_niswan_b200 import Plan
    from nasa_niswan_b200 import _lib
    from nasa_niswan_b200.preprocess import FrameBank
    B, T, C, H, W, N = 2, 3, 8, 12, 16, 6
    lib = _lib.load()
    torch.manual_seed(0)
    frames = torch.randn(N, C, H, W, device="cuda")
    bank = FrameBank.from_frames(frames, "bf16")
    starts = torch.tensor([0, 2], dtype=torch.int32, device="cuda")
    dframes = torch.zeros(N, C, H, W, device="cuda")
    net, _ = _net(C, [16], [3], "bf16")

    def plan(input_grad):
        p = Plan(B, T, H, W, C, [16], [3], training=True, input_grad=input_grad)
        for l, cell in enumerate(net.layers):
            p.set_weights(l, cell.conv.weight, cell.conv.bias)
        p.set_head(net.conv.weight, net.conv.bias)
        return p

    def abi(p, target):
        stream = _lib.stream_ptr(p.device)
        rc = lib.nint_backward_input_bank(p._h, _lib.ptr(target), stream)
        return rc, lib.nint_last_error().decode()

    p = plan(False)                                                  # no NINT_FLAG_INPUT_GRAD
    pred, _ = p.forward_bank(bank.frames, starts)
    p.backward(torch.ones_like(pred))
    rc, msg = abi(p, dframes)
    assert rc != 0 and "NINT_FLAG_INPUT_GRAD" in msg
    p = plan(True)
    pred, _ = p.forward_bank(bank.frames, starts)
    rc, msg = abi(p, dframes)                                        # before BPTT
    assert rc != 0 and "before nint_backward_bptt" in msg
    p.backward(torch.ones_like(pred))
    rc, msg = abi(p, None)                                           # null dframes
    assert rc != 0 and "null dframes" in msg
    assert abi(p, dframes)[0] == 0 and float(dframes.abs().max()) > 0
    pred, _ = p.forward(torch.randn(B, T, C, H, W, device="cuda"))  # last forward not a bank forward
    p.backward(torch.ones_like(pred))
    rc, msg = abi(p, dframes)
    assert rc != 0 and "frame bank" in msg
    with pytest.raises(RuntimeError, match="frame bank"):
        p.backward_input_bank(dframes)
    with pytest.raises(RuntimeError, match="bank.grad"):
        bank.requires_grad_().field_grads()
    with pytest.raises(RuntimeError, match="requires_grad_"):
        FrameBank.from_fields(torch.randn(N, 1, H, W, device="cuda"), torch.randn(N, H, W, device="cuda"),
                              torch.zeros(2, device="cuda"), torch.ones(2, device="cuda")).field_grads()
    torch.cuda.synchronize()
