"""GPU (B200): bit-exact checks of the gate conv, dgrad, wgrad and BPTT kernels on integer-lattice inputs.

The cases (oracle/lattice.py) make every product exact and every partial sum representable in fp32, so the correct
result is unique whatever the accumulation order, split-K factor, tile walk or atomics; test_lattice_oracle.py proves
that on the CPU for every case here.  Every asserted tensor must therefore equal the fp64 reference with torch.equal:
a dropped, duplicated or misplaced term fails with no tolerance to argue about.
  A: the forward implicit GEMM (Plan.debug_raw_gates) against an fp64 conv2d.
  B: one cell step, forward and backward (Plan.cell_forward / cell_backward), deterministic and atomic reductions.
  C: the module's whole BPTT in the zero state, under every schedule: time-fused and per-step launches, sub-batches,
     frame-bank windows, return_sequence, x.grad and the staged backward."""
import functools

import pytest
import torch

from oracle import lattice as Lt

pytestmark = pytest.mark.gpu

CASES = dict(Lt.suite_cases())


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists)")
    prev = torch.backends.cudnn.deterministic
    yield
    torch.backends.cudnn.deterministic = prev


@functools.lru_cache(maxsize=None)
def _ref(cid):
    return Lt.reference(CASES[cid])


def _cu(t):
    return t.float().cuda()


def _assert_exact(got, ref, tag=""):
    for k, v in got.items():
        assert torch.equal(v.detach().cpu().double(), ref[k]), f"{tag} {k}: {int((v.detach().cpu().double() != ref[k]).sum())} " \
                                                               f"elements differ, max |diff| {float((v.detach().cpu().double() - ref[k]).abs().max()):.3e}"


# ------------------------------------------------------------------------------------------------ runners
def run_gate_conv(case):
    from nasa_niswan_b200 import Plan
    B, C, H, W, hc, k = case["B"], case["C"], case["H"], case["W"], case["hidden"][0], case["ks"][0]
    plan = Plan(B, 1, H, W, C, [hc], [k], precision=case["precision"])
    plan.set_weights(0, _cu(case["w"]), None)
    plan.set_head(torch.zeros(1, hc, 1, 1, device="cuda"), torch.zeros(1, device="cuda"))
    h0 = _cu(case["h0"])
    plan.set_state(0, h0, torch.zeros_like(h0))
    return {"gates": plan.debug_raw_gates(_cu(case["x"]))}


def run_cell(case, deterministic):
    from nasa_niswan_b200 import Plan
    B, C, H, W, hc, k = case["B"], case["C"], case["H"], case["W"], case["hidden"][0], case["ks"][0]
    plan = Plan(B, 1, H, W, C, [hc], [k], precision=case["precision"], training=True, input_grad=True,
                deterministic=deterministic)
    plan.set_weights(0, _cu(case["w"]), _cu(case["bias"]))
    plan.set_head(torch.zeros(1, hc, 1, 1, device="cuda"), torch.zeros(1, device="cuda"))
    h, c = plan.cell_forward(_cu(case["x"][:, 0]), _cu(case["h0"]), _cu(case["c0"]))
    dx, dh, dc, gw, gb = plan.cell_backward(_cu(case["dh_out"]), _cu(case["dc_out"]))
    return dict(c=c, h=h[:, case["h_mask"].cuda()], dx=dx, dh=dh, dc=dc, gw=gw, gb=gb)


def _net(case):
    from nasa_niswan_b200 import ConvLSTM
    L = len(case["hidden"])
    net = ConvLSTM(case["C"], case["hidden"], case["ks"], L, precision=case["precision"],
                   return_sequence=case["return_sequence"])
    with torch.no_grad():
        for l in range(L):
            net.layers[l].conv.weight.copy_(case["ws"][l].float())
            net.layers[l].conv.bias.copy_(case["bs"][l].float())
        net.conv.weight.copy_(case["hw"].float())
        net.conv.bias.copy_(case["hb"].float())
    return net.cuda()


def _grads(net, out):
    for l, cell in enumerate(net.layers):
        out[f"gw{l}"], out[f"gb{l}"] = cell.conv.weight.grad, cell.conv.bias.grad
    out["ghw"], out["ghb"] = net.conv.weight.grad, net.conv.bias.grad
    return out


def run_bptt(case, deterministic, need_dx=False, bank=False):
    """module forward + backward of the case's dpred (and dseq); bank: the windows are cut out of a frame bank"""
    prev = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = deterministic        # the module's switch for fixed-order reductions
    try:
        net = _net(case)
        x = _cu(case["x"])
        if bank:       # overlapping windows: consecutive samples read T-1 shared frames through the bank's descriptors
            from nasa_niswan_b200.preprocess import FrameBank
            bank_ = FrameBank.from_frames(_cu(case["frames"]), case["precision"])
            res = net.forward_windows(bank_, case["starts"], case["T"])
        else:
            x.requires_grad_(need_dx)
            res = net(x)
        pred, seq = res if case["return_sequence"] else (res, None)
        if seq is not None:
            torch.autograd.backward([pred, seq], [_cu(case["dpred"]), _cu(case["dseq"])])
        else:
            pred.backward(_cu(case["dpred"]))
        torch.cuda.synchronize()
    finally:
        torch.backends.cudnn.deterministic = prev
    out = {"pred": pred}
    if seq is not None:
        out["seq"] = seq
    if need_dx and not bank:
        out["dx"] = x.grad
    return _grads(net, out)


def run_staged(case):
    """Plan.backward(on_ready=...): BPTT, then one wgrad call per layer, top layer first"""
    from nasa_niswan_b200 import Plan
    B, T, C, H, W = case["B"], case["T"], case["C"], case["H"], case["W"]
    L = len(case["hidden"])
    plan = Plan(B, T, H, W, C, case["hidden"], case["ks"], precision=case["precision"], training=True)
    for l in range(L):
        plan.set_weights(l, _cu(case["ws"][l]), _cu(case["bs"][l]))
    plan.set_head(_cu(case["hw"]), _cu(case["hb"]))
    pred, _ = plan.forward(_cu(case["x"]))
    order = []
    gw, gb, ghw, ghb = plan.backward(_cu(case["dpred"]), on_ready=order.append)
    assert order == list(range(L, -1, -1))
    out = {"pred": pred, "ghw": ghw, "ghb": ghb}
    for l in range(L):
        out[f"gw{l}"], out[f"gb{l}"] = gw[l], gb[l]
    return out


# ------------------------------------------------------------------------------------------------ A, B
@pytest.mark.parametrize("cid", [c for c in CASES if c.startswith("A-")])
def test_gate_conv_is_exact(cid):
    """halos, every tap, K chunks (chunk edges at 15/16/17 tf32 and 31/32/33 bf16 channels), n-blocks and the q-order
    column permutation of the forward implicit GEMM"""
    _assert_exact(run_gate_conv(CASES[cid]), _ref(cid))


@pytest.mark.parametrize("cid", [c for c in CASES if c.startswith("B-")])
def test_cell_step_is_exact(cid):
    """every gate row of dgates, dgrad into x and h, wgrad with the ones-lane bias, deterministic and atomic wgrad"""
    ref = _ref(cid)
    ref = dict(ref, h=ref["h"][:, CASES[cid]["h_mask"]])
    for det in (True, False):
        _assert_exact(run_cell(CASES[cid], det), ref, "deterministic" if det else "atomic")


# ------------------------------------------------------------------------------------------------ C
C_IDS = [c for c in CASES if c.startswith("C-") and not c.endswith("cfg2_b32")]


@pytest.mark.parametrize("cid", C_IDS)
def test_bptt_is_exact(cid):
    """deterministic reductions with x.grad (input-gradient plan), then atomic reductions without"""
    ref = _ref(cid)
    _assert_exact(run_bptt(CASES[cid], True, need_dx=True), ref, "deterministic")
    _assert_exact(run_bptt(CASES[cid], False), ref, "atomic")


@pytest.mark.parametrize("fuse", [None, "3"], ids=["default_rule", "fused"])
def test_cfg2_full_batch_is_exact(monkeypatch, fuse):
    """BASELINE cfg 2 at B=32 (90x144, bf16): one launch per BPTT step under the default rule, one launch per layer
    with NINT_FUSE_STEPS=3; atomic (the training default) and deterministic reductions"""
    if fuse is None:
        monkeypatch.delenv("NINT_FUSE_STEPS", raising=False)
    else:
        monkeypatch.setenv("NINT_FUSE_STEPS", fuse)
    cid = "C-bf16-cfg2_b32"
    ref = _ref(cid)
    _assert_exact(run_bptt(CASES[cid], False), ref, "atomic")
    _assert_exact(run_bptt(CASES[cid], True), ref, "deterministic")


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
@pytest.mark.parametrize("variant", ["per_step_launches", "sub_batch", "frame_bank", "staged_backward"])
def test_schedules_are_exact(monkeypatch, variant, precision):
    """the schedules that the bit-identity tests only compare with each other, here against the exact result"""
    if variant == "per_step_launches":
        monkeypatch.setenv("NINT_FUSE_STEPS", "0")
        for name in ("h64_k3_33x9_T4", "h32_h16_k3_k5_17x13"):
            cid = f"C-{precision}-{name}"
            _assert_exact(run_bptt(CASES[cid], False, need_dx=True), _ref(cid), name)
    elif variant == "sub_batch":
        monkeypatch.setenv("NINT_SUB_BATCH", "2")
        cid = f"C-{precision}-b40_40x36_T4"
        _assert_exact(run_bptt(CASES[cid], True), _ref(cid))
    elif variant == "frame_bank":
        cid = f"C-{precision}-h64_k3_33x9_T4"
        _assert_exact(run_bptt(CASES[cid], False, bank=True), _ref(cid))
    else:
        cid = f"C-{precision}-h128_h64_k3_12x20"
        _assert_exact(run_staged(CASES[cid]), _ref(cid))
