"""GPU (B200): parity of the CUDA path, called through the C ABI, against the CPU oracle and the
reference-generated golden vectors.  Metric and thresholds: SURVEY.md section 8d -- max|a-b| / max|b|
with b the fp32 oracle; <= 1e-3 in tf32 mode, <= 2e-2 in bf16 mode (north star)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import convlstm_oracle as O
from oracle.golden import load_case

pytestmark = pytest.mark.gpu

TOL = {"tf32": 1e-3, "bf16": 2e-2}
CASES = ["lstm_c21_h32_k3", "lstm_3layer_k533", "lstm_c8_h16_k5"]


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists)")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _load(golden_dir, name):
    z = load_case(golden_dir, name)
    meta = z["meta"].tolist()
    B, T, cin, H, W, L = meta[:6]
    hidden, ks = meta[6:6 + L], meta[6 + L:6 + 2 * L]
    crop = z["crop"].tolist()
    return z, dict(B=B, T=T, cin=cin, H=H, W=W, L=L, hidden=hidden, ks=ks, crop=None if crop[0] < 0 else tuple(crop))


def _net(z, m, precision, **kw):
    from nasa_niswan_b200 import ConvLSTM
    net = ConvLSTM(m["cin"], m["hidden"], m["ks"], m["L"], precision=precision, **kw).cuda()
    net.load_state_dict({k[6:]: torch.from_numpy(z[k]) for k in z if k.startswith("param/")})
    return net


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
@pytest.mark.parametrize("shape", [(1, 21, 64, 3, 7, 18), (2, 21, 64, 3, 20, 24), (3, 8, 16, 5, 11, 13),
                                   (2, 21, 128, 3, 20, 24), (2, 5, 32, 5, 18, 22), (1, 21, 64, 3, 90, 144)])
def test_gate_conv_matches_conv2d(precision, shape):
    """the implicit GEMM alone (TMA zero-fill padding, two K segments, UMMA descriptors)"""
    from nasa_niswan_b200 import Plan
    B, C, hc, k, H, W = shape
    torch.manual_seed(1)
    x = torch.randn(B, 1, C, H, W, device="cuda")
    w = torch.randn(4 * hc, C + hc, k, k, device="cuda") * 0.1
    h0 = torch.randn(B, hc, H, W, device="cuda") * 0.5
    plan = Plan(B, 1, H, W, C, [hc], [k], precision=precision)
    plan.set_weights(0, w, None)
    plan.set_head(torch.zeros(1, hc, 1, 1, device="cuda"), torch.zeros(1, device="cuda"))
    plan.set_state(0, h0, torch.zeros_like(h0))
    got = plan.debug_raw_gates(x)
    ref = F.conv2d(torch.cat([x[:, 0], h0], 1).double().cpu(), w.double().cpu(), None, padding=k // 2)  # fp64 on the CPU
    assert O.max_abs_normalised(got.cpu(), ref) < TOL[precision]


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
@pytest.mark.parametrize("name", CASES)
def test_cell_step_matches_golden(golden_dir, name, precision):
    """ConvLSTMCell.forward with non-zero state (model.py:216-231) against the reference's output"""
    from nasa_niswan_b200 import ConvLSTMCell
    z, m = _load(golden_dir, name)
    cell = ConvLSTMCell(m["cin"], m["hidden"][0], m["ks"][0], precision=precision).cuda()
    cell.conv.weight.data.copy_(torch.from_numpy(z["param/layers.0.conv.weight"]))
    cell.conv.bias.data.copy_(torch.from_numpy(z["param/layers.0.conv.bias"]))
    with torch.no_grad():
        h1, c1 = cell(torch.from_numpy(z["cell/x"]).cuda(),
                      (torch.from_numpy(z["cell/h0"]).cuda(), torch.from_numpy(z["cell/c0"]).cuda()))
    assert O.max_abs_normalised(h1.cpu(), z["cell/h1"]) < TOL[precision]
    assert O.max_abs_normalised(c1.cpu(), z["cell/c1"]) < TOL[precision]


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
@pytest.mark.parametrize("name", CASES)
def test_forward_backward_matches_golden(golden_dir, name, precision):
    """ConvLSTM forward + MSE+L1 loss + BPTT (train.py:96-109) against the reference's autograd"""
    z, m = _load(golden_dir, name)
    net = _net(z, m, precision)
    x, y = torch.from_numpy(z["x"]).cuda(), torch.from_numpy(z["y"]).cuda()
    with torch.no_grad():
        pred_inf = net(x)                       # inference plan (2-slot ring, no saved gates)
    pred = net(x)                               # training plan
    assert pred.shape == (m["B"], 1, m["H"], m["W"])
    assert O.max_abs_normalised(pred.detach().cpu(), z["pred"]) < TOL[precision]
    assert torch.equal(pred_inf, pred.detach())
    loss = O.training_loss(pred, y, m["crop"])
    loss.backward()
    assert abs(float(loss.detach()) - float(z["loss"])) < TOL[precision] * max(1.0, abs(float(z["loss"])))
    for k, p in net.named_parameters():
        assert p.grad is not None and p.grad.shape == p.shape
        assert O.max_abs_normalised(p.grad.cpu(), z["grad/" + k]) < TOL[precision], k


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
@pytest.mark.parametrize("ksize", [3, 5])
def test_twelve_step_rollout_against_oracle(precision, ksize):
    """north-star tolerance over a 12-step rollout on the 90x144 grid, 20 levels + emission channel.
    Forward: pred vs the oracle.  Backward: BPTT of the SAME upstream gradient -- d(MSE+L1)/dpred taken
    at the oracle's prediction -- because L1Loss's sign(pred - y) is discontinuous: a 1e-4 difference in
    pred flips the sign at a pixel or two and moves a weight gradient by ~2/sqrt(#pixels) ~ 1e-2, which
    says nothing about the kernels (measured: tests/tools/parity_report.py)."""
    from nasa_niswan_b200 import ConvLSTM
    torch.manual_seed(0)
    B, T, C, H, W, hc = 2, 12, 21, 90, 144, 64
    net = ConvLSTM(C, [hc], [ksize], 1, precision=precision)
    params = {k: v.detach().clone() for k, v in net.state_dict().items()}
    net = net.cuda()
    x, y = torch.randn(B, T, C, H, W), torch.randn(B, H, W)
    leaf = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    ref_pred = O.convlstm_forward(x, leaf, 1)
    dpred = torch.autograd.grad(O.training_loss(ref_pred, y), ref_pred, retain_graph=True)[0]
    ref_pred.backward(dpred)
    pred = net(x.cuda())
    assert O.max_abs_normalised(pred.detach().cpu(), ref_pred.detach()) < TOL[precision]
    pred.backward(dpred.cuda())
    for k, p in net.named_parameters():
        assert O.max_abs_normalised(p.grad.cpu(), leaf[k].grad) < TOL[precision], k


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
@pytest.mark.parametrize("cfg", [
    # (B, T, C, H, W, hidden, ksize): geometries that exercise the other kernel plans
    (2, 3, 21, 20, 24, [128], [3]),          # hidden > 64: several n-blocks per pixel tile, two 256-q wgrad blocks
    (2, 3, 5, 17, 13, [64, 64], [3, 3]),     # stacked layers with no padding lane (cin = 64), ragged 17x13 grid
    (3, 2, 21, 16, 40, [64], [5]),           # 5x5 taps: weights stream through stages (not resident), 25-tap wgrad groups
    (1, 4, 9, 33, 9, [32, 16], [3, 5]),      # small hidden sizes (single-CTA wgrad), odd tile counts, mixed k
    (1, 2, 21, 16, 16, [128, 128], [5, 5]),  # BASELINE cfg 5 in miniature: 256 wgrad columns per tap, 64-channel B panels, 2 B stages
    (1, 2, 9, 12, 20, [128, 64], [3, 3]),    # 128 + 64 channels: N/2 = 96 -> 32-channel B panels (SWIZZLE_64B)
], ids=["h128", "h64x2_ragged", "k5_stream", "h32_h16_mixed", "cfg5_like", "pw32"])
def test_plans_against_oracle(cfg, precision):
    """forward + BPTT against the CPU oracle for geometries whose shared-memory plans differ from the BASELINE one"""
    from nasa_niswan_b200 import ConvLSTM
    B, T, C, H, W, hidden, ks = cfg
    torch.manual_seed(3)
    net = ConvLSTM(C, hidden, ks, len(hidden), precision=precision)
    params = {k: v.detach().clone() for k, v in net.state_dict().items()}
    net = net.cuda()
    x, y = torch.randn(B, T, C, H, W), torch.randn(B, H, W)
    leaf = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    ref_pred = O.convlstm_forward(x, leaf, len(hidden))
    dpred = torch.autograd.grad(O.training_loss(ref_pred, y), ref_pred, retain_graph=True)[0]
    ref_pred.backward(dpred)
    pred = net(x.cuda())
    assert O.max_abs_normalised(pred.detach().cpu(), ref_pred.detach()) < TOL[precision]
    pred.backward(dpred.cuda())
    for k, p in net.named_parameters():
        assert O.max_abs_normalised(p.grad.cpu(), leaf[k].grad) < TOL[precision], k


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
@pytest.mark.parametrize("cfg", [
    (1, 1, 32, 8, 16, [64], [3]),            # one sample, one step, one exact tile; cin = 32: no spare channel -> ones-panel bias MMA at layer 0
    (2, 2, 40, 9, 17, [64], [3]),            # cin = 40 -> two x chunks, ones channel 40 in the second; grid one pixel past the tile in x and y
    (1, 2, 3, 12, 20, [192], [3]),           # 224 wgrad columns: one pair block in bf16, several single-CTA column blocks in tf32
    (1, 2, 3, 12, 20, [256], [3]),           # widest hidden size: 288 wgrad columns -> x-part and h-part column blocks
    (1, 2, 4, 10, 12, [16], [7]),            # 7x7 taps on a grid barely larger than the kernel
    (5, 2, 21, 8, 16, [64], [1]),            # 1x1 "convolution": no halo at all
], ids=["b1_t1_c32", "c40_ragged", "h192", "h256", "k7", "k1"])
def test_edge_geometries_against_oracle(cfg, precision):
    """forward + BPTT against the CPU oracle at the edges of the supported geometry, at the north-star bars (1e-3 tf32,
    2e-2 bf16) even though a gradient here is a short sum of 128..400 signed pixel-steps: in tf32 mode the bias gradient
    also receives the sum of the residuals that rounding the stored dgates to tf32 takes away (nint_kernels.h db_resid);
    until round 2 that rounding left the nearly cancelling bias sums at 1.4e-3..2.5e-3 and this test allowed 2e-3."""
    from nasa_niswan_b200 import ConvLSTM
    B, T, C, H, W, hidden, ks = cfg
    tol = TOL[precision]
    torch.manual_seed(5)
    net = ConvLSTM(C, hidden, ks, len(hidden), precision=precision)
    params = {k: v.detach().clone() for k, v in net.state_dict().items()}
    net = net.cuda()
    x, y = torch.randn(B, T, C, H, W), torch.randn(B, H, W)
    leaf = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    ref_pred = O.convlstm_forward(x, leaf, len(hidden))
    dpred = torch.autograd.grad(O.training_loss(ref_pred, y), ref_pred, retain_graph=True)[0]
    ref_pred.backward(dpred)
    pred = net(x.cuda())
    assert O.max_abs_normalised(pred.detach().cpu(), ref_pred.detach()) < tol
    pred.backward(dpred.cuda())
    for k, p in net.named_parameters():
        assert O.max_abs_normalised(p.grad.cpu(), leaf[k].grad) < tol, k


def test_staged_backward_matches_single_call():
    """nint_backward_bptt + nint_backward_wgrad per layer (what the overlapped all-reduce drives) == nint_backward;
    buckets are announced head first, then layers top-down; wgrad before BPTT is refused"""
    from nasa_niswan_b200 import Plan
    torch.manual_seed(6)
    B, T, C, H, W, hidden, ks = 2, 3, 5, 12, 20, [64, 32], [3, 3]
    plan = Plan(B, T, H, W, C, hidden, ks, precision="bf16", training=True)
    cin = C
    for l, (hc, k) in enumerate(zip(hidden, ks)):
        plan.set_weights(l, torch.randn(4 * hc, cin + hc, k, k, device="cuda") * 0.1, torch.randn(4 * hc, device="cuda") * 0.1)
        cin = hc
    plan.set_head(torch.randn(1, hidden[-1], 1, 1, device="cuda"), torch.zeros(1, device="cuda"))
    x = torch.randn(B, T, C, H, W, device="cuda")
    pred, _ = plan.forward(x)
    dpred = torch.randn_like(pred)
    with pytest.raises(RuntimeError, match="before nint_backward_bptt"):
        _lib_check_wgrad_first(plan)
    ref = plan.backward(dpred)
    pred2, _ = plan.forward(x)
    assert torch.equal(pred, pred2)
    order = []
    got = plan.backward(dpred, on_ready=order.append)
    assert order == [2, 1, 0]
    for a, b in zip([*ref[0], *ref[1], ref[2], ref[3]], [*got[0], *got[1], got[2], got[3]]):
        assert O.max_abs_normalised(b.cpu(), a.cpu()) < 1e-5      # fp32 atomics reorder sums only


def _lib_check_wgrad_first(plan):
    import ctypes
    from nasa_niswan_b200 import _lib
    g = torch.empty(4 * 64 * (5 + 64) * 9, device="cuda")
    b = torch.empty(4 * 64, device="cuda")
    _lib.check(plan.lib.nint_backward_wgrad(plan._h, 0, ctypes.c_void_p(g.data_ptr()), ctypes.c_void_p(b.data_ptr()),
                                            ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "nint_backward_wgrad")


def test_torch_library_op_contract():
    """the dispatcher op behind ConvLSTM.forward: schema, fake-tensor shapes and autograd registration check out
    (torch.library.opcheck), and calling it directly equals the module"""
    from nasa_niswan_b200 import ConvLSTM, ops
    torch.manual_seed(8)
    net = ConvLSTM(5, [16, 16], [3, 3], 2, precision="tf32").cuda()
    x = torch.randn(2, 3, 5, 12, 20, device="cuda")
    plan = net.plan_for(x, True, set_params=False)
    params = net._params()
    pid = ops.register_plan(plan)
    torch.library.opcheck(torch.ops.nint.convlstm_forward, (x, params, pid),
                          test_utils=("test_schema", "test_faketensor", "test_autograd_registration"))
    pred, seq = torch.ops.nint.convlstm_forward(x, params, pid)
    assert seq.numel() == 0 and pred.requires_grad
    assert torch.equal(pred.detach(), net(x).detach())
    del plan
    net.release_workspaces()
    with pytest.raises(RuntimeError, match="no longer exists"):
        torch.ops.nint.convlstm_forward(x, params, pid)


def test_long_inference_rollout_keeps_state_resident():
    """BASELINE cfg 4 in miniature: forward-only T = 40 rollout (2-slot h ring, c updated in place) vs the oracle"""
    from nasa_niswan_b200 import ConvLSTM
    torch.manual_seed(4)
    B, T, C, H, W, hc = 2, 40, 21, 24, 32, 64
    net = ConvLSTM(C, [hc], [3], 1, precision="tf32")
    params = {k: v.detach().clone() for k, v in net.state_dict().items()}
    net = net.cuda()
    x = torch.randn(B, T, C, H, W)
    with torch.no_grad():
        pred = net(x.cuda())
    ref = O.convlstm_forward(x, params, 1)
    assert O.max_abs_normalised(pred.cpu(), ref) < TOL["tf32"]


def test_return_sequence_variant(golden_dir):
    """commented-out variant model.py:264,272,274: (pred, hs[B,T,H,W]); grads flow through every step"""
    z, m = _load(golden_dir, CASES[0])
    net = _net(z, m, "tf32", return_sequence=True)
    x = torch.from_numpy(z["x"]).cuda()
    pred, seq = net(x)
    params = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    ref_pred, ref_seq = O.convlstm_forward(torch.from_numpy(z["x"]), params, m["L"], return_sequence=True)
    assert seq.shape == (m["B"], m["T"], m["H"], m["W"])
    assert O.max_abs_normalised(seq.detach().cpu(), ref_seq) < 1e-3
    assert torch.equal(seq[:, -1:].detach(), pred.detach())
    wts = torch.linspace(0.5, 1.5, m["T"]).view(1, -1, 1, 1)
    ((seq * wts.cuda()).sum() + pred.sum()).backward()
    leaf = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    rp, rs = O.convlstm_forward(torch.from_numpy(z["x"]), leaf, m["L"], return_sequence=True)
    ((rs * wts).sum() + rp.sum()).backward()
    for k, p in net.named_parameters():
        assert O.max_abs_normalised(p.grad.cpu(), leaf[k].grad) < 1e-3, k


def test_linearity_of_backward_at_full_size():
    """size-independent property at BASELINE cfg-2 geometry (B=32 is too slow for the oracle):
    gradients are linear in the upstream gradient -- grad(2*L) == 2*grad(L) and the workspace is
    reusable across steps (same input twice -> identical results)."""
    from nasa_niswan_b200 import ConvLSTM
    torch.manual_seed(0)
    net = ConvLSTM(21, [64], [3], 1, precision="bf16").cuda()
    x = torch.randn(8, 12, 21, 90, 144, device="cuda")
    g = {}
    for scale in (1.0, 2.0, 1.0):
        net.zero_grad(set_to_none=True)
        (net(x).square().mean() * scale).backward()
        g.setdefault(scale, []).append([p.grad.clone() for p in net.parameters()])
    for a, b in zip(g[1.0][0], g[2.0][0]):
        assert O.max_abs_normalised((2 * a).cpu(), b.cpu()) < 1e-4
    for a, b in zip(g[1.0][0], g[1.0][1]):
        assert O.max_abs_normalised(a.cpu(), b.cpu()) < 1e-4   # fp32 atomics reorder sums only


def test_stale_workspace_is_detected(golden_dir):
    z, m = _load(golden_dir, CASES[0])
    net = _net(z, m, "bf16")
    x = torch.from_numpy(z["x"]).cuda()
    p1 = net(x)
    net(x)
    with pytest.raises(RuntimeError, match="overwrote the ConvLSTM workspace"):
        p1.sum().backward()


@pytest.mark.parametrize("crop", [None, (5, 95, 5, 149)])
def test_fused_loss_matches_torch(crop):
    """nint_loss_mse_l1 = MSELoss + L1Loss on the cropped prediction (train.py:74-75,102,105): value and gradient"""
    import ctypes
    from nasa_niswan_b200 import _lib
    torch.manual_seed(5)
    B, H, W = 4, 100, 154
    y0, y1, x0, x1 = crop if crop else (0, H, 0, W)
    pred = torch.randn(B, 1, H, W, device="cuda", requires_grad=True)
    y = torch.randn(B, y1 - y0, x1 - x0, device="cuda")
    ref = O.training_loss(pred, y, crop)
    ref.backward()
    dpred, loss, stats = torch.empty_like(pred), torch.empty(1, device="cuda"), torch.zeros(8, device="cuda")
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(_lib.load().nint_loss_mse_l1(vp(pred.detach()), vp(y), B, H, W, y0, y1, x0, x1, vp(dpred), vp(loss), vp(stats), st),
               "nint_loss_mse_l1")
    assert abs(float(loss.detach()) - float(ref.detach())) < 1e-5 * max(1.0, abs(float(ref.detach())))
    assert torch.allclose(dpred, pred.grad, rtol=1e-5, atol=1e-9)
    # the two extra sums give R^2 (train.py:114) without leaving the device
    r2 = 1.0 - float(stats[0]) / (float(stats[3]) - float(stats[2]) ** 2 / y.numel())
    p = pred.detach()[:, 0, y0:y1, x0:x1]
    r2_ref = 1.0 - float(((p - y) ** 2).sum()) / float(((y - y.mean()) ** 2).sum())
    assert abs(r2 - r2_ref) < 1e-4


def test_native_adam_matches_torch():
    """nint_adam_step vs torch.optim.Adam(lr, betas=(0.5, 0.999)) (train.py:71) over several steps"""
    from nasa_niswan_b200.parallel import NativeAdam
    torch.manual_seed(6)
    shapes = [(64, 10, 3, 3), (64,), (1, 16, 1, 1), (1,)]
    ref_p = [torch.nn.Parameter(torch.randn(s, device="cuda")) for s in shapes]
    our_p = [torch.nn.Parameter(p.detach().clone()) for p in ref_p]
    flat_g = torch.zeros(sum(p.numel() for p in our_p), device="cuda")
    ours = NativeAdam(our_p, flat_g, lr=1e-3, betas=(0.5, 0.999))
    ref = torch.optim.Adam(ref_p, lr=1e-3, betas=(0.5, 0.999))
    for step in range(5):
        g = torch.randn_like(flat_g) * (10.0 ** (step - 2))
        flat_g.copy_(g)
        off = 0
        for p in ref_p:
            p.grad = g[off:off + p.numel()].view_as(p).clone()
            off += p.numel()
        versions = [p._version for p in our_p]
        ours.step()
        ref.step()
        assert all(p._version > v for p, v in zip(our_p, versions))   # in-place update is visible to autograd
    for a, b in zip(our_p, ref_p):
        assert torch.allclose(a, b, rtol=2e-5, atol=1e-7)
    sd = ours.state_dict()
    assert torch.allclose(sd["state"][0]["exp_avg"], ref.state_dict()["state"][0]["exp_avg"], rtol=1e-5, atol=1e-8)


def test_native_step_matches_autograd_step():
    """Trainer(native=True) (fused loss, BPTT into the flat buffer, one Adam kernel) follows Trainer(native=False)"""
    from nasa_niswan_b200 import ConvLSTM
    from nasa_niswan_b200.parallel import Trainer
    torch.manual_seed(7)
    x = torch.randn(2, 4, 21, 30, 40, device="cuda")
    y = torch.randn(2, 20, 30, device="cuda")
    losses = {}
    for native in (False, True):
        torch.manual_seed(8)
        net = ConvLSTM(21, [64], [3], 1, precision="tf32").cuda()
        tr = Trainer(net, lr=1e-3, betas=(0.5, 0.999), crop=(5, 25, 5, 35), native=native)
        losses[native] = [float(tr.step(x, y)) for _ in range(4)]
        losses[("w", native)] = net.layers[0].conv.weight.detach().clone()
    assert losses[True][0] == pytest.approx(losses[False][0], rel=1e-5)
    assert losses[True] == pytest.approx(losses[False], rel=2e-3)
    assert losses[True][-1] < losses[True][0] and losses[False][-1] < losses[False][0]   # both train (weights are
    # repacked every forward: torch's fused Adam does not bump parameter versions)
    assert O.max_abs_normalised(losses[("w", True)].cpu(), losses[("w", False)].cpu()) < 5e-3


@pytest.mark.parametrize("mode", ["reflect", "reference_rnn"])
@pytest.mark.parametrize("shape", [(3, 20, 90, 144, 100, 154), (2, 4, 12, 20, 22, 30), (1, 0, 9, 7, 9, 7)])
def test_fuse_inputs_matches_oracle(shape, mode):
    """preprocessing fusion kernel vs the oracle restatement of dataset.py:520-537 / 67-98: bit-exact (fp32 in, fp32 out)"""
    from nasa_niswan_b200.preprocess import fuse_inputs
    T, L, H, W, Hp, Wp = shape
    rng = np.random.default_rng(9)
    lev = rng.standard_normal((T, L, H, W)).astype(np.float32) * 7 + 3
    em = np.abs(rng.standard_normal((T, H, W))).astype(np.float32) * 1e-9
    mean = rng.standard_normal(L + 1).astype(np.float32)
    std = (np.abs(rng.standard_normal(L + 1)) + 0.5).astype(np.float32)
    std[-1] *= 1e-9
    ref = O.fuse_inputs(lev, em, mean, std, (Hp, Wp), mode)
    got = fuse_inputs(*(torch.from_numpy(a).cuda() for a in (lev, em, mean, std)), (Hp, Wp), mode)
    assert got.shape == ref.shape
    assert np.array_equal(got.cpu().numpy(), ref)


@pytest.mark.parametrize("mode", ["reflect", "reference_rnn"])
def test_fuse_inputs_with_static_attributes(mode):
    """dataset.py:100-122, 532-533: z-scored static fields appended to every frame before the halo (so the shipped
    dataset's channel flip in the latitude halo runs over dynamic AND static channels): bit-exact"""
    from nasa_niswan_b200.preprocess import fuse_inputs, normalise_static_attributes
    T, L, S, H, W, Hp, Wp = 3, 4, 3, 18, 24, 24, 32
    rng = np.random.default_rng(19)
    lev = rng.standard_normal((T, L, H, W)).astype(np.float32)
    em = np.abs(rng.standard_normal((T, H, W))).astype(np.float32)
    mean = rng.standard_normal(L + 1).astype(np.float32)
    std = (np.abs(rng.standard_normal(L + 1)) + 0.5).astype(np.float32)
    raw = (rng.standard_normal((S, H, W)) * 40 + 100).astype(np.float32)
    st = O.normalise_static_attributes(raw).astype(np.float32)
    ref = O.fuse_inputs(lev, em, mean, std, (Hp, Wp), mode, statics=st)
    got = fuse_inputs(*(torch.from_numpy(a).cuda() for a in (lev, em, mean, std)), (Hp, Wp), mode,
                      statics=torch.from_numpy(st).cuda())
    assert got.shape == ref.shape == (T, L + 1 + S, Hp, Wp)
    assert np.array_equal(got.cpu().numpy(), ref)
    dev = normalise_static_attributes(torch.from_numpy(raw).cuda()).cpu().numpy()
    assert np.allclose(dev, st, rtol=1e-5, atol=1e-5)


def test_fuse_inputs_rejects_oversized_halo():
    from nasa_niswan_b200.preprocess import fuse_inputs
    z = torch.zeros(1, 1, 4, 4, device="cuda")
    with pytest.raises(RuntimeError, match="larger than width"):
        fuse_inputs(z, z[:, 0], torch.zeros(2, device="cuda"), torch.ones(2, device="cuda"), (4, 20))


def test_val_loop_r2_matches_sklearn():
    """utils.py:52-75: mean per-batch sklearn r2_score on the cropped prediction, computed on the device here"""
    from sklearn.metrics import r2_score
    from nasa_niswan_b200 import ConvLSTM
    from nasa_niswan_b200.utils import val_loop
    torch.manual_seed(10)
    net = ConvLSTM(5, [16], [3], 1, precision="tf32").cuda()
    data = [(torch.randn(2, 3, 5, 100, 154), torch.randn(2, 90, 144)) for _ in range(2)]
    import argparse
    got = val_loop(argparse.Namespace(model="LSTM-E33OMA"), data, net)     # utils.py:52 signature, train.py:122 call
    assert abs(got - val_loop(None, data, net)) < 1e-5          # (the R^2 sums are reduced with fp32 atomics)
    ref = 0.0
    with torch.no_grad():
        for X, y in data:
            pred = net(X.cuda())[:, :, 5:95, 5:149].squeeze()
            ref += r2_score(y.numpy().flatten(), pred.cpu().numpy().flatten())
    assert abs(got - ref / len(data)) < 1e-4


def test_sensitivity_sweep_matches_notebook_loop():
    """test.ipynb:2430-2462: one-at-a-time +5 % perturbation of every input feature, cropped, de-normalised"""
    from nasa_niswan_b200 import ConvLSTM
    from nasa_niswan_b200.utils import sensitivity_sweep
    torch.manual_seed(12)
    net = ConvLSTM(5, [16], [3], 1, precision="tf32").cuda()
    data = [(torch.randn(2, 3, 5, 100, 154), torch.randn(2, 90, 144)) for _ in range(2)]
    got = sensitivity_sweep(data, net, num_features=5, perturbation=0.05, y_mean=2.0, y_std=3.0)
    assert got.shape == (5, 4, 90, 144)
    net.eval()
    with torch.no_grad():
        for i in range(5):
            k = 0
            for X, _ in data:
                Xp = X.clone()
                Xp[:, :, i] *= 1.05
                p = net(Xp.cuda())[:, :, 5:95, 5:149].squeeze(1).cpu() * 3.0 + 2.0
                assert torch.allclose(got[i, k:k + 2], p, rtol=1e-5, atol=1e-5)
                k += 2
    for X, _ in data:          # borrowed inputs are left as they were
        assert X.is_cpu


def test_trainer_step_lr_schedule():
    """train.py:72,120: StepLR stepped per epoch changes the learning rate the native Adam kernel uses"""
    from nasa_niswan_b200 import ConvLSTM
    from nasa_niswan_b200.parallel import Trainer
    torch.manual_seed(13)
    x, y = torch.randn(2, 2, 5, 20, 24, device="cuda"), torch.randn(2, 20, 24, device="cuda")
    net = ConvLSTM(5, [16], [3], 1, precision="tf32").cuda()
    ref = ConvLSTM(5, [16], [3], 1, precision="tf32").cuda()
    ref.load_state_dict(net.state_dict())
    tr = Trainer(net, lr=1e-2, betas=(0.5, 0.999), native=True, scheduler_config=(1, 0.5))
    tr_ref = Trainer(ref, lr=1e-2, betas=(0.5, 0.999), native=False)
    sched = torch.optim.lr_scheduler.StepLR(tr_ref.optimizer, step_size=1, gamma=0.5)
    for epoch in range(3):
        tr.step(x, y)
        tr_ref.step(x, y)
        sched.step()
        assert abs(tr.end_epoch()[0] - sched.get_last_lr()[0]) < 1e-12
    for (n, a), (_, b) in zip(net.state_dict().items(), ref.state_dict().items()):
        assert torch.allclose(a, b, rtol=2e-3, atol=2e-5), n


def test_checkpoint_moves_between_native_and_torch_adam(tmp_path):
    """optimizer_state_dict written by NativeAdam loads into torch.optim.Adam and back (utils.py:23-50)"""
    from nasa_niswan_b200 import ConvLSTM
    from nasa_niswan_b200.parallel import Trainer
    from nasa_niswan_b200.utils import load_checkpoint, save_checkpoint
    torch.manual_seed(11)
    x, y = torch.randn(2, 2, 5, 20, 24, device="cuda"), torch.randn(2, 20, 24, device="cuda")
    net = ConvLSTM(5, [16], [3], 1, precision="tf32").cuda()
    tr = Trainer(net, lr=1e-3, betas=(0.5, 0.999), native=True)
    tr.step(x, y)
    f = str(tmp_path / "generator.pth.tar")
    save_checkpoint(net, tr.optimizer, f, learning_rate=1e-3, epoch=1)
    net2 = ConvLSTM(5, [16], [3], 1, precision="tf32").cuda()
    opt2 = torch.optim.Adam(net2.parameters(), lr=1e-3, betas=(0.5, 0.999))
    load_checkpoint(f, net2, opt2)
    assert all(torch.equal(a, b) for a, b in zip(net.state_dict().values(), net2.state_dict().values()))
    s0 = opt2.state_dict()["state"][0]
    assert torch.allclose(s0["exp_avg"].cpu(), tr.optimizer.state_dict()["state"][0]["exp_avg"].cpu())
    tr2 = Trainer(net2, lr=1e-3, betas=(0.5, 0.999), native=True)
    load_checkpoint(f, net2, tr2.optimizer)
    assert tr2.optimizer.step_count == 1
    l1, l2 = float(tr.step(x, y)), float(tr2.step(x, y))
    assert l1 == pytest.approx(l2, rel=1e-5)


def test_cuda_graph_capture_of_the_forward():
    """SURVEY 8b: everything the op does is stream-ordered (kernels, memsets, TMA descriptors built on the host), so an
    inference rollout can be captured in a CUDA graph and replayed on new input"""
    from nasa_niswan_b200 import ConvLSTM
    torch.manual_seed(14)
    net = ConvLSTM(5, [32], [3], 1, precision="bf16").cuda().eval()
    x = torch.randn(2, 4, 5, 24, 32, device="cuda")
    with torch.no_grad():
        first = net(x).clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            net(x)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = net(x)
        x.copy_(torch.randn_like(x))
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, net(x))
        assert not torch.equal(out, first)


def _ddp_worker(rank, world, port, out):
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP
    from nasa_niswan_b200 import ConvLSTM
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)   # both ranks share cuda:0 here; gloo moves CUDA tensors
    torch.manual_seed(21)
    net = ConvLSTM(5, [16, 16], [3, 3], 2, precision="tf32").cuda()
    ddp = DDP(net)
    torch.manual_seed(22)
    X, Y = torch.randn(4, 3, 5, 12, 20), torch.randn(4, 12, 20)
    a, b = rank * 2, rank * 2 + 2
    pred = ddp(X[a:b].cuda())
    F.mse_loss(pred.squeeze(1), Y[a:b].cuda()).backward()
    if rank == 0:
        torch.save({k: p.grad.cpu() for k, p in net.named_parameters()}, out)
    dist.destroy_process_group()


def test_distributed_data_parallel_wrapper(tmp_path):
    """SURVEY 8b/8e: the dispatcher op is an ordinary autograd node, so torch's DistributedDataParallel (gradient
    hooks, bucketed all-reduce) works on the module unchanged: 2 ranks x 2 samples == the 4-sample gradient"""
    import socket
    import torch.multiprocessing as mp
    from nasa_niswan_b200 import ConvLSTM
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = str(tmp_path / "ddp.pt")
    mp.spawn(_ddp_worker, args=(2, port, out), nprocs=2, join=True)
    got = torch.load(out)
    torch.manual_seed(21)
    net = ConvLSTM(5, [16, 16], [3, 3], 2, precision="tf32").cuda()
    torch.manual_seed(22)
    X, Y = torch.randn(4, 3, 5, 12, 20), torch.randn(4, 12, 20)
    F.mse_loss(net(X.cuda()).squeeze(1), Y.cuda()).backward()
    for k, p in net.named_parameters():
        assert O.max_abs_normalised(got[k], p.grad.cpu()) < 1e-4, k
