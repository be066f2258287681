"""CPU: input gradients through the frame bank and the preprocessing, without a GPU -- the torch restatement of the
fusion against the numpy oracle, the ordered adjoint reference against autograd, the (t, b) window scatter on a lattice
case, the C ABI's new entry points and the new ops' schemas."""
import inspect

import numpy as np
import pytest
import torch

from nasa_niswan_b200 import _lib
from oracle import convlstm_oracle as O
from oracle import lattice as Lt
from oracle.adjoint_oracle import fuse_adjoint_reference, fuse_inputs_torch, scatter_windows

# (N, L, S, H, W, Hp, Wp): no halo; even halos; odd halos (top != bottom, left != right); a halo as wide as the grid
# (the 5 -> 13 known answer of the dataset notebook); statics; no level (emission only)
SHAPES = [(3, 2, 0, 7, 9, 7, 9), (2, 1, 0, 8, 10, 12, 16), (3, 2, 2, 9, 11, 12, 14), (2, 1, 1, 5, 5, 13, 13),
          (2, 0, 3, 6, 8, 9, 11)]
MODES = ["reflect", "reference_rnn"]


def fields(N, L, S, H, W, seed=0):
    rng = np.random.default_rng(seed)
    lev = (rng.standard_normal((N, L, H, W)) * 3 + 1).astype(np.float32)
    emis = np.abs(rng.standard_normal((N, H, W))).astype(np.float32)
    mean = rng.standard_normal(L + 1).astype(np.float32)
    std = (rng.random(L + 1) + 0.3).astype(np.float32)
    stat = rng.standard_normal((S, H, W)).astype(np.float32) if S else None
    return lev, emis, mean, std, stat


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_torch_restatement_equals_the_numpy_oracle(shape, mode):
    N, L, S, H, W, Hp, Wp = shape
    lev, emis, mean, std, stat = fields(N, L, S, H, W)
    ref = O.fuse_inputs(lev, emis, mean, std, (Hp, Wp), mode, stat)
    t = lambda a: None if a is None else torch.from_numpy(a)
    got = fuse_inputs_torch(t(lev), t(emis), t(mean), t(std), (Hp, Wp), mode, t(stat))
    assert torch.equal(got, torch.from_numpy(ref))


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_ordered_adjoint_reference_agrees_with_autograd(shape, mode):
    N, L, S, H, W, Hp, Wp = shape
    lev, emis, mean, std, stat = fields(N, L, S, H, W)
    lev_t, emis_t = torch.from_numpy(lev).requires_grad_(), torch.from_numpy(emis).requires_grad_()
    stat_t = torch.from_numpy(stat).requires_grad_() if S else None
    out = fuse_inputs_torch(lev_t, emis_t, torch.from_numpy(mean), torch.from_numpy(std), (Hp, Wp), mode, stat_t)
    g = torch.randn(out.shape, generator=torch.Generator().manual_seed(1))
    out.backward(g)
    ref = fuse_adjoint_reference(g, torch.from_numpy(std), L, S, H, W, mode)
    pairs = [(ref["levels3d"], lev_t.grad), (ref["emis2d"], emis_t.grad)] + ([(ref["statics"], stat_t.grad)] if S else [])
    for a, b in pairs:
        if b.numel():
            assert float((a - b).abs().max()) <= 1e-6 * float(b.abs().max())
    if not S:
        assert ref["statics"] is None


def test_halo_as_wide_as_the_grid_sums_every_copy():
    """5 x 5 -> 13 x 13: an interior element has up to three row and three column copies; a gradient of ones counts them"""
    ref = fuse_adjoint_reference(torch.ones(1, 2, 13, 13), torch.ones(2), 1, 0, 5, 5, "reflect")
    counts = ref["emis2d"][0]
    assert float(counts.sum()) == 13 * 13 and float(counts.max()) == 9.0


def test_scatter_of_a_frame_bank_lattice_case_stays_exact():
    """the bank's gradient on the lattice case with overlapping windows: the (t, b) scatter of the reference dx is exact
    in fp32 (every partial sum within the 2^20 grid steps of the exactness headroom), so the GPU must equal it bit for bit"""
    for prec in ("tf32", "bf16"):
        case = Lt.c_case("h64_k3_33x9_T4", prec)
        ref = Lt.reference(case)
        starts = case["starts"].tolist()
        n = case["frames"].shape[0]
        assert len(set(s + t for s in starts for t in range(case["T"]))) < len(starts) * case["T"]   # frames are shared
        dx = ref["dx"]
        s64 = scatter_windows(dx, starts, n)
        assert torch.equal(scatter_windows(dx.float(), starts, n).double(), s64)
        grid = min(Lt.grid(dx), Lt.grid(s64))
        assert float(scatter_windows(dx.abs(), starts, n).max()) / grid <= 2.0 ** 20


def test_abi_exports_the_bank_gradient_entry_points():
    lib = _lib.load()
    for name in ("nint_backward_input_bank", "nint_fuse_inputs_adjoint"):
        assert hasattr(lib, name) and name in _lib.EXPORTS


def test_ops_are_registered_with_fakes():
    import nasa_niswan_b200.preprocess  # noqa: F401  (registers nint::fuse_inputs)
    from torch._library.simple_registry import singleton
    assert str(torch.ops.nint.convlstm_forward_bank_dx.default._schema) == \
        ("nint::convlstm_forward_bank_dx(Tensor frames, Tensor win_start, Tensor[] params, Tensor[] h0, Tensor[] c0, "
         "Tensor anchor, Tensor dframes, SymInt plan_id) -> (Tensor, Tensor, Tensor[], Tensor[])")
    assert str(torch.ops.nint.bank_input_grad_.default._schema) == \
        "nint::bank_input_grad_(Tensor(a0!) dframes, SymInt plan_id, SymInt generation) -> ()"
    assert str(torch.ops.nint.fuse_inputs.default._schema) == \
        ("nint::fuse_inputs(Tensor levels3d, Tensor emis2d, Tensor mean, Tensor std, Tensor? statics, "
         "SymInt padded_height, SymInt padded_width, SymInt mode) -> Tensor")
    for name in ("nint::convlstm_forward_bank_dx", "nint::bank_input_grad_", "nint::fuse_inputs"):
        assert singleton.find(name).fake_impl.kernel is not None, name
    # the existing bank ops keep their schemas
    assert str(torch.ops.nint.convlstm_forward_bank.default._schema) == \
        "nint::convlstm_forward_bank(Tensor frames, Tensor win_start, Tensor[] params, SymInt plan_id) -> (Tensor, Tensor)"


def test_from_fields_records_what_field_grads_needs():
    from nasa_niswan_b200 import preprocess as P
    rec = P._adjoint_record(torch.ones(3), 2, 1, 9, 11, "reference_rnn")
    params = set(inspect.signature(P.fuse_inputs_adjoint).parameters) - {"dframes", "want"}
    assert set(rec) == params
    assert rec["levels"] == 2 and rec["n_static"] == 1 and (rec["height"], rec["width"]) == (9, 11)
    assert rec["mode"] == "reference_rnn" and torch.equal(rec["std"], torch.ones(3))
    src = inspect.getsource(P.FrameBank.from_fields)
    assert "_adjoint_record(std, L, S, H, W, mode)" in src
