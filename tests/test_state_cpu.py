"""CPU: the stateful ConvLSTM surface without a GPU -- the oracle's stateful loop against the stateless one, chaining
it over a split window, the C ABI's new flag and entry points, and the schemas of the stateful ops."""
import ctypes

import torch

from nasa_niswan_b200 import _lib
from oracle import convlstm_oracle as O
from oracle.state_oracle import convlstm_forward_state


def _setup(L=2, seed=0, B=2, T=5, C=3, H=9, W=11):
    hidden, ks = [8, 4][:L], [3, 5][:L]
    params = O.init_params(C, hidden, ks, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(B, T, C, H, W, generator=g)
    return x, params, hidden


def test_oracle_zero_state_equals_stateless_forward():
    x, params, _ = _setup()
    for seq in (False, True):
        ref = O.convlstm_forward(x, params, 2, return_sequence=seq)
        for state in (None, [(None, None), (None, None)]):
            out, final = convlstm_forward_state(x, params, 2, state, return_sequence=seq)
            for a, b in zip(ref if seq else (ref,), out if seq else (out,)):
                assert torch.equal(a, b)
            assert len(final) == 2 and all(h.shape == c.shape for h, c in final)


def test_oracle_chained_windows_equal_the_whole_window():
    x, params, hidden = _setup()
    g = torch.Generator().manual_seed(7)
    state = [(torch.randn(2, hc, 9, 11, generator=g), torch.randn(2, hc, 9, 11, generator=g)) for hc in hidden]
    (pred, seq), final = convlstm_forward_state(x, params, 2, state, return_sequence=True)
    (_, seq1), mid = convlstm_forward_state(x[:, :2], params, 2, state, return_sequence=True)
    (pred2, seq2), final2 = convlstm_forward_state(x[:, 2:], params, 2, mid, return_sequence=True)
    assert torch.equal(pred, pred2) and torch.equal(seq, torch.cat([seq1, seq2], 1))
    for (h, c), (h2, c2) in zip(final, final2):
        assert torch.equal(h, h2) and torch.equal(c, c2)
    # gradients flow through the carried state: the chain differentiates like the whole window
    h0 = state[0][0].clone().requires_grad_(True)
    whole = convlstm_forward_state(x, params, 2, [(h0, state[0][1])] + state[1:])[0]
    gw, = torch.autograd.grad(whole.sum(), h0)
    mid = convlstm_forward_state(x[:, :2], params, 2, [(h0, state[0][1])] + state[1:])[1]
    gc, = torch.autograd.grad(convlstm_forward_state(x[:, 2:], params, 2, mid)[0].sum(), h0)
    assert torch.allclose(gw, gc, rtol=1e-5, atol=1e-7)


def test_abi_exports_the_state_entry_points_and_reserves_the_state_buffers():
    lib = _lib.load()
    for name in ("nint_backward_bptt_state", "nint_backward_initial_state"):
        assert hasattr(lib, name) and name in _lib.EXPORTS
    assert _lib.FLAG_STATE_GRAD == 4

    def ws(flags, hidden=(64, 20)):
        cfg = _lib.NintConfig()
        cfg.batch, cfg.seq_len, cfg.height, cfg.width, cfg.in_channels = 4, 5, 90, 144, 21
        cfg.num_layers = len(hidden)
        for i, hc in enumerate(hidden):
            cfg.hidden[i], cfg.ksize[i] = hc, 3
        cfg.dtype, cfg.training, cfg.flags = 0, 1, flags
        h = ctypes.c_void_p()
        assert lib.nint_plan_create(ctypes.byref(cfg), ctypes.byref(h)) == 0, lib.nint_last_error()
        n = lib.nint_plan_workspace_bytes(h)
        lib.nint_plan_destroy(h)
        return n
    npix = 4 * 90 * 144
    # per layer a dL/dh_T buffer (hidden 20 runs padded to 32), plus the dgrad dump of dh0 (widest padded layer: 64)
    assert ws(_lib.FLAG_STATE_GRAD) - ws(0) >= npix * (64 + 32 + 64) * 4
    # with the input gradient the dump is shared
    both = ws(_lib.FLAG_STATE_GRAD | _lib.FLAG_INPUT_GRAD) - ws(_lib.FLAG_INPUT_GRAD)
    assert npix * (64 + 32) * 4 <= both < npix * (64 + 32 + 64) * 4


def test_stateful_ops_are_registered_next_to_the_stateless_ones():
    import nasa_niswan_b200  # noqa: F401  (registers the ops)
    assert str(torch.ops.nint.convlstm_forward_state.default._schema) == \
        ("nint::convlstm_forward_state(Tensor x, Tensor[] params, Tensor[] h0, Tensor[] c0, SymInt plan_id) -> "
         "(Tensor, Tensor, Tensor[], Tensor[])")
    assert str(torch.ops.nint.convlstm_forward_bank_state.default._schema) == \
        ("nint::convlstm_forward_bank_state(Tensor frames, Tensor win_start, Tensor[] params, Tensor[] h0, "
         "Tensor[] c0, SymInt plan_id) -> (Tensor, Tensor, Tensor[], Tensor[])")
    assert "nint::convlstm_backward_state" in str(torch.ops.nint.convlstm_backward_state.default._schema)
