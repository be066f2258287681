"""CPU: the tangent-linear surface without a GPU -- the oracle's forward-mode derivative (the reference the GPU tests
compare against) checked by central differences and by the dot-product identity with its adjoint, the C ABI's new flag
and entry points, and the workspace: plans without the flag keep their sizes, plans with it reserve the tangent
buffers."""
import ctypes

import pytest
import torch

from nasa_niswan_b200 import _lib
from oracle import convlstm_oracle as O
from oracle.state_oracle import convlstm_forward_state


def _oracle_fn(params, L):
    """(x, h0s, c0s) -> (pred, seq, h_Ts, c_Ts) of the reference loop, a function torch.func can differentiate"""
    def f(x, hs, cs):
        (pred, seq), final = convlstm_forward_state(x, params, L, list(zip(hs, cs)), return_sequence=True)
        return pred, seq, tuple(h for h, _ in final), tuple(c for _, c in final)
    return f


def _setup(seed=0, B=2, T=4, C=3, H=9, W=11, hidden=(8, 4), ks=(3, 5)):
    params = {k: v.double() for k, v in O.init_params(C, list(hidden), list(ks), seed=seed).items()}
    g = torch.Generator().manual_seed(seed + 1)
    r = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    x = r(B, T, C, H, W)
    state = (tuple(r(B, hc, H, W) * 0.5 for hc in hidden), tuple(r(B, hc, H, W) * 0.5 for hc in hidden))
    v = (r(B, T, C, H, W), tuple(r(B, hc, H, W) for hc in hidden), tuple(r(B, hc, H, W) for hc in hidden))
    return params, len(hidden), (x,) + state, v


def test_oracle_jvp_matches_central_differences():
    params, L, primals, v = _setup()
    f = _oracle_fn(params, L)
    _, jv = torch.func.jvp(f, primals, v)
    eps = 1e-5
    shift = lambda s: (primals[0] + s * v[0], tuple(a + s * b for a, b in zip(primals[1], v[1])),
                       tuple(a + s * b for a, b in zip(primals[2], v[2])))
    plus, minus = f(*shift(eps)), f(*shift(-eps))
    flat = lambda o: [o[0], o[1], *o[2], *o[3]]
    for j, p, m in zip(flat(jv), flat(plus), flat(minus)):
        fd = (p - m) / (2 * eps)
        assert O.max_abs_normalised(j, fd) < 1e-8


def test_oracle_jvp_and_vjp_satisfy_the_dot_product_identity():
    params, L, primals, v = _setup(seed=3)
    f = _oracle_fn(params, L)
    out, jv = torch.func.jvp(f, primals, v)
    g = torch.Generator().manual_seed(9)
    u = (torch.randn(out[0].shape, generator=g, dtype=torch.float64), torch.randn(out[1].shape, generator=g, dtype=torch.float64),
         tuple(torch.randn(t.shape, generator=g, dtype=torch.float64) for t in out[2]),
         tuple(torch.randn(t.shape, generator=g, dtype=torch.float64) for t in out[3]))
    _, vjp = torch.func.vjp(f, *primals)
    ju = vjp(u)
    dot = lambda a, b: sum(float((p * q).sum()) for p, q in zip(torch.utils._pytree.tree_leaves(a),
                                                               torch.utils._pytree.tree_leaves(b)))
    lhs, rhs = dot(u, jv), dot(ju, v)
    assert abs(lhs - rhs) <= 1e-12 * max(abs(lhs), abs(rhs))


def test_abi_exports_the_tangent_entry_points():
    lib = _lib.load()
    for name in ("nint_forward_tangent", "nint_forward_tangent_bank"):
        assert hasattr(lib, name) and name in _lib.EXPORTS
    assert _lib.FLAG_TANGENT == 8


def _ws(B, T, H, W, C, hidden, ks, dtype, training, return_sequence, flags):
    lib = _lib.load()
    cfg = _lib.NintConfig()
    cfg.batch, cfg.seq_len, cfg.height, cfg.width, cfg.in_channels = B, T, H, W, C
    cfg.num_layers = len(hidden)
    for i, (hc, k) in enumerate(zip(hidden, ks)):
        cfg.hidden[i], cfg.ksize[i] = hc, k
    cfg.dtype, cfg.training, cfg.return_sequence, cfg.flags = dtype, training, return_sequence, flags
    h = ctypes.c_void_p()
    assert lib.nint_plan_create(ctypes.byref(cfg), ctypes.byref(h)) == 0, lib.nint_last_error()
    n = lib.nint_plan_workspace_bytes(h)
    lib.nint_plan_destroy(h)
    return n


# workspace bytes of plans without the tangent flag, as the library computed them before the flag existed
PINNED = [
    ((32, 12, 90, 144, 21, [64], [3], 0, 1, 0, 0), 5044623360),               # BASELINE cfg 2, bf16 training
    ((32, 12, 90, 144, 21, [64], [3], 0, 1, 0, 6), 5363275776),               # + input and state gradients
    ((2, 6, 100, 154, 5, [64, 32, 16], [5, 3, 3], 1, 1, 1, 7), 778169344),    # shipped model, tf32, every flag
    ((2, 4, 20, 24, 5, [20, 48, 64], [5, 3, 3], 0, 1, 1, 0), 14523392),       # padded hidden sizes, return_sequence
    ((4, 5, 90, 144, 21, [64], [3], 1, 0, 0, 0), 73879552),                   # tf32 inference
]


@pytest.mark.parametrize("cfg,nbytes", PINNED)
def test_flagless_workspace_sizes_are_unchanged(cfg, nbytes):
    assert _ws(*cfg) == nbytes


def test_the_flag_reserves_the_tangent_buffers():
    B, T, H, W, C, hidden = 4, 5, 90, 144, 21, [64, 20]
    npix = B * H * W
    for dtype, esize in ((0, 2), (1, 4)):
        base = _ws(B, T, H, W, C, hidden, [3, 3], dtype, 1, 0, 0)
        extra = _ws(B, T, H, W, C, hidden, [3, 3], dtype, 1, 0, _lib.FLAG_TANGENT) - base
        # input tangent (21 channels padded to 32), per layer a 2-slot dh ring (hidden 20 runs padded to 32 lanes) and a
        # dc buffer (hidden 20 runs as 32 channels), one fp32 dump of the widest layer's 4 * 64 gate columns
        need = T * npix * 32 * esize + 2 * npix * (64 + 32) * esize + npix * (64 + 32) * 4 + npix * 4 * 64 * 4
        assert need <= extra < need + 64 * 1024
        # inference plans keep no saved gates: the flag reserves nothing there
        assert _ws(B, T, H, W, C, hidden, [3, 3], dtype, 0, 0, _lib.FLAG_TANGENT) == \
            _ws(B, T, H, W, C, hidden, [3, 3], dtype, 0, 0, 0)
