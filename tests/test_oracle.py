"""CPU: pin the oracle (oracle/convlstm_oracle.py) against the reference-generated
golden vectors and the reference notebooks' printed known answers."""
import os

import numpy as np
import pytest
import torch

from oracle import convlstm_oracle as O
from oracle.golden import load_case

CASES = ["lstm_c21_h32_k3", "lstm_3layer_k533", "lstm_c8_h16_k5"]


def load(golden_dir, name):
    z = load_case(golden_dir, name)
    meta = z["meta"].tolist()
    B, T, cin, H, W, L = meta[:6]
    hidden, ks = meta[6:6 + L], meta[6 + L:6 + 2 * L]
    params = {k[6:]: torch.from_numpy(z[k]) for k in z if k.startswith("param/")}
    grads = {k[5:]: torch.from_numpy(z[k]) for k in z if k.startswith("grad/")}
    crop = z["crop"].tolist()
    crop = None if crop[0] < 0 else tuple(crop)
    return z, dict(B=B, T=T, cin=cin, H=H, W=W, L=L, hidden=hidden, ks=ks, crop=crop), params, grads


def test_golden_inputs_are_checked_against_the_reference_digest(golden_dir, tmp_path):
    # a case stores the reference's outputs and the seed of its inputs; inputs drawn from another seed are refused
    z = np.load(os.path.join(golden_dir, CASES[0] + ".npz"))
    np.savez(tmp_path / "case.npz", **{k: z[k] for k in z.files if k != "seed"}, seed=z["seed"] + 1)
    with pytest.raises(RuntimeError, match="draws other inputs"):
        load_case(str(tmp_path), "case")


def test_param_count_known_answer():
    # test.ipynb:4698-4699: ConvLSTM(5,[64,32,16],[5,3,3],3)
    shapes = O.param_shapes(5, [64, 32, 16], [5, 3, 3])
    counts = [int(np.prod(s)) for s in shapes.values()]
    assert counts == [441600, 256, 110592, 128, 27648, 64, 16, 1]
    assert sum(counts) == 580305
    assert list(shapes) == ["layers.0.conv.weight", "layers.0.conv.bias", "layers.1.conv.weight",
                            "layers.1.conv.bias", "layers.2.conv.weight", "layers.2.conv.bias",
                            "conv.weight", "conv.bias"]
    assert shapes["layers.0.conv.weight"] == (256, 69, 5, 5)
    assert shapes["layers.1.conv.weight"] == (128, 96, 3, 3)
    assert shapes["layers.2.conv.weight"] == (64, 48, 3, 3)


@pytest.mark.parametrize("name", CASES)
def test_forward_matches_reference(golden_dir, name):
    z, m, params, _ = load(golden_dir, name)
    assert {k: tuple(v.shape) for k, v in params.items()} == O.param_shapes(m["cin"], m["hidden"], m["ks"])
    pred = O.convlstm_forward(torch.from_numpy(z["x"]), params, m["L"])
    assert pred.shape == (m["B"], 1, m["H"], m["W"])          # model.py:291-292
    assert O.max_abs_normalised(pred, z["pred"]) < 2e-6
    loss = O.training_loss(pred, torch.from_numpy(z["y"]), m["crop"])
    assert abs(float(loss) - float(z["loss"])) < 1e-5


@pytest.mark.parametrize("name", CASES)
def test_cell_matches_reference(golden_dir, name):
    z, m, params, _ = load(golden_dir, name)
    h1, c1 = O.cell_forward(torch.from_numpy(z["cell/x"]), torch.from_numpy(z["cell/h0"]),
                            torch.from_numpy(z["cell/c0"]), params["layers.0.conv.weight"],
                            params["layers.0.conv.bias"])
    assert O.max_abs_normalised(h1, z["cell/h1"]) < 2e-6
    assert O.max_abs_normalised(c1, z["cell/c1"]) < 2e-6


@pytest.mark.parametrize("name", CASES)
def test_autograd_backward_matches_reference(golden_dir, name):
    z, m, params, grads = load(golden_dir, name)
    _, loss, g = O.forward_backward(torch.from_numpy(z["x"]), torch.from_numpy(z["y"]), params, m["L"], m["crop"])
    for k in grads:
        assert O.max_abs_normalised(g[k], grads[k]) < 2e-5, k


@pytest.mark.parametrize("name", CASES)
def test_manual_bptt_matches_reference(golden_dir, name):
    """The explicit BPTT formulas (what the CUDA kernels implement) reproduce the
    reference's autograd gradients."""
    z, m, params, grads = load(golden_dir, name)
    x, y = torch.from_numpy(z["x"]), torch.from_numpy(z["y"])
    pred = torch.from_numpy(z["pred"]).clone().requires_grad_(True)
    O.training_loss(pred, y, m["crop"]).backward()
    g = O.manual_backward(x, params, m["L"], pred.grad)
    for k in grads:
        assert O.max_abs_normalised(g[k], grads[k]) < 5e-5, k


def test_gate_order_and_zero_padding():
    # gate blocks i,f,g,o (model.py:221) and zero padding k//2 (model.py:204-211):
    # with W = 0 the gates are the bias -> closed form.
    hc, cin = 4, 3
    w = torch.zeros(4 * hc, cin + hc, 3, 3)
    b = torch.cat([torch.full((hc,), 1.0), torch.full((hc,), -2.0), torch.full((hc,), 0.5), torch.full((hc,), 3.0)])
    c0 = torch.full((1, hc, 5, 6), 0.7)
    h, c = O.cell_forward(torch.randn(1, cin, 5, 6), torch.randn(1, hc, 5, 6), c0, w, b)
    sig = lambda v: 1 / (1 + np.exp(-v))
    c_exp = 0.7 * sig(-2.0) + sig(1.0) * np.tanh(0.5)
    assert torch.allclose(c, torch.full_like(c, c_exp), atol=1e-6)
    assert torch.allclose(h, torch.full_like(h, sig(3.0) * np.tanh(c_exp)), atol=1e-6)
    # zero padding: an all-ones 3x3 filter on all-ones input counts valid taps
    w = torch.zeros(4 * hc, cin + hc, 3, 3)
    w[2 * hc:3 * hc, 0] = 1.0   # g gate sees channel 0 of x
    x = torch.ones(1, cin, 5, 6)
    _, c = O.cell_forward(x, torch.zeros(1, hc, 5, 6), torch.zeros(1, hc, 5, 6), w, torch.zeros(4 * hc))
    assert torch.allclose(c[0, 0, 0, 0], torch.tanh(torch.tensor(4.0)) * 0.5)   # corner: 4 taps
    assert torch.allclose(c[0, 0, 2, 2], torch.tanh(torch.tensor(9.0)) * 0.5)   # interior: 9 taps


def test_return_sequence_variant(golden_dir):
    z, m, params, _ = load(golden_dir, CASES[0])
    x = torch.from_numpy(z["x"])
    pred, seq = O.convlstm_forward(x, params, m["L"], return_sequence=True)
    assert seq.shape == (m["B"], m["T"], m["H"], m["W"])
    assert torch.equal(seq[:, -1:], pred)
    assert O.max_abs_normalised(O.convlstm_forward(x[:, :2], params, m["L"]), seq[:, 1:2]) < 1e-6


def test_padding_known_answer_from_notebook(golden_dir):
    z = np.load(os.path.join(golden_dir, "padding.npz"))
    printed = np.array([[21, 22, 23, 24, 20, 21, 22, 23, 24, 20, 21, 22, 23],
                        [16, 17, 18, 19, 15, 16, 17, 18, 19, 15, 16, 17, 18],
                        [11, 12, 13, 14, 10, 11, 12, 13, 14, 10, 11, 12, 13],
                        [6, 7, 8, 9, 5, 6, 7, 8, 9, 5, 6, 7, 8],
                        [1, 2, 3, 4, 0, 1, 2, 3, 4, 0, 1, 2, 3],
                        [6, 7, 8, 9, 5, 6, 7, 8, 9, 5, 6, 7, 8],
                        [11, 12, 13, 14, 10, 11, 12, 13, 14, 10, 11, 12, 13],
                        [16, 17, 18, 19, 15, 16, 17, 18, 19, 15, 16, 17, 18],
                        [21, 22, 23, 24, 20, 21, 22, 23, 24, 20, 21, 22, 23],
                        [16, 17, 18, 19, 15, 16, 17, 18, 19, 15, 16, 17, 18],
                        [11, 12, 13, 14, 10, 11, 12, 13, 14, 10, 11, 12, 13],
                        [6, 7, 8, 9, 5, 6, 7, 8, 9, 5, 6, 7, 8],
                        [1, 2, 3, 4, 0, 1, 2, 3, 4, 0, 1, 2, 3]])[None]   # dataset_config.ipynb:484-496
    assert np.array_equal(z["arange_out"], printed)
    assert np.array_equal(O.halo_pad(z["arange_in"], (13, 13), "reflect"), printed)


def test_padding_matches_reference(golden_dir):
    z = np.load(os.path.join(golden_dir, "padding.npz"))
    assert np.array_equal(O.halo_pad(z["pad3_in"], (22, 30), "reflect"), z["pad3_out"])
    assert np.array_equal(O.halo_pad(z["pad3_in"], (22, 30), "reflect"),
                          np.pad(np.concatenate([z["pad3_in"][..., -5:], z["pad3_in"], z["pad3_in"][..., :5]], -1),
                                 ((0, 0), (5, 5), (0, 0)), mode="reflect"))
    assert np.array_equal(O.halo_pad(z["pad4_in"], (22, 30), "reference_rnn"), z["pad4_out"])
    assert np.array_equal(O.halo_pad(z["pad4_full_in"], (100, 154), "reference_rnn"), z["pad4_full_out"])
    # the quirk is real: the true reflect differs from what the RNN dataset feeds the model
    assert not np.array_equal(O.halo_pad(z["pad4_in"], (22, 30), "reflect"), z["pad4_out"])
    with pytest.raises(AttributeError):
        O.cyclic_pad_lon(np.zeros((1, 1, 4, 4)), 20)


def test_fuse_inputs_shapes():
    rng = np.random.default_rng(1)
    lev = rng.standard_normal((3, 20, 9, 12)).astype(np.float32) * 4 + 2
    em = rng.standard_normal((3, 9, 12)).astype(np.float32)
    mean, std = rng.standard_normal(21), rng.random(21) + 0.5
    X = O.fuse_inputs(lev, em, mean, std, (19, 22), "reference_rnn")
    assert X.shape == (3, 21, 19, 22) and X.dtype == np.float32
    core = X[:, :, 5:14, 5:17]
    assert np.allclose(core[:, 20], (em - mean[20]) / std[20], atol=1e-5)
    assert np.allclose(core[:, 3], (lev[:, 3] - mean[3]) / std[3], atol=1e-5)
