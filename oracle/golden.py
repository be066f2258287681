"""The reference ConvLSTM's golden vectors (tests/golden/lstm_*.npz): what the reference computed, stored; the inputs
it computed them from, drawn again.

A case file holds the reference's outputs (prediction, loss, every parameter gradient, one cell step's h1 and c1), the
case geometry (`meta`, `crop`), the seed of the inputs and a SHA-256 of the reference's own inputs.  The inputs -- x, y,
the default-initialised parameters of the reference constructor (model.py:235-251: one nn.Conv2d per layer, then the
1x1 head), the cell step's x, h0 and c0 -- are drawn again from that seed with plain torch in the order the reference
drew them, and must hash to the stored digest.  The files stay small, and a torch whose generator draws other numbers
fails loudly instead of comparing against other inputs."""
import hashlib
import os

import numpy as np
import torch


def convlstm_inputs(meta, crop, seed):
    """The inputs of a case, in the order oracle/make_golden.py stores them: x, y, param/<state_dict name>..., cell/x,
    cell/h0, cell/c0."""
    meta = [int(v) for v in meta]
    B, T, cin, H, W, L = meta[:6]
    hidden, ks = meta[6:6 + L], meta[6 + L:6 + 2 * L]
    crop = [int(v) for v in crop]
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(seed)
        params, c = {}, cin
        for l, (hc, k) in enumerate(zip(hidden, ks)):
            conv = torch.nn.Conv2d(c + hc, 4 * hc, k, padding=k // 2)
            params[f"param/layers.{l}.conv.weight"], params[f"param/layers.{l}.conv.bias"] = conv.weight, conv.bias
            c = hc
        head = torch.nn.Conv2d(hidden[-1], 1, 1)
        params["param/conv.weight"], params["param/conv.bias"] = head.weight, head.bias
        x = torch.randn(B, T, cin, H, W)
        y = torch.randn(B, H, W) if crop[0] < 0 else torch.randn(B, crop[1] - crop[0], crop[3] - crop[2])
        torch.manual_seed(seed + 1)
        cell_x = torch.randn(B, cin, H, W)
        h0 = torch.randn(B, hidden[0], H, W) * 0.5
        c0 = torch.randn(B, hidden[0], H, W)
    out = {"x": x, "y": y, **params, "cell/x": cell_x, "cell/h0": h0, "cell/c0": c0}
    return {k: v.detach().numpy() for k, v in out.items()}


def input_digest(arrays) -> str:
    """SHA-256 over names, dtypes, shapes and bytes, in the given order"""
    h = hashlib.sha256()
    for k, v in arrays.items():
        a = np.ascontiguousarray(v)
        h.update(f"{k}|{a.dtype.str}|{a.shape}|".encode())
        h.update(a.tobytes())
    return h.hexdigest()


def save_case(path, arrays, seed):
    """Writes a case from every array of the reference run; refuses when plain torch does not draw the reference's
    inputs from `seed`."""
    drawn = convlstm_inputs(arrays["meta"], arrays["crop"], seed)
    ref_inputs = {k: arrays[k] for k in arrays if k in drawn}
    if input_digest(ref_inputs) != input_digest(drawn):
        raise ValueError(f"{path}: the inputs drawn from seed {seed} are not the reference's")
    kept = {k: v for k, v in arrays.items() if k not in drawn}
    np.savez(path, **kept, seed=np.int64(seed), input_sha256=np.array(input_digest(ref_inputs)))


def load_case(golden_dir, name):
    """{array name: array} of a case: the stored outputs and the inputs drawn again"""
    z = np.load(os.path.join(golden_dir, name + ".npz"))
    out = {k: z[k] for k in z.files}
    seed, digest = int(out.pop("seed")), str(out.pop("input_sha256"))
    drawn = convlstm_inputs(out["meta"], out["crop"], seed)
    if input_digest(drawn) != digest:
        raise RuntimeError(f"{name}: torch {torch.__version__} draws other inputs from seed {seed} than the reference "
                           "run did; regenerate tests/golden with oracle/make_golden.py")
    return {**drawn, **out}
