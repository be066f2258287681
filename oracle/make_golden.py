"""Generate tests/golden/*.npz by running the UNMODIFIED reference.

Needs a checkout of the upstream repository (smhassanerfani/nasa-niswan):

    PYTHONDONTWRITEBYTECODE=1 python oracle/make_golden.py <path of the upstream checkout>

* ConvLSTM vectors: imports the upstream ``model.py`` as-is, seeds torch,
  runs forward + ``MSELoss+L1Loss`` + backward (train.py:96-109) on CPU fp32
  and stores prediction, loss and every parameter gradient; the inputs
  (x, y, state_dict, cell-step inputs) are stored as their seed and digest
  (oracle/golden.py).
* Padding vectors: ``dataset.py`` cannot be imported here (xarray missing), so
  the two padding classes (dataset.py:13-98) are pulled out of the source with
  ``ast`` and executed against numpy only, exactly as written upstream.
The files are small and committed; the tests never read the upstream checkout.
"""
import ast
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from oracle import golden  # noqa: E402

REF = None                # the upstream checkout, from the command line
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")


def _ref_model():
    sys.dont_write_bytecode = True
    sys.path.insert(0, REF)
    import model as ref_model  # noqa: E402  (the reference's model.py)
    sys.path.pop(0)
    return ref_model


def _ref_padding_classes():
    src = open(os.path.join(REF, "dataset.py")).read()
    tree = ast.parse(src)
    keep = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name in ("E33OMAPAD", "E33OMAPADRNN")]
    # drop add_static_attributes (needs xarray + a file that is not in the repo)
    for cls in keep:
        cls.body = [b for b in cls.body if not (isinstance(b, ast.FunctionDef) and b.name == "add_static_attributes")]
    mod = ast.Module(body=keep, type_ignores=[])
    ns = {"np": np, "Dataset": object}
    exec(compile(mod, "dataset.py[padding classes]", "exec"), ns)
    return ns["E33OMAPAD"], ns["E33OMAPADRNN"]


def convlstm_case(name, B, T, cin, hidden, ks, H, W, seed, crop=None, with_sequence=False):
    ref = _ref_model()
    torch.manual_seed(seed)
    net = ref.ConvLSTM(cin, hidden, ks, len(hidden))
    x = torch.randn(B, T, cin, H, W)
    if crop is None:
        y = torch.randn(B, H, W)
    else:
        y = torch.randn(B, crop[1] - crop[0], crop[3] - crop[2])
    pred = net(x)
    p = pred if crop is None else pred[:, :, crop[0]:crop[1], crop[2]:crop[3]]
    p = p.squeeze(1)
    loss = torch.nn.MSELoss()(y, p) + torch.nn.L1Loss()(y, p)      # train.py:74-75,105
    loss.backward()
    out = {"x": x.numpy(), "y": y.numpy(), "pred": pred.detach().numpy(),
           "loss": np.float32(loss.item()),
           "meta": np.array([B, T, cin, H, W, len(hidden)] + list(hidden) + list(ks), dtype=np.int64),
           "crop": np.array(crop if crop is not None else [-1, -1, -1, -1], dtype=np.int64)}
    for k, v in net.state_dict().items():
        out["param/" + k] = v.detach().numpy()
    for k, v in net.named_parameters():
        out["grad/" + k] = v.grad.detach().numpy()
    # single-cell step with non-zero state (model.py:216-231)
    cell = net.layers[0]
    torch.manual_seed(seed + 1)
    xs = torch.randn(B, cin, H, W)
    h0 = torch.randn(B, hidden[0], H, W) * 0.5
    c0 = torch.randn(B, hidden[0], H, W)
    with torch.no_grad():
        h1, c1 = cell(xs, (h0, c0))
    out.update({"cell/x": xs.numpy(), "cell/h0": h0.numpy(), "cell/c0": c0.numpy(),
                "cell/h1": h1.numpy(), "cell/c1": c1.numpy()})
    golden.save_case(os.path.join(OUT, name + ".npz"), out, seed)
    print(name, "loss", float(loss), "pred", tuple(pred.shape))


def padding_case():
    PAD3, PAD4 = _ref_padding_classes()
    rng = np.random.default_rng(0)
    out = {}
    # the notebook's printed known answer (dataset_config.ipynb:511-515 -> 484-496)
    p3 = PAD3("train", "bc", (13, 13))
    out["arange_in"] = np.arange(25).reshape(1, 5, 5)
    out["arange_out"] = p3._padding_data(out["arange_in"])
    # 3-D variant on a (C,H,W) field, production padding 90x144 -> 100x154 scaled down
    p3 = PAD3("train", "bc", (22, 30))
    a = rng.standard_normal((3, 12, 20)).astype(np.float32)
    out["pad3_in"], out["pad3_out"] = a, p3._padding_data(a)
    # 4-D RNN variant (T,C,H,W) incl. the fliplr-on-channels quirk (dataset.py:96)
    p4 = PAD4("train", "bc", (22, 30), sequence_length=4)
    b = rng.standard_normal((4, 5, 12, 20)).astype(np.float32)
    out["pad4_in"], out["pad4_out"] = b, p4._padding_data(b)
    # the real geometry, one frame only to stay small
    p4 = PAD4("train", "bc", (100, 154), sequence_length=1)
    c = rng.standard_normal((1, 2, 90, 144)).astype(np.float32)
    out["pad4_full_in"], out["pad4_full_out"] = c, p4._padding_data(c)
    np.savez(os.path.join(OUT, "padding.npz"), **out)
    print("padding", out["arange_out"].shape, out["pad4_out"].shape, out["pad4_full_out"].shape)


def main():
    global REF
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    REF = os.path.abspath(sys.argv[1])
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(1)  # bit-reproducible reductions
    # single layer, BASELINE channel geometry (20 levels + emission), small grid; GPU-tile friendly
    convlstm_case("lstm_c21_h32_k3", B=2, T=3, cin=21, hidden=[32], ks=[3], H=20, W=24, seed=0)
    # scaled-down version of the shipped 3-layer recipe (launcher.sh:17-25): k 5/3/3, halo crop
    convlstm_case("lstm_3layer_k533", B=1, T=3, cin=5, hidden=[32, 16, 16], ks=[5, 3, 3], H=18, W=22, seed=1,
                  crop=(5, 13, 5, 17))
    # 5x5, ragged grid (not a multiple of any tile), batch 3
    convlstm_case("lstm_c8_h16_k5", B=3, T=2, cin=8, hidden=[16], ks=[5], H=11, W=13, seed=2)
    padding_case()


if __name__ == "__main__":
    main()
