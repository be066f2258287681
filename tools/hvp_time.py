"""Cost of the second-order adjoint (ConvLSTM.hvp / Plan.backward_second_order), bf16, at BASELINE cfg 2 (B=32, T=12,
21 channels, 90x144, 21 -> 64, 3x3) and the shipped model (B=8, T=48, 5 channels, 100x154, [64, 32, 16], [5, 3, 3]).

  1. ms per forward, per tangent pass and per second-order pass on one training plan made with second_order=True
     (CUDA events around --steps calls after --warmup; the tangent and second-order passes only read the forward, so
     each is repeated on the same forward), alternated --rounds times in the same process.
  2. device time per launch of soa_cell_kernel and of the pass's dgrad (conv) launches, from torch.profiler over one
     second-order pass in a run of its own; achieved bytes/s of soa_cell_kernel on its algorithmic bytes against the
     device-to-device copy bandwidth measured in the same run.
Prints one JSON line with the card name and power limit; --out also writes it to a file.

    python tools/hvp_time.py --steps 10 --rounds 3 --out hvp_time.json
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402
from nasa_niswan_b200 import ConvLSTM  # noqa: E402
from tangent_time import copy_bandwidth, kernel_us, power_limit, time_ms  # noqa: E402

# name: (B, T, C, H, W, hidden, ks)
GEOMS = {"cfg2": (32, 12, 21, 90, 144, [64], [3]),
         "shipped": (8, 48, 5, 100, 154, [64, 32, 16], [5, 3, 3])}


def soa_cell_bytes(B, T, H, W, hidden, esize):
    """algorithmic bytes of all soa_cell_kernel launches of one pass: gates (E) and the tangent dump (fp32) read, c and
    dc at t-1 and t read, kappa and its tangent read and written, eta and its tangent read (not at the top layer's
    last step), dgates and their tangents written (E); the per-pixel head seeds are left out"""
    tot = 0
    for l, hc in enumerate(hidden):
        per = B * H * W * hc * (4 * esize + 16 + 8 + 8 + 16 + 8 * esize)
        tot += T * per + (T - (1 if l == len(hidden) - 1 else 0)) * B * H * W * hc * 8
    return tot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--geoms", default="cfg2,shipped")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: these are GPU times")
    res = {"device": torch.cuda.get_device_name(0), "power_limit": power_limit()}
    bw = copy_bandwidth()
    res["copy_bandwidth_TBps"] = round(bw / 1e12, 3)
    for name in a.geoms.split(","):
        B, T, C, H, W, hidden, ks = GEOMS[name]
        torch.manual_seed(0)
        net = ConvLSTM(C, hidden, ks, len(hidden), precision="bf16").cuda()
        g = torch.Generator(device="cuda").manual_seed(0)
        x = torch.randn(B, T, C, H, W, device="cuda", generator=g)
        dx = torch.randn(B, T, C, H, W, device="cuda", generator=g)
        u = torch.randn(B, 1, H, W, device="cuda", generator=g)
        du = torch.randn(B, 1, H, W, device="cuda", generator=g)
        plan = net.plan_for(x, True, second_order=True)
        plan.forward(x)
        passes = {"forward": lambda: plan.forward(x), "tangent": lambda: plan.forward_tangent(dx),
                  "second_order": lambda: plan.backward_second_order(u, du)}
        times = {k: [] for k in passes}
        for r in range(a.rounds):
            for k, fn in passes.items():
                if r == 0:
                    for _ in range(a.warmup):
                        fn()
                times[k].append(time_ms(fn, a.steps))
        ks_ = kernel_us(passes["second_order"], ["soa_cell_kernel", "conv_halo_kernel"])
        cb = soa_cell_bytes(B, T, H, W, hidden, 2)
        n_cell = ks_["soa_cell_kernel"][1]
        cell_s = ks_["soa_cell_kernel"][0] * n_cell * 1e-6
        res[name] = {
            "workspace_GB": round(plan.workspace_bytes / 1e9, 2),
            **{f"{k}_ms": [round(v, 3) for v in t] for k, t in times.items()},
            "soa_cell_us_per_launch": round(ks_["soa_cell_kernel"][0], 2), "soa_cell_launches": n_cell,
            "soa_cell_MB_per_launch": round(cb / max(n_cell, 1) / 1e6, 1),
            "soa_cell_TBps": round(cb / cell_s / 1e12, 3),
            "soa_cell_fraction_of_copy_bw": round(cb / cell_s / bw, 3),
            "dgrad_us_per_launch": round(ks_["conv_halo_kernel"][0], 2), "dgrad_launches": ks_["conv_halo_kernel"][1],
        }
        del net, plan
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
