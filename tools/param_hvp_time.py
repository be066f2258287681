"""Cost of parameter-space directions, bf16, at BASELINE cfg 2 (B=32, T=12, 21 channels, 90x144, 21 -> 64, 3x3) and
the shipped model (B=8, T=48, 5 channels, 100x154, [64, 32, 16], [5, 3, 3]), on one training plan made with
second_order=True and param_tangent=True:

ms per forward; per tangent pass without and with a parameter direction (every layer and the head); per second-order
pass after each; per params call (Plan.backward_second_order_params) with and without its gradient part.  CUDA events
around --steps calls after --warmup (the passes only read the forward, so each repeats on the same forward),
alternated --rounds times in one process.  Prints one JSON line with the card name and power limit; --out also writes it.

    python tools/param_hvp_time.py --steps 10 --rounds 3 --out param_hvp_time.json
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
from tangent_time import power_limit, time_ms  # noqa: E402

# name: (B, T, C, H, W, hidden, ks)
GEOMS = {"cfg2": (32, 12, 21, 90, 144, [64], [3]),
         "shipped": (8, 48, 5, 100, 154, [64, 32, 16], [5, 3, 3])}


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
    for name in a.geoms.split(","):
        B, T, C, H, W, hidden, ks = GEOMS[name]
        torch.manual_seed(0)
        net = ConvLSTM(C, hidden, ks, len(hidden), precision="bf16").cuda()
        g = torch.Generator(device="cuda").manual_seed(0)
        x = torch.randn(B, T, C, H, W, device="cuda", generator=g)
        dx = torch.randn(B, T, C, H, W, device="cuda", generator=g)
        direction = net.param_direction({n: torch.randn(p.shape, device="cuda", generator=g) * 0.01
                                         for n, p in net.named_parameters()})
        u = torch.randn(B, 1, H, W, device="cuda", generator=g)
        du = torch.randn(B, 1, H, W, device="cuda", generator=g)
        plan = net.plan_for(x, True, second_order=True, param_tangent=True)
        plan.forward(x)
        clear = plan.clear_param_tangent
        with_dir = lambda: plan.set_param_tangent(*direction)
        tangent = lambda: plan.forward_tangent(dx)
        # name: (set-up outside the timed calls, timed call)
        passes = {"forward": (lambda: None, lambda: plan.forward(x)),
                  "tangent": (clear, tangent),
                  "second_order": (lambda: (clear(), tangent()), lambda: plan.backward_second_order(u, du)),
                  "tangent_with_params": (with_dir, tangent),
                  "second_order_with_params": (lambda: (with_dir(), tangent()),
                                               lambda: plan.backward_second_order(u, du)),
                  "params_call": (lambda: (with_dir(), tangent(), plan.backward_second_order(u, du)),
                                  lambda: plan.backward_second_order_params(grad=True)),
                  "params_call_hvp_only": (lambda: (with_dir(), tangent(), plan.backward_second_order(u, du)),
                                           lambda: plan.backward_second_order_params(grad=False))}
        times = {k: [] for k in passes}
        for r in range(a.rounds):
            for k, (setup, fn) in passes.items():
                setup()
                if r == 0:
                    for _ in range(a.warmup):
                        fn()
                times[k].append(time_ms(fn, a.steps))
        res[name] = {"workspace_GB": round(plan.workspace_bytes / 1e9, 2),
                     **{f"{k}_ms": [round(v, 3) for v in t] for k, t in times.items()}}
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
