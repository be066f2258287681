"""Stage-by-stage diagnostic of the CUDA path against torch fp32 references (run on the GPU box).

    python tests/tools/gpu_probe.py            # runs every stage in its own process (a CUDA fault in one
                                         # stage must not poison the others)
    python tests/tools/gpu_probe.py STAGE ...  # run the named stage(s) in-process
"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def _err(a, b):
    import torch
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def stage_raw(precision, B, C, hc, k, H, W, with_state):
    import torch
    import torch.nn.functional as F
    from nasa_niswan_b200 import Plan
    torch.manual_seed(0)
    dev = "cuda"
    x = torch.randn(B, 1, C, H, W, device=dev)
    w = torch.randn(4 * hc, C + hc, k, k, device=dev) * 0.1
    b = torch.randn(4 * hc, device=dev)
    plan = Plan(B, 1, H, W, C, [hc], [k], precision=precision, training=False)
    plan.set_weights(0, w, b)
    plan.set_head(torch.zeros(1, hc, 1, 1, device=dev), torch.zeros(1, device=dev))
    h0 = torch.randn(B, hc, H, W, device=dev) * 0.5
    c0 = torch.randn(B, hc, H, W, device=dev)
    if with_state:
        plan.set_state(0, h0, c0)
    got = plan.debug_raw_gates(x)
    torch.cuda.synchronize()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    comb = torch.cat([x[:, 0], h0 if with_state else torch.zeros_like(h0)], 1)
    ref = F.conv2d(comb.double().cpu(), w.double().cpu(), None, padding=k // 2)
    got = got.cpu()
    e = _err(got, ref)
    print(f"raw[{precision} B{B} C{C} hc{hc} k{k} {H}x{W} state={with_state}] err={e:.3e}")
    if e > 2e-2:
        d = (got - ref).abs()
        idx = torch.nonzero(d > 0.05 * ref.abs().max())[:10]
        print("  first bad idx (b,n,y,x):", idx.tolist())
        print("  per-channel-block err:", [round(float(d[:, i * hc:(i + 1) * hc].max()), 3) for i in range(4)])
        print("  err by row:", [round(float(d[:, :, y].max()), 2) for y in range(min(H, 16))])
        print("  err by col:", [round(float(d[:, :, :, xx].max()), 2) for xx in range(min(W, 32))])
    return e


def run_stage(name):
    import torch
    if name == "raw_bf16_small":
        stage_raw("bf16", 1, 21, 64, 3, 7, 18, False)
        stage_raw("bf16", 1, 21, 64, 3, 7, 18, True)
    elif name == "raw_bf16":
        stage_raw("bf16", 2, 21, 64, 3, 20, 24, True)
        stage_raw("bf16", 3, 8, 16, 5, 11, 13, True)
        stage_raw("bf16", 2, 21, 128, 3, 20, 24, True)
        stage_raw("bf16", 2, 5, 32, 5, 18, 22, True)
    elif name == "raw_tf32":
        stage_raw("tf32", 1, 21, 64, 3, 7, 18, True)
        stage_raw("tf32", 3, 8, 16, 5, 11, 13, True)
    elif name in ("fwd_bf16", "fwd_tf32", "bwd_bf16", "bwd_tf32"):
        from oracle.golden import load_case
        from nasa_niswan_b200 import ConvLSTM
        prec = name.split("_")[1]
        for case in ["lstm_c21_h32_k3", "lstm_c8_h16_k5", "lstm_3layer_k533"]:
            z = load_case(os.path.join(ROOT, "tests", "golden"), case)
            meta = z["meta"].tolist()
            B, T, cin, H, W, L = meta[:6]
            hidden, ks = meta[6:6 + L], meta[6 + L:6 + 2 * L]
            net = ConvLSTM(cin, hidden, ks, L, precision=prec).cuda()
            net.load_state_dict({k[6:]: torch.from_numpy(z[k]) for k in z if k.startswith("param/")})
            x = torch.from_numpy(z["x"]).cuda()
            if name.startswith("fwd"):
                with torch.no_grad():
                    pred = net(x)
                print(f"{name} {case}: pred err={_err(pred, torch.from_numpy(z['pred'])):.3e}")
            else:
                y = torch.from_numpy(z["y"]).cuda()
                crop = z["crop"].tolist()
                pred = net(x)
                p = pred if crop[0] < 0 else pred[:, :, crop[0]:crop[1], crop[2]:crop[3]]
                p = p.squeeze(1)
                loss = torch.nn.functional.mse_loss(p, y) + torch.nn.functional.l1_loss(p, y)
                loss.backward()
                print(f"{name} {case}: pred err={_err(pred.detach(), torch.from_numpy(z['pred'])):.3e} "
                      f"loss {float(loss):.6f} vs {float(z['loss']):.6f}")
                for k, v in net.named_parameters():
                    print(f"    grad {k}: err={_err(v.grad, torch.from_numpy(z['grad/' + k])):.3e}")
    else:
        raise SystemExit(f"unknown stage {name}")
    torch.cuda.synchronize()


STAGES = ["raw_bf16_small", "raw_bf16", "raw_tf32", "fwd_bf16", "fwd_tf32", "bwd_bf16", "bwd_tf32"]

if __name__ == "__main__":
    if len(sys.argv) > 1:
        for s in sys.argv[1:]:
            run_stage(s)
    else:
        for s in STAGES:
            t0 = time.time()
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), s], timeout=240, capture_output=True, text=True)
                out = (r.stdout + r.stderr).strip().splitlines()
                print(f"=== {s}: rc={r.returncode} ({time.time() - t0:.1f}s)")
                for line in out[-40:]:
                    print("   ", line)
            except subprocess.TimeoutExpired:
                print(f"=== {s}: TIMEOUT")
            sys.stdout.flush()
