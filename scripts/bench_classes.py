"""Cost of many classes on the tensor-core engine at the config-2 shape (16 x 3 x 512^2, dice_bce_mc, FusedSGD, CUDA graphs).

Prints one JSON object:
  * GPU name and power limit (read in the same run as the numbers);
  * ms/step and img/s of UNet(3, 2) and UNet(3, C) (default C = 21), alternated over several rounds;
  * CUDA-event kernel times at C classes of the head forward, the loss forward and backward and the head backward, each next
    to a plain device copy of the same number of bytes timed in the same run (bytes from the shapes: what each kernel
    must read and write at least).

    python scripts/bench_classes.py [--classes 21] [--steps 20] [--rounds 3] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SGD = dict(lr=0.01, momentum=0.9, weight_decay=1e-4)


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit, max_sm_clock"] = r.stdout.strip()
    except Exception as e:  # noqa: BLE001
        info["power_limit, max_sm_clock"] = f"nvidia-smi unavailable ({e})"
    return info


def ev_time(fn, reps):
    fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--classes", type=int, default=21)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_classes.py measures on a CUDA device; none is visible")
    import unet_torch_b200 as U
    from unet_torch_b200 import ops

    dev = torch.device("cuda", 0)
    n, s, C = args.batch, args.size, args.classes
    g = torch.Generator(device=dev).manual_seed(1)
    x = torch.randn(n, 3, s, s, device=dev, generator=g)
    res = {"gpu": gpu_info(), "shape": [n, 3, s, s], "classes": C}

    legs = {}
    for ncls in (2, C):
        torch.manual_seed(0)
        net = U.UNet(3, ncls).to(dev).train()
        opt = U.FusedSGD(net, **SGD)
        y = torch.randint(0, ncls, (n, s, s), device=dev, generator=g).float()

        def step(net=net, opt=opt, y=y, ncls=ncls):
            U.loss.CLASS_NUMBER = ncls
            loss = U.calc_loss(net(x), y, loss_type="dice_bce_mc")
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()

        step()
        net.enable_cuda_graphs(True, share_grads=True)
        for _ in range(max(args.warmup, 3)):
            step()
        legs[ncls] = step
    times = {k: [] for k in legs}
    for _ in range(args.rounds):
        for ncls, step in legs.items():
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            times[ncls].append(e0.elapsed_time(e1) / args.steps)
    for ncls, ts in times.items():
        ms = sorted(ts)[len(ts) // 2]
        res[f"classes_{ncls}"] = {"ms_per_step_rounds": [round(t, 3) for t in ts], "ms_per_step_median": round(ms, 3),
                                  "img_per_s": round(n / (ms / 1e3), 1)}
    res["ratio_many_over_2"] = round(res[f"classes_{C}"]["ms_per_step_median"] / res["classes_2"]["ms_per_step_median"], 4)
    del legs
    torch.cuda.empty_cache()

    # ---- the four class-count-dependent kernels at C classes, each against a copy of the bytes it must move
    P = n * s * s
    a = torch.randn(n, s, s, 64, device=dev).to(torch.bfloat16)
    w = torch.randn(C, 64, 1, 1, device=dev) * 0.1
    b = torch.randn(C, device=dev) * 0.1
    logits = torch.empty(n, C, s, s, device=dev)
    ops.head_fprop(a, w, b, logits)
    y = torch.randint(0, C, (n, s, s), device=dev, generator=g).float()
    out, sums, _ = ops.loss_ce_dice_fwd(logits, y, 0)
    go = torch.ones(1, device=dev)
    dz = ops.loss_ce_dice_bwd(logits, y, sums, go, 0)
    da, dw, db = torch.empty_like(a), torch.empty_like(w), torch.empty_like(b)
    kernels = {
        # name: (call, bytes it reads + writes at least)
        "head_fprop": (lambda: ops.head_fprop(a, w, b, logits), P * (64 * 2 + C * 4)),
        "loss_fwd": (lambda: ops.loss_ce_dice_fwd(logits, y, 0), P * (C * 4 + 4)),
        "loss_bwd": (lambda: ops.loss_ce_dice_bwd(logits, y, sums, go, 0), P * (2 * C * 4 + 4)),
        # two kernels (da, then dW / db) each read dz: it crosses HBM twice
        "head_bwd": (lambda: ops.head_bwd(dz, a, w, da, dw, db), P * (2 * C * 4 + 64 * 2 * 2)),
    }
    src = torch.empty(max(v[1] for v in kernels.values()) // 2 // 4 + 1, dtype=torch.float32, device=dev)
    dst = torch.empty_like(src)
    res["kernels"] = {}
    for name, (fn, nbytes) in kernels.items():
        t = ev_time(fn, args.reps)
        m = nbytes // 2 // 4
        t_copy = ev_time(lambda m=m: dst[:m].copy_(src[:m]), args.reps)
        res["kernels"][name] = {"bytes": nbytes, "ms": round(t, 4), "TB_per_s": round(nbytes / (t / 1e3) / 1e12, 2),
                                "copy_ms": round(t_copy, 4), "copy_TB_per_s": round(nbytes / (t_copy / 1e3) / 1e12, 2),
                                "share_of_copy_rate": round(t_copy / t, 3)}
    res["wall_clock"] = time.strftime("%Y-%m-%d %H:%M:%S")
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
