"""Cost of dropout on the tensor-core engine, config-2 shape (16 x 3 x 512^2, 2 classes, dice_bce_mc, FusedSGD, CUDA graphs).

Prints one JSON object:
  * GPU name and power limit (read in the same run as the numbers);
  * ms/step and img/s of UNet(3, 2) and UNet(3, 2, dropout=True, dropout_p=0.5), alternated over several rounds;
  * a few steps of the generic fp32 engine on the dropout network (what dropout=True ran on before the tensor-core engine
    took it);
  * from a separate torch.profiler run: the kernel time of the dropout passes per step, the bytes they move, and a
    standalone comparison of one dropout pass with a plain copy of the same bytes (bound by bytes or by Philox instructions).

    python scripts/bench_dropout.py [--steps 20] [--rounds 3] [--generic-steps 2] [--out result.json]
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


def dropout_bytes(n, h, w, width=64):
    """Bytes one training step's dropout passes read and write: 8 sites, forward and backward, bf16 in place (2 B read +
    2 B written per element)."""
    elems = 0
    for l in range(4):
        elems += n * (h >> (l + 1)) * (w >> (l + 1)) * (width << l)    # pooled tensor of down(l + 1)
        elems += n * (h >> l) * (w >> l) * 2 * (width << l)            # concat tensor of level l
    return 2 * elems * 4


def make(dropout, args, dev):
    import unet_torch_b200 as U

    torch.manual_seed(0)
    net = U.UNet(3, 2, dropout=dropout, dropout_p=args.p).to(dev).train()
    return net


def timed(step, x, y, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        step(x, y)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--p", type=float, default=0.5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--generic-steps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dropout.py measures on a CUDA device; none is visible")
    import unet_torch_b200 as U
    from unet_torch_b200 import ops

    dev = torch.device("cuda", 0)
    U.loss.CLASS_NUMBER = 2
    n, s = args.batch, args.size
    g = torch.Generator(device=dev).manual_seed(1)
    x = torch.randn(n, 3, s, s, device=dev, generator=g)
    y = (torch.rand(n, s, s, device=dev, generator=g) > 0.5).float()
    res = {"gpu": gpu_info(), "shape": [n, 3, s, s], "p": args.p}

    legs = {}
    for name, dropout in (("dropout_off", False), ("dropout_on", True)):
        net = make(dropout, args, dev)
        opt = U.FusedSGD(net, **SGD)

        def step(xx, yy, net=net, opt=opt):
            loss = U.calc_loss(net(xx), yy, loss_type="dice_bce_mc")
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()

        step(x, y)
        net.enable_cuda_graphs(True, share_grads=True)
        for _ in range(max(args.warmup, 3)):
            step(x, y)
        legs[name] = (net, step)
    times = {k: [] for k in legs}
    for _ in range(args.rounds):
        for name, (_, step) in legs.items():
            times[name].append(timed(step, x, y, args.steps))
    for name, ts in times.items():
        ms = sorted(ts)[len(ts) // 2]
        res[name] = {"ms_per_step_rounds": [round(t, 3) for t in ts], "ms_per_step_median": round(ms, 3),
                     "img_per_s": round(n / (ms / 1e3), 1)}
    res["ratio_on_over_off"] = round(res["dropout_on"]["ms_per_step_median"] / res["dropout_off"]["ms_per_step_median"], 4)
    del legs
    torch.cuda.empty_cache()

    # ---- the generic fp32 engine on the dropout network
    if args.generic_steps > 0:
        net = make(True, args, dev).set_check_mode(True)
        opt = torch.optim.SGD(net.parameters(), **SGD)

        def gstep(xx, yy):
            loss = U.calc_loss(net(xx), yy, loss_type="dice_bce_mc")
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()

        try:
            gstep(x, y)
            ms = timed(gstep, x, y, args.generic_steps)
            res["generic_engine_dropout_on"] = {"ms_per_step": round(ms, 1), "img_per_s": round(n / (ms / 1e3), 2)}
        except RuntimeError as e:
            res["generic_engine_dropout_on"] = {"error": str(e)[:300]}
        del net, opt
        torch.cuda.empty_cache()

    # ---- kernel time of the dropout passes (separate run under the profiler, eager launches)
    from torch.profiler import ProfilerActivity, profile

    net = make(True, args, dev)
    opt = U.FusedSGD(net, **SGD)

    def pstep():
        loss = U.calc_loss(net(x), y, loss_type="dice_bce_mc")
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()

    for _ in range(2):
        pstep()
    torch.cuda.synchronize()
    k_steps = 3
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(k_steps):
            pstep()
        torch.cuda.synchronize()
    drop_us = total_us = 0.0
    launches = 0
    for e in prof.key_averages():
        if e.device_type != torch.autograd.DeviceType.CUDA or e.key.startswith(("Memset", "Memcpy")):
            continue
        t = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        total_us += t
        if "dropout_mul_kernel" in e.key:
            drop_us += t
            launches += e.count
    nbytes = dropout_bytes(n, s, s)
    drop_ms = drop_us / 1e3 / k_steps
    res["dropout_passes"] = {"launches_per_step": launches // k_steps, "kernel_ms_per_step": round(drop_ms, 3),
                             "kernel_ms_all_kernels_per_step": round(total_us / 1e3 / k_steps, 3),
                             "bytes_per_step": nbytes, "achieved_TB_per_s": round(nbytes / (drop_ms / 1e3) / 1e12, 2)}
    del net, opt
    torch.cuda.empty_cache()

    # ---- bytes or instructions: one dropout pass against a copy of the same bytes (concat of level 0: 1.07 GB at config 2)
    buf = torch.randn(n, s, s, 128, device=dev).to(torch.bfloat16)
    dst = torch.empty_like(buf)
    seed = torch.zeros(1, dtype=torch.int64, device=dev).random_()
    reps = 20

    def ev_time(fn):
        fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    t_drop = ev_time(lambda: ops.dropout_mul(buf, 4, seed, args.p))
    t_drop_sums = ev_time(lambda: ops.dropout_mul(buf, 4, seed, args.p, sums=(64, torch.empty(64, device=dev))))
    t_copy = ev_time(lambda: ops.nhwc_copy(buf, dst))
    b = buf.numel() * 2 * 2
    res["single_pass_level0_concat"] = {
        "bytes": b, "dropout_ms": round(t_drop, 3), "dropout_with_sums_ms": round(t_drop_sums, 3), "copy_ms": round(t_copy, 3),
        "dropout_TB_per_s": round(b / (t_drop / 1e3) / 1e12, 2), "copy_TB_per_s": round(b / (t_copy / 1e3) / 1e12, 2),
        "dropout_over_copy": round(t_drop / t_copy, 3)}
    res["wall_clock"] = time.strftime("%Y-%m-%d %H:%M:%S")
    out = json.dumps(res, indent=1)
    print(out)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(out)


if __name__ == "__main__":
    main()
