"""Cost of H and W that are not multiples of 16 on the tensor-core engine (`UNet.allow_unaligned_sizes()`).

Prints one JSON object:
  * GPU name and power limit (read in the same run as the numbers);
  * training (UNet(3, 2), dice_bce_mc, FusedSGD, CUDA graphs): ms/step and img/s at 16 x 3 x 500^2 and 16 x 3 x 512^2,
    alternated over several rounds;
  * inference (`predict`, UNet(3, 5), eval): ms/call and img/s at 32 x 3 x 1000^2 and 32 x 3 x 1024^2, alternated;
  * the generic fp32 engine (what a 500^2 input runs on without the opt-in) for two training steps at 16 x 3 x 500^2.

At 500^2 the levels are 500, 250, 125, 62, 31: two of the four concat levels are odd. Its 16 x 8 tile count is 98 % of
512^2's (32 x 63 vs 32 x 64 tiles at level 0), so the target is a 500^2 step no slower than a 512^2 step.

    python scripts/bench_unaligned.py [--steps 20] [--rounds 3] [--out result.json]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402

from bench_classes import SGD, gpu_info  # noqa: E402


def timed(fn, steps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def alternate(legs, steps, rounds, batch):
    times = {k: [] for k in legs}
    for _ in range(rounds):
        for k, fn in legs.items():
            times[k].append(timed(fn, steps))
    out = {}
    for k, ts in times.items():
        ms = sorted(ts)[len(ts) // 2]
        out[k] = {"ms_rounds": [round(t, 3) for t in ts], "ms_median": round(ms, 3), "img_per_s": round(batch / (ms / 1e3), 1)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--infer-batch", type=int, default=32)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--generic-steps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_unaligned.py measures on a CUDA device; none is visible")
    import unet_torch_b200 as U
    from unet_torch_b200.generic import GenericEngine
    from unet_torch_b200.model import UNetEngine

    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1)
    res = {"gpu": gpu_info()}

    # ---- training
    n = args.batch
    legs = {}
    for s in (500, 512):
        torch.manual_seed(0)
        net = U.UNet(3, 2).allow_unaligned_sizes().to(dev).train()
        opt = U.FusedSGD(net, **SGD)
        x = torch.randn(n, 3, s, s, device=dev, generator=g)
        y = torch.randint(0, 2, (n, s, s), device=dev, generator=g).float()
        assert isinstance(net._engine_for(x), UNetEngine)

        def step(net=net, opt=opt, x=x, y=y):
            U.loss.CLASS_NUMBER = 2
            loss = U.calc_loss(net(x), y, loss_type="dice_bce_mc")
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()

        step()
        net.enable_cuda_graphs(True, share_grads=True)
        for _ in range(max(args.warmup, 3)):
            step()
        legs[f"train_{s}"] = step
    res["train"] = {"shapes": {f"train_{s}": [n, 3, s, s] for s in (500, 512)}}
    res["train"].update(alternate(legs, args.steps, args.rounds, n))
    res["train"]["ratio_500_over_512"] = round(res["train"]["train_500"]["ms_median"] / res["train"]["train_512"]["ms_median"], 4)
    del legs, net, opt
    torch.cuda.empty_cache()

    # ---- inference
    m = args.infer_batch
    legs = {}
    for s in (1000, 1024):
        torch.manual_seed(0)
        net = U.UNet(3, 5).allow_unaligned_sizes().to(dev).eval()
        x = torch.randn(m, 3, s, s, device=dev, generator=g)

        def infer(net=net, x=x):
            with torch.no_grad():
                net.predict(x)

        for _ in range(max(args.warmup, 2)):
            infer()
        legs[f"predict_{s}"] = infer
    res["predict"] = {"shapes": {f"predict_{s}": [m, 3, s, s] for s in (1000, 1024)}}
    res["predict"].update(alternate(legs, max(args.steps // 4, 3), args.rounds, m))
    res["predict"]["ratio_1000_over_1024"] = round(res["predict"]["predict_1000"]["ms_median"] /
                                                   res["predict"]["predict_1024"]["ms_median"], 4)
    del legs, net
    torch.cuda.empty_cache()

    # ---- before: the generic fp32 engine at 500^2 (what the input runs on without allow_unaligned_sizes)
    torch.manual_seed(0)
    net = U.UNet(3, 2).to(dev).train()
    opt = torch.optim.SGD(net.parameters(), **SGD)
    x = torch.randn(n, 3, 500, 500, device=dev, generator=g)
    y = torch.randint(0, 2, (n, 500, 500), device=dev, generator=g).float()
    assert isinstance(net._engine_for(x), GenericEngine)

    def gstep():
        U.loss.CLASS_NUMBER = 2
        loss = U.calc_loss(net(x), y, loss_type="dice_bce_mc")
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()

    gstep()
    ms = timed(gstep, args.generic_steps)
    res["generic_fp32_train_500"] = {"ms_per_step": round(ms, 1), "img_per_s": round(n / (ms / 1e3), 2)}
    res["speedup_over_generic_500"] = round(ms / res["train"]["train_500"]["ms_median"], 1)
    res["wall_clock"] = time.strftime("%Y-%m-%d %H:%M:%S")
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
