#!/usr/bin/env python
"""Benchmark of the U-Net hot path (BASELINE.json metric: UNet train img/s @512^2 bf16).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME] [--dump-outputs DIR]

--config (default train512 = the headline, BASELINE.json configs[1]; the others give the remaining named shapes a line):
  train512       UNet(3,2) training step, 16 x 3x512x512 per GPU, dice_bce_mc + SGD; N > 1 = data parallel + SyncBN (weak)
  train512_g128  the same with configs[2]'s FIXED global batch 128 (128/N images per GPU; strong scaling)
  infer1024      configs[3]: UNet(3,5).eval(), 32 x 3x1024x1024 tiles -> uint8 class mask (replicas only at N > 1)
  reg768         configs[4]: regression head, F.relu + 'mseMC' + SGD, 8 x 3x768x768 per GPU
  attn512        UNet_attention(3,2) (Model.py:257-391, SURVEY 8f-4) training step at train512's shape

ours      : `value`   images/s with the batch already resident in HBM, CUDA-event timed, max over ranks.
            `e2e`     the same through the public API with HOST buffers: pinned-host -> device copy of inputs (and labels)
                      and a device -> host read of the result (loss / mask) inside the timed region, every step.
            `roofline` tcgen05 conv3x3 implicit-GEMM launches, algorithmic FLOPs / CUDA-event time of those launches.
            `cpu_baseline` the reference's CPU path timed on this box's host cores (rank 0, N = 1, bounded sample).
reference : the UNMODIFIED reference modules (oracle/_ref/Model.py + loss.py, staged by oracle/build_ref.py) running the
            same step on the host CPU with all host threads; each step is a bounded sample (fewer images) of the same
            workload. Falls back to the oracle port (kind "port") only if the staged copy is missing.

--dump-outputs DIR (ours): after the timed steps, the arrays the last timed step handed its caller are written as
DIR/<name>.npy (float32; float64 where the tensor is fp64 or integer): `loss`, `output` (the network output the loss saw),
`grad.<parameter>` and `state.<state_dict key>` (after the optimizer step) for training, `mask` for inference. Inputs and
initial weights are seeded, so two builds run with the same arguments can be compared array for array. An array of more
than 2^18 elements is cut to a fixed seeded sample of 2^18 of them (the same elements for the same size), which keeps
the whole dump within 64 MB.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SGD = dict(lr=0.01, momentum=0.9, weight_decay=1e-4)  # config.yml:15-18
# gflop_per_img: SURVEY.md section 8(d) (train = fwd + dgrad + wgrad; infer = fwd); conv_share = the part of it in the
# 3x3 conv fprop+dgrad launches the roofline object covers (train: 2 x 5889 - 14.5 of 18483 GFLOP per 16-image batch)
WORKLOADS = {
    "train512": dict(kind="train", ch=3, cls=2, H=512, W=512, batch=16, loss="dice_bce_mc", relu=False,
                     metric="unet_train_img_per_s_512", gflop_per_img=1155.21, scaling="weak", cpu_sample=4,
                     what="BASELINE configs[1]: UNet(3,2) training step (fwd + dice_bce_mc loss + bwd + SGD), 3x512x512"),
    "train512_g128": dict(kind="train", ch=3, cls=2, H=512, W=512, global_batch=128, loss="dice_bce_mc", relu=False,
                          metric="unet_train_img_per_s_512_global128", gflop_per_img=1155.21, scaling="strong", cpu_sample=4,
                          what="BASELINE configs[2]: UNet(3,2) data-parallel training step, FIXED global batch 128, 3x512x512"),
    "infer1024": dict(kind="infer", ch=3, cls=5, H=1024, W=1024, batch=32, loss=None, relu=False,
                      metric="unet_infer_img_per_s_1024", gflop_per_img=1541.89, scaling="weak", cpu_sample=2,
                      what="BASELINE configs[3]: UNet(3,5).eval() forward + softmax/argmax -> uint8 mask, 3x1024x1024 tiles"),
    "reg768": dict(kind="train", ch=3, cls=2, H=768, W=768, batch=8, loss="mseMC", relu=True,
                   metric="unet_train_img_per_s_768_regression", gflop_per_img=2599.23, scaling="weak", cpu_sample=2,
                   what="BASELINE configs[4]: UNet(3,2) regression training step (fwd + F.relu + mseMC loss + bwd + SGD), 3x768x768"),
    # SURVEY 8f rank 4: the attention-gated network (Model.py:257-391) at config 2's shape. gflop_per_img counts the gates as the
    # reference executes them (ConvTranspose2d C_q->C_q, two 1x1 convolutions, psi: 47.3 GFLOP forward per image); the B200
    # path composes up and W_q on the weight side and executes about a third of the gates' FLOPs.
    "attn512": dict(kind="train", model="UNet_attention", ch=3, cls=2, H=512, W=512, batch=16, loss="dice_bce_mc", relu=False,
                    metric="unet_attention_train_img_per_s_512", gflop_per_img=1297.0, scaling="weak", cpu_sample=2,
                    what="UNet_attention(3,2) training step (fwd + dice_bce_mc loss + bwd + SGD), 3x512x512"),
}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sust=p["bf16_tflops_sustained"], src="measured")
    except Exception:
        return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


def conv_traffic():
    """DRAM bytes per conv3x3 fprop/dgrad launch (dram__bytes_read.sum + dram__bytes_write.sum averaged over the launches
    of one train512 step) from the committed ncu capture of the current kernels, or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "conv_traffic.json")) as f:
            return json.load(f)["dram_bytes_per_launch"]
    except Exception:
        return None


DUMP_BYTES = 64_000_000   # --dump-outputs: the whole dump, .npy headers included
DUMP_ELEMS = 1 << 18       # --dump-outputs: elements kept of any one array


def dump_outputs(out_dir, arrays):
    """Write {name: tensor} as out_dir/<name>.npy. An array of more than DUMP_ELEMS elements is replaced by a fixed seeded
    sample of DUMP_ELEMS of its flattened elements, in index order. The sample depends on nothing but the array's own size,
    so the dumps of two builds line up element for element even where their sets of arrays differ.
    Returns (bytes of data, sampled names)."""
    import numpy as np

    wide = {k: t.dtype in (torch.float64, torch.int64, torch.int32) for k, t in arrays.items()}  # exact in float64 only
    nbytes = sum(min(t.numel(), DUMP_ELEMS) * (8 if wide[k] else 4) + 256 for k, t in arrays.items())
    if nbytes > DUMP_BYTES:
        raise RuntimeError(f"--dump-outputs: {len(arrays)} arrays need {nbytes} bytes, more than {DUMP_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    sampled = []
    for k, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_ELEMS:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_ELEMS].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
            sampled.append(k)
        a = t.to(torch.float64 if wide[k] else torch.float32).cpu().numpy()
        np.save(os.path.join(out_dir, k + ".npy"), a)
    return nbytes, sampled


def batch_per_gpu(wl, n_gpus):
    if "global_batch" in wl:
        if wl["global_batch"] % n_gpus:
            raise SystemExit(f"global batch {wl['global_batch']} does not divide over {n_gpus} GPUs")
        return wl["global_batch"] // n_gpus
    return wl["batch"]


def workload_config(name, n_gpus):
    """Identical for both arms: it names the workload, not how an arm executes it."""
    wl = WORKLOADS[name]
    b = batch_per_gpu(wl, n_gpus)
    par = "single" if n_gpus == 1 else (f"replicas{n_gpus}" if wl["kind"] == "infer" else f"dp{n_gpus}")
    cfg = {
        "workload": f"{wl['what']}, batch {b} per GPU"
                    + (", data parallel + SyncBN" if n_gpus > 1 and wl["kind"] == "train" else ""),
        "name": name, "global_batch": b * n_gpus, "image": [wl["ch"], wl["H"], wl["W"]], "n_classes": wl["cls"],
        "loss": ("relu+" if wl["relu"] else "") + wl["loss"] if wl["loss"] else None,
        "optimizer": "SGD(lr=0.01, momentum=0.9, weight_decay=1e-4)" if wl["kind"] == "train" else None,
        "parallelism": par,
        "l2": "per-step working set (GBs of bf16 activations) is far larger than the 126 MB L2; no explicit flush",
    }
    return cfg


class ClockSampler:
    """nvidia-smi clocks / throttle reasons. The process is started before the warm-up (its start-up takes longer than
    a short timed region); only samples that ARRIVE between mark_begin() and mark_end() are reported."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.proc = index, [], None
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.perf_counter(), line.strip()))

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        t0 = self.t0 if self.t0 is not None else 0.0
        t1 = (self.t1 if self.t1 is not None else time.perf_counter()) + 0.06  # a sample describes the period before it
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, s in self.samples:
            if t < t0 or t > t1:
                continue
            parts = [p.strip() for p in s.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------- reference arm
def synthetic_batch(wl, batch, seed):
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(batch, wl["ch"], wl["H"], wl["W"], generator=gen)
    if wl["kind"] == "infer":
        return x, None
    if wl["loss"] == "mseMC":  # density x 200, sparse (DataLoader.py:369-370)
        y = torch.rand(batch, wl["cls"], wl["H"], wl["W"], generator=gen) * 200.0 * (
            torch.rand(batch, wl["cls"], wl["H"], wl["W"], generator=gen) > 0.9)
    else:
        y = torch.randint(0, wl["cls"], (batch, wl["H"], wl["W"]), generator=gen).float()
    return x, y


def reference_cpu_step(wl, batch, seed=0):
    """step() = the workload's step on the host CPU in fp32 through the reference's own modules (kind "reference":
    oracle/_ref/Model.py + loss.py, unmodified), or through the oracle port when the staged copy is missing."""
    from oracle import ref_loader

    x, y = synthetic_batch(wl, batch, 1234 + seed)
    if ref_loader.available():
        RefModel, ref_loss = ref_loader.load()
        torch.manual_seed(seed)
        net = getattr(RefModel, wl.get("model", "UNet"))(wl["ch"], wl["cls"])
        ref_loss.CLASS_NUMBER = wl["cls"]
        if wl["kind"] == "infer":
            net.eval()

            def step():  # test_mc3serousv5.py:878-887
                with torch.no_grad():
                    out = net(x)
                    return torch.argmax(torch.nn.functional.softmax(out, dim=1), dim=1).to(torch.uint8)
        else:
            net.train()
            opt = torch.optim.SGD(net.parameters(), **SGD)

            def step():  # Trainer.py:706-722
                out = net(x)
                if wl["relu"]:
                    out = torch.nn.functional.relu(out)
                loss = ref_loss.calc_loss(out, y, loss_type=wl["loss"])
                opt.zero_grad()
                loss.backward()
                opt.step()
                return float(loss)
        return step, "reference"
    from oracle import cpu_baseline

    if wl.get("model", "UNet") != "UNet":
        raise RuntimeError(f"the oracle port covers UNet only; workload {wl['metric']} needs the staged reference (oracle/_ref, "
                           "python oracle/build_ref.py in the build container)")
    return cpu_baseline.make_step(wl["ch"], wl["cls"], batch, wl["H"], wl["W"], seed, loss_type=wl["loss"],
                                  relu=wl["relu"], train=wl["kind"] == "train", sgd=SGD), "port"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = WORKLOADS[args.config]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    batch = min(wl["cpu_sample"], batch_per_gpu(wl, args.gpus))
    try:
        step, kind = reference_cpu_step(wl, batch)
    except RuntimeError as e:  # a workload without an oracle port on a box without the staged reference: say so, exit 0
        print(json.dumps({"impl": "reference", "unavailable": str(e).replace("\n", " ")}))
        return 0
    for _ in range(max(args.warmup, 0)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    v = batch / dt
    what = "fwd + loss + bwd + SGD" if wl["kind"] == "train" else "eval fwd + softmax/argmax"
    sample = (f"each step = {what} on a {batch}-image sample of the workload's batch, fp32, {torch.get_num_threads()} host "
              f"threads, " + ("unmodified reference Model.py + loss.py (oracle/_ref)" if kind == "reference"
                              else "oracle port (torch CPU ops the reference dispatches to)"))
    line = {
        "impl": "reference", "metric": wl["metric"], "value": v, "unit": "img/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.config, args.gpus),
        "cpu_baseline": {"value": v, "unit": "img/s", "cores": torch.get_num_threads(), "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def cpu_baseline_leg(wl):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    batch = 1 if wl["H"] * wl["W"] > 512 * 512 else 2
    step, kind = reference_cpu_step(wl, batch)
    step()  # warm-up
    n, t0 = 0, time.perf_counter()
    while n < 4 and time.perf_counter() - t0 < 20.0:
        step()
        n += 1
    dt = (time.perf_counter() - t0) / n
    what = "fwd + loss + bwd + SGD" if wl["kind"] == "train" else "eval fwd + softmax/argmax"
    return {"value": batch / dt, "unit": "img/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"{n} steps ({what}) of a {batch}-image sample, {wl['ch']}x{wl['H']}x{wl['W']} fp32, "
                      + ("unmodified reference Model.py + loss.py (oracle/_ref)" if kind == "reference" else "oracle port")}


# --------------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import unet_torch_b200 as U
    from unet_torch_b200 import _lib, ops

    wl = WORKLOADS[args.config]
    train = wl["kind"] == "train"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (impl=ours) needs a CUDA device: the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    dist_on = world > 1
    dp = U.init_from_env(sync_bn=True, graphs=not args.no_graphs) if dist_on else None
    if dist_on and not train:
        U.DataParallelContext.disable()  # inference: replicas only, no data-path collective (process group kept for timing)
        dp = None
    dev = torch.device("cuda", local)

    torch.manual_seed(0)
    net = getattr(U, wl.get("model", "UNet"))(wl["ch"], wl["cls"]).to(dev)
    net = net.train() if train else net.eval()
    U.loss.CLASS_NUMBER = wl["cls"]
    if dist_on:
        import torch.distributed as dist

        for p in list(net.parameters()) + list(net.buffers()):
            dist.broadcast(p.data, 0)
    opt = None
    if train:
        opt = torch.optim.SGD(net.parameters(), **SGD) if args.torch_optim else U.FusedSGD(net, **SGD)
    B, H, W = batch_per_gpu(wl, world), wl["H"], wl["W"]
    x_host, y_host = synthetic_batch(wl, B, 1234 + rank)
    x_host = x_host.pin_memory()
    x_dev = x_host.to(dev)
    y_dev = None
    if y_host is not None:
        y_host = y_host.pin_memory()
        y_dev = y_host.to(dev)

    # step() returns (what the timing reads back every step, the network output)
    if train:
        def step(x, y):
            out = net(x)
            if wl["relu"]:
                out = torch.nn.functional.relu(out)  # Trainer.py:709-710
            loss = U.calc_loss(out, y, loss_type=wl["loss"])
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
            return loss, out
    else:
        def step(x, y):
            with torch.no_grad():
                mask = net.predict(x)  # OutConv + softmax + argmax + uint8 fused (test_mc3serousv5.py:878-887)
            return mask, mask

    def barrier():
        if dist_on:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if dist_on:
            import torch.distributed as dist

            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # one eager step: configures the kernels and counts OUR launches per step (graph replays bypass the counter)
    l0 = _lib.query("b200unet_launch_count")
    step(x_dev, y_dev)
    launches_per_step = _lib.query("b200unet_launch_count") - l0
    use_graphs = train and not args.no_graphs
    net.enable_cuda_graphs(use_graphs, share_grads=use_graphs)  # step() clears gradients with set_to_none=True every step
    for _ in range(max(args.warmup, 3)):
        step(x_dev, y_dev)
    # what actually replays as a graph (data parallel: only with B200UNET_DP_GRAPHS=1 and the NVLink SyncBN path)
    graphs_live = bool(getattr(net, "_engine", None) is not None and net._engine._graphs)
    # ---- device-resident timing
    barrier()
    sampler.mark_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step(x_dev, y_dev)
    e1.record()
    barrier()
    sampler.mark_end()
    launches = launches_per_step * args.steps
    ms = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = ms / args.steps
    value = B * world * args.steps / (ms / 1e3)

    # ---- end to end: host buffers in, result out, every step
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # Double-buffered input pipeline (what a pin_memory DataLoader + non_blocking copies amount to): the pinned host batch
    # of step i+1 crosses PCIe on a copy stream into one of two persistent device buffers while step i computes.
    copy_stream = torch.cuda.Stream()
    cur = torch.cuda.current_stream()
    xbuf = [torch.empty_like(x_dev), torch.empty_like(x_dev)]
    ybuf = [torch.empty_like(y_dev), torch.empty_like(y_dev)] if y_dev is not None else [None, None]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    done = [torch.cuda.Event(), torch.cuda.Event()]

    def fetch(i):
        b = i & 1
        with torch.cuda.stream(copy_stream):
            if i >= 2:
                copy_stream.wait_event(done[b])  # the step that last read this buffer has finished
            xbuf[b].copy_(x_host, non_blocking=True)
            if y_host is not None:
                ybuf[b].copy_(y_host, non_blocking=True)
            ready[b].record(copy_stream)

    # The result of every step (loss scalar / uint8 mask) is copied to pinned host memory and read one step behind its
    # launch, so the host keeps enqueueing step i+1 while step i runs; all reads complete inside the timed region.
    res_shape = () if train else (B, H, W)
    res_dtype = torch.float32 if train else torch.uint8
    res_host = [torch.empty(res_shape, dtype=res_dtype).pin_memory() for _ in range(2)]
    res_ready = [torch.cuda.Event(), torch.cuda.Event()]
    torch.cuda.synchronize()
    e0.record()
    last = None
    fetch(0)
    for i in range(args.steps):
        b = i & 1
        if i + 1 < args.steps:
            fetch(i + 1)  # issued BEFORE this step's kernels, so it overlaps them; every step's inputs cross PCIe in the region
        cur.wait_event(ready[b])
        res, out = step(xbuf[b], ybuf[b])
        done[b].record(cur)
        res_host[b].copy_(res.detach(), non_blocking=True)  # device -> host read of the step's result, every step
        res_ready[b].record(cur)
        if i >= 1:
            res_ready[1 - b].synchronize()
            last = float(res_host[1 - b].float().mean())
    res_ready[(args.steps - 1) & 1].synchronize()
    last = float(res_host[(args.steps - 1) & 1].float().mean())
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    e2e_value = B * world * args.steps / (ms_e2e / 1e3)
    if args.dump_outputs and rank == 0:
        if train:
            arrays = {"loss": res, "output": out}
            arrays.update({"grad." + k: p.grad for k, p in net.named_parameters() if p.grad is not None})
            arrays.update({"state." + k: v for k, v in net.state_dict().items()})
        else:
            arrays = {"mask": res}
        nbytes, sampled = dump_outputs(args.dump_outputs, arrays)
        print(f"bench.py: {len(arrays)} arrays of the last timed step -> {args.dump_outputs} ({nbytes / 1e6:.1f} MB; "
              f"{len(sampled)} sampled)", file=sys.stderr)

    # ---- roofline of the dominant kernel class (tcgen05 conv3x3 implicit GEMM), CUDA events around each launch
    net.enable_cuda_graphs(False)  # per-launch CUDA events need the eager launch path
    prof = []
    orig, orig_eval = ops.conv3x3, ops.conv3x3_bn_relu

    def timed(fn, out_index):
        def wrapper(*a, **k):
            t0_, t1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0_.record()
            r = fn(*a, **k)
            t1_.record()
            x, out = a[0], a[out_index]
            n, h, w, cin = x.shape
            prof.append((2.0 * n * h * w * out.shape[3] * 9 * cin, t0_, t1_))
            return r
        return wrapper

    ops.conv3x3, ops.conv3x3_bn_relu = timed(orig, 2), timed(orig_eval, 4)
    try:
        for _ in range(2):
            step(x_dev, y_dev)
        torch.cuda.synchronize()
    finally:
        ops.conv3x3, ops.conv3x3_bn_relu = orig, orig_eval
    flops = sum(p[0] for p in prof)
    kms = sum(p[1].elapsed_time(p[2]) for p in prof)
    pk = peaks()
    achieved = flops / (kms / 1e3) / 1e12 if kms > 0 else 0.0
    step_tflop = B * wl["gflop_per_img"] / 1e3
    roofline = {"bound": "tensor",
                "kernel": "conv3x3 " + ("fprop+dgrad" if train else "fprop (BatchNorm+ReLU folded)")
                          + " implicit GEMMs (conv3_pair / conv3_res2 / conv3_res kernels, tcgen05); "
                          f"{len(prof) // 2} launches and {flops / 2 / 1e12:.2f} of the {step_tflop:.2f} TFLOP of a step",
                "achieved": achieved, "peak": pk["tf_sust"], "unit": "TFLOP/s", "frac": achieved / pk["tf_sust"],
                "peak_source": f"{pk['src']} bf16_tflops_sustained (kernels timed inside a long step)",
                "peak_burst": pk["tf_burst"], "frac_of_burst": achieved / pk["tf_burst"],
                "launches_timed": len(prof), "share_of_step": (kms / 2) / ms_per_step,
                "traffic": conv_traffic() if args.config == "train512" else None}

    if rank != 0:
        return 0
    if train:
        how = ("pinned host batch + labels -> one of two device buffers on a copy stream, one step ahead; the loss of every "
               "step is copied to pinned host memory and read one step behind its launch")
        h2d, d2h = int(x_host.numel() * 4 + y_host.numel() * 4), 4
    else:
        how = ("pinned host tiles -> one of two device buffers on a copy stream, one step ahead; the uint8 mask of every step "
               "is copied to pinned host memory and read one step behind its launch")
        h2d, d2h = int(x_host.numel() * 4), int(B * H * W)
    line = {
        "metric": wl["metric"], "value": value, "unit": "img/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": wl["scaling"],
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": workload_config(args.config, world),
        "execution": {
            "optimizer_impl": None if not train else ("torch.optim.SGD" if args.torch_optim else
                                                      "unet_torch_b200.FusedSGD (torch.optim.SGD arithmetic fused with the bf16 operand re-cast)"),
            "cuda_graphs": ("forward and backward of the network replayed as captured CUDA graphs (net.enable_cuda_graphs(True, "
                            "share_grads=True): .grad aliases the graph's gradient buffers); loss and optimizer eager"
                            if graphs_live else "off (every kernel launched eagerly)"),
            "sync_bn": bool(dp is not None and dp.sync_bn),
            "sync_bn_path": None if dp is None else ("nvlink peer-memory kernel" if dp.has_nvl else "nccl"),
        },
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "img/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / args.steps, "last_result_mean": last, "how": how},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "model_tflops": value * wl["gflop_per_img"] / 1e3 / world,
    }
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_leg(wl)
    print(json.dumps(line), flush=True)
    return 0


def _shutdown_dist():
    try:
        import torch.distributed as dist

        if dist.is_available() and dist.is_initialized():
            try:
                import unet_torch_b200 as U

                U.DataParallelContext.disable()  # drops CUDA graphs that captured NCCL kernels (they block the teardown)
            except Exception:
                pass
            dist.destroy_process_group()
    except Exception:
        pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="train512", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--torch-optim", action="store_true", help="step with stock torch.optim.SGD instead of FusedSGD")
    ap.add_argument("--no-graphs", action="store_true", help="launch every kernel eagerly (no CUDA-graph replay)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy (ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    try:
        return run_ours(args)
    finally:
        _shutdown_dist()


if __name__ == "__main__":
    sys.exit(main())
