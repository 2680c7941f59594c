"""Benchmarks of the B200 3D U-Net engine at the BASELINE.json configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W]                 # headline: cfg2 = UNet3D f32 d4, 2x1x128^3, fwd+BCEDice+bwd
    python bench.py --workload cfg3|cfg4|cfg5 ...                       # ResidualUNet3D 4x96^3 | ResidualUNetSE3D 1x160^3 | sliding window
    python bench.py --impl reference ...                                # the reference's own torch-CPU path (oracle port), all host cores
    python bench.py --impl torch-gpu ...                                # the reference's own GPU path: torch eager + cuDNN on this B200
                                                                        # (arms: fp32 NCDHW as shipped, bf16 autocast + channels_last_3d)
    python bench.py --dump-outputs DIR ...                              # also write what the last timed step returned, DIR/<name>.npy

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for the definition of every field.  A "step" of the training
workloads = zero grads, model(x, return_logits=True), BCEDiceLoss(logits, target), backward, gradient allreduce (N > 1); the optimizer
step is timed separately (`adam_ms`), as the reference reports it separately too (SURVEY.md section 8(d)).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# BASELINE.json configs[1..4]; GFLOP per patch: SURVEY.md section 8(a) table (conv/deconv/linear MACs x 2; bwd = dgrad + wgrad)
WORKLOADS = {
    "cfg2": dict(cfg=dict(name="UNet3D", in_channels=1, out_channels=1, f_maps=32, num_levels=4), batch=2, size=128, gflop=2841.5,
                 text="UNet3D f_maps=32 depth=4, batch 2x1x128^3, fwd+BCEDiceLoss+bwd (BASELINE cfg 2)",
                 metric="UNet3D patches/sec (1x128^3 bf16) train step"),
    "cfg3": dict(cfg=dict(name="ResidualUNet3D", in_channels=1, out_channels=1, f_maps=32), batch=4, size=96, gflop=1190.7,
                 text="ResidualUNet3D f_maps=32 (5 levels), batch 4x1x96^3 per GPU, fwd+BCEDiceLoss+bwd + NCCL grad allreduce (BASELINE cfg 3)",
                 metric="ResidualUNet3D patches/sec (1x96^3 bf16) train step"),
    "cfg4": dict(cfg=dict(name="ResidualUNetSE3D", in_channels=1, out_channels=1, f_maps=64), batch=1, size=160, gflop=22052.1,
                 text="ResidualUNetSE3D f_maps=64 (5 levels), batch 1x1x160^3, fwd+BCEDiceLoss+bwd (BASELINE cfg 4)",
                 metric="ResidualUNetSE3D patches/sec (1x160^3) train step"),
    "cfg5": dict(cfg=dict(name="UNet3D", in_channels=1, out_channels=1, f_maps=32, num_levels=4), batch=1, size=128, gflop=947.8,
                 volume=(256, 512, 512), patch=(128, 128, 128), stride=(64, 64, 64),
                 text="predict: UNet3D f_maps=32 depth=4 sliding window over a 256x512x512 volume, 128^3 patches stride 64 (147 patches), "
                      "patch i -> GPU i mod N (BASELINE cfg 5)",
                 metric="UNet3D sliding-window inference patches/sec (128^3 patches, stride 64)"),
}

DUMP_MAX_ELEMS = 1 << 22   # 16 MB of float32 per dumped array; the training path writes three of them and the loss


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "torch-gpu"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--size", type=int, default=None)
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--operand-dtype", default=None, choices=["bf16", "fp16"], help="16-bit type of activations / tensor-core operands "
                    "(default: fp16 for cfg4, as BASELINE names it; bf16 otherwise)")
    ap.add_argument("--buckets", type=int, default=4, help="gradient allreduce buckets (launched as backward finishes them)")
    ap.add_argument("--fused-loss", type=int, default=int(os.environ.get("B200UNET_FUSED_LOSS", "1")),
                    help="1: BCEDiceLoss through the engine's two-pass kernels (csrc/loss_ops.cu) instead of eager torch ops")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (rank 0) as DIR/<name>.npy in float32; "
                         "an array of more than %d elements is written as a fixed seeded sample of its flattened values" % DUMP_MAX_ELEMS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 engine's path (--impl b200)")
    return args


def dump_outputs(out_dir, arrays):
    """Write each tensor as out_dir/<name>.npy (float32).  Larger ones: the values at 2^22 flat indices drawn with a fixed seed
    (sorted, duplicates dropped), so that two builds given the same arguments write comparable files."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = torch.randint(t.numel(), (DUMP_MAX_ELEMS,), generator=torch.Generator().manual_seed(0)).unique()
            t = t.flatten()[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], False
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "samples": len(self.rows), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------------------------
# reference arms (the oracle port = plain torch ops = what the reference executes; the reference package cannot travel)
# ----------------------------------------------------------------------------------------------------------------------
def cpu_reference_steps(wl, size, batch, steps, warmup, forward_only=False):
    """The reference's own torch-CPU path on ALL host cores (whatever OMP_NUM_THREADS the launcher exported).  Seconds per step (median)."""
    import torch
    from oracle import unet3d_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    cfg = wl["cfg"]
    sd = {k: v.requires_grad_(not forward_only) for k, v in O.random_state_dict(cfg, seed=0).items()}
    x = torch.rand(batch, 1, size, size, size)
    t = (torch.rand(batch, 1, size, size, size) > 0.5).float()
    times = []
    for i in range(warmup + steps):
        for v in sd.values():
            v.grad = None
        t0 = time.perf_counter()
        if forward_only:
            with torch.no_grad():
                O.forward(sd, cfg, x)
        else:
            _, logits = O.forward(sd, cfg, x)
            O.bce_dice_loss(logits, t).backward()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    times.sort()
    return times[len(times) // 2], torch.get_num_threads()


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    size = args.size or wl["size"]
    inference = args.workload == "cfg5"
    # bounded sample: ONE patch of the workload's size per step (cfg4: 96^3 instead of 160^3 -- a 160^3 f64 step is ~minutes on CPU)
    sample_size = min(size, 96) if args.workload == "cfg4" else size
    steps = args.steps
    warm = min(args.warmup, 1)
    sec, threads = cpu_reference_steps(wl, sample_size, 1, steps, warm, forward_only=inference)
    scale = (size / sample_size) ** 3  # FLOP-proportional extrapolation when the sample patch is smaller than the workload's
    val = 1.0 / (sec * scale)
    sample = (f"{steps} steps x 1 patch {sample_size}^3 {'forward only' if inference else 'fwd+BCEDice+bwd'}, fp32, torch CPU ({threads} threads) "
              f"via oracle/unet3d_oracle.py" + (f"; extrapolated x{scale:.2f} by FLOPs to {size}^3" if scale != 1.0 else ""))
    line = {"metric": wl["metric"], "value": val, "unit": "patches/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": wl["text"], "sample": sample, "note": "batch 1 per step (patches/s is batch-independent on the CPU path)"},
            "cpu_baseline": {"value": val, "unit": "patches/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "patches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


def torch_gpu_arm(wl, batch, size, steps, warmup, dev, bf16, forward_only=False):
    """The reference's GPU path = the same torch ops dispatched to cuDNN.  bf16=False: fp32 NCDHW eager as shipped (TF32 off);
    bf16=True: best-effort torch, autocast(bfloat16) + channels_last_3d.  Returns ms per step (CUDA events)."""
    import torch
    from oracle import unet3d_oracle as O
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = True
    cfg = wl["cfg"]
    torch.manual_seed(0)
    sd = {k: v.to(dev).requires_grad_(not forward_only) for k, v in O.random_state_dict(cfg, seed=0).items()}
    if bf16:
        sd = {k: (v.detach().to(memory_format=torch.channels_last_3d).requires_grad_(not forward_only) if v.dim() == 5 else v) for k, v in sd.items()}
    x = torch.rand(batch, 1, size, size, size, device=dev)
    t = (torch.rand(batch, 1, size, size, size, device=dev) > 0.5).float()
    if bf16:
        x = x.to(memory_format=torch.channels_last_3d)

    def step():
        for v in sd.values():
            v.grad = None
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=bf16):
            if forward_only:
                with torch.no_grad():
                    O.forward(sd, cfg, x)
                return
            _, logits = O.forward(sd, cfg, x)
        O.bce_dice_loss(logits.float(), t).backward()

    for _ in range(max(warmup, 3)):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    del sd, x, t
    torch.cuda.empty_cache()
    return ms


def gpu_baseline(wl, batch, size, dev, forward_only=False, steps=5):
    out = {}
    for key, bf in (("fp32_eager_ncdhw", False), ("bf16_autocast_channels_last_3d", True)):
        try:
            ms = torch_gpu_arm(wl, batch, size, steps, 3, dev, bf, forward_only)
            out[key] = {"ms_per_step": ms, "patches_per_s": batch / (ms / 1e3)}
        except Exception as e:  # e.g. out of memory at cfg4 in fp32
            out[key] = {"error": f"{type(e).__name__}: {str(e)[:160]}"}
    out["what"] = "the reference's own GPU path (same torch ops -> cuDNN) on this GPU, same batch / size / loss, CUDA events, 3 warm-up + %d timed steps" % steps
    return out


def run_torch_gpu(args, wl):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    B, S = args.batch or wl["batch"], args.size or wl["size"]
    inference = args.workload == "cfg5"
    gb = gpu_baseline(wl, B, S, dev, forward_only=inference, steps=args.steps)
    best = min((v["ms_per_step"] for v in gb.values() if isinstance(v, dict) and "ms_per_step" in v), default=None)
    line = {"metric": wl["metric"], "value": (B / (best / 1e3)) if best else None, "unit": "patches/s", "n_gpus": 1, "steps": args.steps,
            "warmup": 3, "ms_per_step": best, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "impl": "torch-gpu", "config": {"workload": wl["text"], "per_gpu_batch": B}, "gpu_baseline": gb}
    print(json.dumps(line))


ALLOC_SETTLE_STEPS = 8


# ----------------------------------------------------------------------------------------------------------------------
# training workloads (cfg2 / cfg3 / cfg4)
# ----------------------------------------------------------------------------------------------------------------------
def run_train(args, wl):
    import torch
    import torch.distributed as dist
    import pytorch3dunet_b200 as P
    from pytorch3dunet_b200 import engine as E

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    torch.manual_seed(0)  # identical replicas on every rank (the reference's DataParallel broadcasts rank-0 weights)
    odt = args.operand_dtype or ("fp16" if args.workload == "cfg4" else "bf16")
    model = P.get_model({**wl["cfg"], "operand_dtype": odt}).to(dev)
    flat = P.optim.FlatParameters(model)          # parameters / gradients as views of two flat buffers; the engine writes wgrads in place
    reducer = P.optim.BucketedAllReduce(flat, world, n_buckets=args.buckets)
    adam = P.optim.FusedAdam(flat, lr=2e-4, weight_decay=1e-5, grad_scale=1.0 / world)   # the shipped configs' optimizer (utils.py:246-316)
    torch.manual_seed(1000 + rank)  # rank-dependent synthetic patches (weak scaling: per-GPU batch fixed)
    B, S = args.batch or wl["batch"], args.size or wl["size"]
    x_host = torch.rand(B, 1, S, S, S).pin_memory()
    t_host = (torch.rand(B, 1, S, S, S) > 0.5).float().pin_memory()
    x_dev, t_dev = x_host.to(dev), t_host.to(dev)

    def step(x, t):
        out, logits = model(x, return_logits=True)
        loss = P.losses.bce_dice_loss(logits, t, fused=bool(args.fused_loss))
        loss.backward()     # gradients land in flat.grad; each bucket's allreduce starts as soon as backward has written it
        reducer.finish()    # one sum-allreduce of every gradient per step over NVLink (replaces DataParallel's reduce-to-GPU-0)
        return out, logits, loss

    last = {}

    def timed_step():
        res = step(x_dev, t_dev)
        if args.dump_outputs:
            last["step"] = res

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    # setup, not warm-up: let torch's caching allocator reach its steady state (it keeps cudaMalloc-ing new segments -- a device
    # synchronisation each -- for the first ~8 identical steps while its best-fit split pattern converges; tools/alloc_probe.py)
    for _ in range(ALLOC_SETTLE_STEPS):
        step(x_dev, t_dev)
    W = max(args.warmup, 3)
    for _ in range(W):
        step(x_dev, t_dev)
    barrier()
    fwd_l, bwd_l = P.last_launch_counts()

    # ---- timed region 1 (`value`): inputs resident in HBM, no instrumentation ----
    with ClockSampler(local) as clk:
        ms = timed(timed_step, args.steps)
    patches = world * B * args.steps
    value = patches / (ms / 1e3)
    if args.dump_outputs and rank == 0:   # before later steps overwrite the gradients (the engine writes them in place)
        out, logits, loss = last.pop("step")
        dump_outputs(args.dump_outputs, {"probabilities": out, "logits": logits, "loss": loss,
                                         "param_grads": torch.cat([p.grad.flatten() for p in model.parameters()])})
        del out, logits, loss

    # ---- timed region 2 (`e2e`): through the public nn.Module API with HOST buffers: pinned H2D of input + target on a copy stream,
    # double-buffered against the previous step's compute, loss read back every step (trainer.py:241) ----
    copy_stream = torch.cuda.Stream(dev)
    staged = {}

    def stage():
        with torch.cuda.stream(copy_stream):
            xs = x_host.to(dev, non_blocking=True)
            ts = t_host.to(dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        staged["next"] = (xs, ts, ev)

    def e2e_step():
        xs, ts, ev = staged.pop("next")
        torch.cuda.current_stream().wait_event(ev)
        xs.record_stream(torch.cuda.current_stream())
        ts.record_stream(torch.cuda.current_stream())
        _, _, loss = step(xs, ts)
        stage()                 # the next step's H2D copies run while this step's kernels drain
        return loss.item()      # device -> host read of the loss

    stage()
    e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    staged.clear()
    e2e_value = patches / (ms_e2e / 1e3)

    # ---- optimizer, reported separately ----
    adam_ms = timed(adam.step, args.steps) / args.steps

    # ---- roofline leg: per-launch CUDA events around the tensor-core conv launches, in a SEPARATE pass ----
    E.TIMING = []
    ms_instr = timed(lambda: step(x_dev, t_dev), 3)
    timing, E.TIMING = E.TIMING, None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk, pk_src = peaks()
    by = {}
    blocks = {}
    for tag, fl, a, b, layer in timing:
        d = by.setdefault(tag, [0.0, 0.0, 0])
        t_ms = a.elapsed_time(b)
        d[0] += fl
        d[1] += t_ms
        d[2] += 1
        if layer:
            bl = blocks.setdefault(layer.rstrip("."), {})
            e = bl.setdefault(tag.split("_")[0], [0.0, 0.0])
            e[0] += fl
            e[1] += t_ms
    tc = {k: v for k, v in by.items() if k.endswith("_tc")}
    tc_flops = sum(v[0] for v in tc.values())
    tc_ms = sum(v[1] for v in tc.values())
    achieved = tc_flops / (tc_ms / 1e3) / 1e12 if tc_ms > 0 else 0.0
    peak = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
    traffic, traffic_note = None, None
    try:  # dram bytes of the longest launch of the largest-share kernel, from the committed ncu --set full capture of one cfg-2 step
        prof = json.load(open(os.path.join(ROOT, "profiles", "ncu_r02_full_summary.json")))["conv3_zs_kernel<32, 2>"]
        mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        traffic = sum(float(prof[k]["value"]) * mult.get(prof[k]["unit"], 1.0) for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
        traffic_note = ("dram read+write bytes of ONE conv3_zs_kernel<32,2> launch, the longest of the step: decoders.2.SingleConv1's encoder "
                        "half, 32->32 @ 2x128^3 with the phase-conv result as residual input (algorithmic 805 MB = x + R + y; the plain "
                        "32->32 launches move 701 MB against 537 MB = x + y), profiles/ncu_r02_full_summary.md")
    except Exception:
        pass
    roofline = {"bound": "tensor", "kernel": "tcgen05 conv kernels: conv3_zs_kernel / conv3_upzs_kernel / conv3_updzs_kernel / conv3_igemm_kernel (fprop+dgrad), wgrad_hs_kernel / wgrad_up_kernel / wgrad_halo_kernel / conv3_wgrad_igemm_kernel",
                "achieved": achieved, "peak": peak,
                "unit": "TFLOP/s", "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_note": traffic_note,
                "peak_source": pk_src + " sustained bf16",
                "share_of_step": (tc_ms / 3) / (ms_instr / 3) if ms_instr else None,
                "measured_in": "a separate instrumented pass of 3 steps (per-launch CUDA events), not the pass that produced `value`",
                "per_kernel": {k: {"tflops": v[0] / (v[1] / 1e3) / 1e12 if v[1] else None, "ms_per_step": v[1] / 3, "launches_per_step": v[2] / 3}
                               for k, v in by.items()},
                # every fused block (SingleConv = GroupNorm + conv + activation): achieved TFLOP/s of its fprop / dgrad / wgrad launches
                # (algorithmic FLOPs as executed; a virtual-concat conv counts its encoder conv and its phase conv together) and the
                # fraction of the measured sustained bf16 peak
                "per_block": {name: {kind: {"ms": round(v[1] / 3, 4), "tflops": round(v[0] / (v[1] / 1e3) / 1e12, 1), "frac": round(v[0] / (v[1] / 1e3) / 1e12 / peak, 3)}
                                     for kind, v in kinds.items() if v[1] > 0} for name, kinds in blocks.items()}}

    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1:
        sample_size = min(S, 96) if args.workload == "cfg4" else S
        sec, threads = cpu_reference_steps(wl, sample_size, 1, 2, 1)
        scale = (S / sample_size) ** 3
        cpu_baseline = {"value": 1.0 / (sec * scale), "unit": "patches/s", "cores": threads, "kind": "port",
                        "sample": f"2 steps x 1 patch {sample_size}^3 fwd+BCEDice+bwd, fp32 torch CPU ({threads} threads) via oracle/unet3d_oracle.py"
                                  + (f"; x{scale:.2f} by FLOPs to {S}^3" if scale != 1.0 else "")}
    gb = None
    if not args.no_gpu_baseline and world == 1:
        del x_dev, t_dev
        model.zero_grad(set_to_none=True)
        torch.cuda.empty_cache()
        gb = gpu_baseline(wl, B, S, dev)
        for v in gb.values():
            if isinstance(v, dict) and "ms_per_step" in v:
                v["b200_speedup"] = v["ms_per_step"] / (ms / args.steps)

    line = {"metric": wl["metric"], "value": value, "unit": "patches/s", "n_gpus": world,
            "steps": args.steps, "warmup": W, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": odt, "data": "synthetic",
            "config": {"workload": wl["text"] if (S == wl["size"] and B == wl["batch"]) else f"{wl['cfg']['name']} batch {B}x1x{S}^3", "per_gpu_batch": B,
                       "parallelism": f"dp{world}", "l2": "per-step working set (~1 GB of bf16 activations per patch) >> 126 MB L2; no explicit flush",
                       "setup_steps_before_warmup": ALLOC_SETTLE_STEPS, "grad_allreduce_buckets": len(reducer.buckets) if world > 1 else 0,
                       "grad_bytes": flat.numel * 4, "loss": "fused b200 kernels" if args.fused_loss else "torch ops"},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "gpu_baseline": gb,
            "e2e": {"value": e2e_value, "unit": "patches/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": x_host.numel() * 4 + t_host.numel() * 4, "d2h_bytes_per_step": 4,
                    "staging": "pinned host buffers, copy stream, next step's H2D overlapped with this step's compute"},
            "adam_ms": adam_ms,
            "gpu_launches": (fwd_l + bwd_l + (3 if args.fused_loss else 0)) * args.steps, "clocks": clk.summary(),
            "tflops_effective": value * wl["gflop"] / 1e3}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------------------------------
# sliding-window inference (cfg5)
# ----------------------------------------------------------------------------------------------------------------------
def run_predict(args, wl):
    import numpy as np
    import torch
    import torch.distributed as dist
    import pytorch3dunet_b200 as P

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(0)
    model = P.get_model(wl["cfg"]).to(dev).eval()
    np.random.seed(0)
    vol = np.random.rand(*wl["volume"]).astype(np.float32)     # (Z,Y,X), SURVEY.md section 8(d)
    vp = P.pipeline.VolumePredictor(model, wl["patch"], wl["stride"], (0, 0, 0), device=dev, world=world, rank=rank)
    dvol = torch.from_numpy(vol)[None].to(dev)
    n_patches = len(P.pipeline.PatchPlan(wl["volume"], wl["patch"], wl["stride"]))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    def device_volume():   # volume resident in HBM -> output volume resident in HBM (+ the cross-GPU merge)
        out = vp.predict_device(dvol)
        if world > 1:
            dist.reduce(out, dst=0, op=dist.ReduceOp.SUM)
        return out

    def host_volume():     # host array in -> host array out: staging ring + H2D, patches, write-back, D2H
        return vp.predict(vol)

    last = {}

    def timed_volume():
        out = device_volume()
        if args.dump_outputs:
            last["out"] = out

    steps = args.steps
    W = max(args.warmup, 3)
    for _ in range(W):
        device_volume()
    with ClockSampler(local) as clk:
        ms = timed(timed_volume, steps)
    fwd_l, _ = P.last_launch_counts()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"probabilities": last.pop("out")})
    host_volume()
    t0 = time.perf_counter()
    ms_e2e = timed(host_volume, steps)
    wall_e2e = (time.perf_counter() - t0) * 1e3
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk, pk_src = peaks()
    value = n_patches * steps / (ms / 1e3)
    e2e_value = n_patches * steps / (ms_e2e / 1e3)
    peak = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
    achieved = value * wl["gflop"] / 1e3
    gb = None
    if not args.no_gpu_baseline and world == 1:
        gb = gpu_baseline(wl, 1, wl["size"], dev, forward_only=True)
        for v in gb.values():
            if isinstance(v, dict) and "ms_per_step" in v:
                v["b200_speedup"] = v["ms_per_step"] / (ms / steps / n_patches)
    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1:
        sec, threads = cpu_reference_steps(wl, wl["size"], 1, 2, 1, forward_only=True)
        cpu_baseline = {"value": 1.0 / sec, "unit": "patches/s", "cores": threads, "kind": "port",
                        "sample": f"2 forward passes x 1 patch {wl['size']}^3, fp32 torch CPU ({threads} threads) via oracle/unet3d_oracle.py"}
    vol_bytes = int(np.prod(wl["volume"])) * 4
    line = {"metric": wl["metric"], "value": value, "unit": "patches/s", "n_gpus": world, "steps": steps, "warmup": W,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": wl["text"], "patches_per_volume": n_patches, "patches_on_busiest_gpu": -(-n_patches // world),
                       "step": "one whole volume", "parallelism": f"patch-sharded x{world}",
                       "l2": "every patch's activations (~0.5 GB bf16) >> 126 MB L2; no explicit flush"},
            "volumes_per_s": steps / (ms / 1e3),
            "roofline": {"bound": "tensor", "kernel": "whole forward pass (all tcgen05 conv launches + fused elementwise)", "achieved": achieved / world,
                         "peak": peak, "unit": "TFLOP/s", "frac": achieved / world / peak, "traffic": None, "peak_source": pk_src + " sustained bf16",
                         "note": "algorithmic forward FLOPs (947.8 GF/patch) x patches/s per GPU"},
            "cpu_baseline": cpu_baseline, "gpu_baseline": gb,
            "e2e": {"value": e2e_value, "unit": "patches/s", "ms_per_step": ms_e2e / steps, "volumes_per_s": steps / (ms_e2e / 1e3),
                    "host_wall_ms_per_volume": wall_e2e / steps,
                    "h2d_bytes_per_step": vol_bytes, "d2h_bytes_per_step": vol_bytes * wl["cfg"]["out_channels"],
                    "staging": "Z-slabs through a pinned ring on a copy stream; output rows of the patch grid copied back while later rows compute"},
            "gpu_launches": (fwd_l + 2) * (-(-n_patches // world)) * steps, "clocks": clk.summary()}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference(args, wl)
    if args.impl == "torch-gpu":
        return run_torch_gpu(args, wl)
    if args.workload == "cfg5":
        return run_predict(args, wl)
    return run_train(args, wl)


if __name__ == "__main__":
    main()
