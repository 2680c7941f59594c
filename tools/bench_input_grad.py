"""Timing of the input gradient at BASELINE cfg 2 (UNet3D f_maps=32, 4 levels, 2x1x128^3, BCEDice), CUDA events over K steps after W
warm-up steps (DESIGN.md section 6).  Prints one JSON line:
  train_ms            (a) training step (forward, loss, backward, fused Adam) without input gradient
  train_xgrad_ms      (b) the same with x.requires_grad
  frozen_ms           (c) every parameter frozen: forward, loss and the input gradient only
  frozen_torch_ms     (d) the same frozen step through the oracle on torch/cuDNN (bf16 autocast, channels_last_3d)
  kernel_us / kernel_TBps   the first layer's data-gradient kernel (b200_input_dgrad_conv3 with the GroupNorm partial sums) alone, and
                      its achieved bytes/s over the bytes it must move (dz read, x read, dx written), computed from the shapes
  apply_us            the GroupNorm-backward apply pass over dx that follows it

    python tools/bench_input_grad.py [--steps K] [--warmup W] [--size S] [--batch B]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines()[0].split(",") + ["?"])[:2]
    return name.strip(), power.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--size", type=int, default=128)
    ap.add_argument("--batch", type=int, default=2)
    args = ap.parse_args()
    import torch
    import pytorch3dunet_b200 as P
    from pytorch3dunet_b200._lib import lib
    from oracle import unet3d_oracle as O
    if not torch.cuda.is_available():
        raise SystemExit("bench_input_grad.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda")
    cfg = dict(name="UNet3D", in_channels=1, out_channels=1, f_maps=32, num_levels=4)
    B, S = args.batch, args.size
    torch.manual_seed(0)
    model = P.get_model(cfg).to(dev)
    frozen = P.get_model(cfg).to(dev)
    frozen.load_state_dict(model.state_dict())
    frozen.requires_grad_(False)
    flat = P.optim.FlatParameters(model)
    adam = P.optim.FusedAdam(flat, lr=2e-4, weight_decay=1e-5)
    x = torch.rand(B, 1, S, S, S, device=dev)
    t = (torch.rand(B, 1, S, S, S, device=dev) > 0.5).float()
    xg = x.clone().requires_grad_(True)

    def train(inp):
        def fn():
            inp.grad = None
            _, logits = model(inp, return_logits=True)
            P.losses.bce_dice_loss(logits, t).backward()
            adam.step()
        return fn

    def frozen_step():
        xg.grad = None
        _, logits = frozen(xg, return_logits=True)
        P.losses.bce_dice_loss(logits, t).backward()

    sd_t = {k: (v.detach().to(memory_format=torch.channels_last_3d) if v.dim() == 5 else v.detach()) for k, v in model.state_dict().items()}
    x_cl = x.to(memory_format=torch.channels_last_3d).requires_grad_(True)

    def frozen_torch():
        x_cl.grad = None
        with torch.autocast("cuda", dtype=torch.bfloat16):
            _, logits = O.forward(sd_t, cfg, x_cl)
        O.bce_dice_loss(logits.float(), t).backward()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    res = {}
    # (a) and (b) alternate twice so that a drift of the card shows up as a spread
    for rep in range(2):
        res.setdefault("train_ms", []).append(timed(train(x), args.steps, args.warmup))
        res.setdefault("train_xgrad_ms", []).append(timed(train(xg), args.steps, args.warmup))
    res["frozen_ms"] = [timed(frozen_step, args.steps, args.warmup)]
    res["frozen_torch_ms"] = [timed(frozen_torch, args.steps, args.warmup)]

    # the first layer's data gradient alone (cfg 2: C_in 1 -> C_out 16, GroupNorm in front: partial sums on)
    L = lib()
    stream = torch.cuda.current_stream().cuda_stream
    cout = 16
    W = torch.randn(cout, 1, 3, 3, 3, device=dev) * 0.2
    dz = torch.randn(B, S, S, S, cout, device=dev).bfloat16()
    dx = torch.empty(B, 1, S, S, S, device=dev)
    Pn = L.query("b200_input_dgrad_partials_count", B, S, S, S, 1, cout)
    parts = torch.empty(B, Pn, 1, 2, device=dev)
    coef = torch.rand(B, 1, 3, device=dev)
    vox = S ** 3
    kernel = lambda: L.call("b200_input_dgrad_conv3", dz.data_ptr(), W.data_ptr(), B, S, S, S, 1, cout, 1.0, x.data_ptr(), dx.data_ptr(),  # noqa: E731
                            parts.data_ptr(), stream)
    apply = lambda: L.call("b200_gn_bwd_apply_ncdhw_f32", dx.data_ptr(), x.data_ptr(), coef.data_ptr(), B, 1, vox, 1.0, dx.data_ptr(), stream)  # noqa: E731
    kms = timed(kernel, 50, 5)
    ams = timed(apply, 50, 5)
    kbytes = B * vox * (cout * 2 + 4 + 4)
    name, power = _card()
    out = {"tool": "bench_input_grad", "card": name, "power_limit": power, "workload": f"cfg2 UNet3D f32 d4 {B}x1x{S}^3 BCEDice",
           "steps": args.steps, "warmup": args.warmup,
           **{k: [round(v, 3) for v in vs] for k, vs in res.items()},
           "kernel_us": round(kms * 1e3, 2), "kernel_bytes": kbytes, "kernel_TBps": round(kbytes / (kms * 1e-3) / 1e12, 3),
           "apply_us": round(ams * 1e3, 2), "apply_TBps": round(B * vox * 12 / (ams * 1e-3) / 1e12, 3)}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
