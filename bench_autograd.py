#!/usr/bin/env python
"""
bench_autograd.py -- cost of the differentiable public methods of the VAE on one GPU.

    python bench_autograd.py [--batches 64 1024] [--iters 50] [--warmup 5]

For each batch size, the median over --iters iterations (CUDA events on the current stream,
after --warmup untimed iterations of the same shape) of:
  (a) train_fwd_bwd        loss = model(x); loss.backward()                in train mode
  (b) eval_fwd_bwd         the same in eval mode (BatchNorm with the running buffers)
  (c) train_fwd_bwd_xgrad  (a) with x.requires_grad (adds layer 0's data gradient and one
                           elementwise pass for the reconstruction term)
  (d) encode_bwd           the backward alone of encode(x) seeded on (mu, u, d)
  (e) decode_bwd           the backward alone of decode(z) seeded on x_rec
Prints one JSON line per (batch, case) with the device name and its power limit.  Inputs and
parameters are seeded; nothing is written to the tree.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
PKG = "autoencoded-vocal-analysis_b200"


def power_limit(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30)
        return out.stdout.strip() or None
    except Exception:
        return None


def timed(fn, iters, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        pre = fn.__dict__.get("prepare")
        if pre is not None:
            pre()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    times.sort()
    return times[len(times) // 2], times[0], times[-1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[64, 1024])
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_autograd.py needs a CUDA device")
    from oracle import vae_oracle
    vae = importlib.import_module(PKG + ".models.vae")
    torch.cuda.set_device(0)
    dev = {"device": torch.cuda.get_device_name(0), "power_limit": power_limit(0)}
    for B in args.batches:
        model = vae.VAE(save_dir='', device_name='cuda')
        model.load_flat_state(vae_oracle.make_params(0))
        x = vae_oracle.make_input(0, B).cuda()
        noise = tuple(t.cuda() for t in vae_oracle.make_noise(0, B))
        g = torch.Generator(device="cuda").manual_seed(1)
        seeds = [torch.randn(B, model.z_dim, device="cuda", generator=g) for _ in range(3)]
        seed_x = torch.randn(B, 128 * 128, device="cuda", generator=g)
        z0 = torch.randn(B, model.z_dim, device="cuda", generator=g)
        xg = x.clone().requires_grad_(True)

        def fwd_bwd(train, inp):
            def f():
                model.train(train)
                model(inp, noise=noise).backward()
            return f

        state = {}

        def enc_prepare():
            model.train()
            state["out"] = model.encode(x)

        def enc_bwd():
            if "out" not in state:
                enc_prepare()
            mu, u, d = state.pop("out")
            torch.autograd.backward([mu, u.squeeze(-1), d], seeds)

        def dec_prepare():
            model.train()
            state["xr"] = model.decode(z0.clone().requires_grad_(True))

        def dec_bwd():
            if "xr" not in state:
                dec_prepare()
            state.pop("xr").backward(seed_x)
        enc_bwd.prepare, dec_bwd.prepare = enc_prepare, dec_prepare
        cases = [("train_fwd_bwd", fwd_bwd(True, x)), ("eval_fwd_bwd", fwd_bwd(False, x)),
                 ("train_fwd_bwd_xgrad", fwd_bwd(True, xg)), ("encode_bwd", enc_bwd), ("decode_bwd", dec_bwd)]
        for name, fn in cases:
            med, lo, hi = timed(fn, args.iters, args.warmup)
            print(json.dumps({"batch": B, "case": name, "median_ms": round(med, 4), "min_ms": round(lo, 4),
                              "max_ms": round(hi, 4), "iters": args.iters, **dev}), flush=True)
        del model
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
