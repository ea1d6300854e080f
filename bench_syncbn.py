#!/usr/bin/env python
"""
Cost of synchronised BatchNorm (VAE.enable_data_parallel(sync_bn=True)) in the data-parallel step.

  python bench_syncbn.py --gpus 8 --batch 64 1024      # one process per GPU (NCCL + symmetric memory)
  python bench_syncbn.py --gpus 1 --virtual 2 8         # exchange latency only, W virtual ranks on one GPU

With two or more GPUs, for each per-GPU batch: a local-BatchNorm model and a sync-BatchNorm model take
turns (`--rounds` rounds of `--steps` timed train steps each, after `--warmup` steps), so both see the
same machine state; then `--exchanges` back-to-back statistics exchanges on every rank give the latency
of one exchange.  Step and exchange times come from CUDA events.  With one GPU only the kernel itself can
be timed: W virtual ranks on W streams of one device (no NVLink in the path).  One JSON line per
configuration; the GPU name and power limit are read in the same run.
"""
import argparse
import ctypes
import importlib
import json
import os
import socket
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = "autoencoded-vocal-analysis_b200"


def _device_info():
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    except OSError:
        power = "unknown"
    return {"gpu": torch.cuda.get_device_name(), "power_limit": power}


def _median(v):
    v = sorted(v)
    return v[len(v) // 2]


def _time(fn, n):
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(n):
        fn()
    s1.record()
    s1.synchronize()
    return s0.elapsed_time(s1) / n


def _worker(rank, world, port, args):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    sys.path.insert(0, ROOT)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    vm = importlib.import_module(PKG + ".models.vae")
    torch.manual_seed(0)
    for B in args.batch:
        x = torch.rand(B, 128, 128, device="cuda")
        models = {}
        for mode in ("local", "sync"):
            m = vm.VAE(save_dir='', device_name='cuda')
            m.enable_data_parallel(sync_bn=mode == "sync")
            m.train()
            for _ in range(args.warmup):
                m.train_step(x)
            models[mode] = m
        times = {"local": [], "sync": []}
        for _ in range(args.rounds):
            for mode, m in models.items():
                torch.cuda.synchronize()
                dist.barrier()
                times[mode].append(_time(lambda: m.train_step(x), args.steps))
        m = models["sync"]
        block = torch.zeros(64, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        dist.barrier()
        ex_us = 1e3 * _time(lambda: m._bn_exchange(1, B, block, forward=False), args.exchanges)
        for mm in models.values():
            mm.dp_check_status()
        res = {"world": world, "batch_per_gpu": B,
               "step_ms_local": round(_median(times["local"]), 4), "step_ms_sync": round(_median(times["sync"]), 4),
               "step_ms_local_all": [round(t, 4) for t in times["local"]],
               "step_ms_sync_all": [round(t, 4) for t in times["sync"]],
               "exchange_us": round(ex_us, 2)}
        res["overhead"] = round(res["step_ms_sync"] / res["step_ms_local"] - 1, 4)
        out = [None] * world
        dist.all_gather_object(out, res)
        if rank == 0:
            res["exchange_us_per_rank"] = [o["exchange_us"] for o in out]
            res.update(_device_info())
            _emit(res, args)
    dist.destroy_process_group()


def _virtual(W, args):
    sys.path.insert(0, ROOT)
    vm = importlib.import_module(PKG + ".models.vae")
    lib = importlib.import_module(PKG + "._lib")
    L = lib.lib()
    buf = torch.zeros(W, 2 * vm._BN_SYNC_SLOT + 2, dtype=torch.float64, device="cuda")
    peers = vm._BnSyncPeers()
    for r in range(W):
        peers.slots[r] = buf[r].data_ptr()
        peers.flags[r] = buf[r].data_ptr() + 8 * 2 * vm._BN_SYNC_SLOT
    local = torch.zeros(W, 2, dtype=torch.int32, device="cuda")
    sums = torch.ones(W, 64, dtype=torch.float64, device="cuda")
    streams = [torch.cuda.Stream() for _ in range(W)]

    def round_():
        for r in range(W):
            rc = L.ava_b200_bn_stats_exchange(ctypes.byref(peers), r, W, sums[r].data_ptr(), 32, 1024, None, 0, 32,
                                              None, 0.1, local[r].data_ptr(), streams[r].cuda_stream)
            assert rc == 0, lib.last_error()
    for s in streams:
        s.wait_stream(torch.cuda.current_stream())
    for _ in range(100):
        round_()
    res = []
    for _ in range(args.rounds):
        e0 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in streams:
            s.wait_event(e0)
        for _ in range(args.exchanges):
            round_()
        for s in streams:
            torch.cuda.current_stream().wait_stream(s)
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        e1.synchronize()
        res.append(1e3 * e0.elapsed_time(e1) / args.exchanges)
    assert int(local[:, 1].abs().sum()) == 0
    out = {"virtual_world": W, "exchange_us": round(_median(res), 2), "exchange_us_all": [round(t, 2) for t in res]}
    out.update(_device_info())
    _emit(out, args)


def _emit(res, args):
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--gpus", type=int, default=torch.cuda.device_count())
    ap.add_argument("--batch", type=int, nargs="+", default=[64, 1024], help="samples per GPU")
    ap.add_argument("--virtual", type=int, nargs="+", default=[2, 8], help="virtual ranks (one-GPU mode)")
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--exchanges", type=int, default=2000)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_syncbn.py needs a CUDA device")
    if args.gpus >= 2:
        import torch.multiprocessing as mp
        s = socket.socket()
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
        s.close()
        mp.spawn(_worker, args=(args.gpus, port, args), nprocs=args.gpus, join=True)
    else:
        for W in args.virtual:
            _virtual(W, args)


if __name__ == "__main__":
    main()
