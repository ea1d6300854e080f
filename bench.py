#!/usr/bin/env python
"""
bench.py -- headline benchmark of the AVA VAE hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one full VAE train step (forward + ELBO + backward + Adam) on one batch of
synthetic 128x128 spectrograms, `--batch` per GPU (default 1024, the per-GPU batch of
BASELINE.json's configs[1]/[2]).  Prints ONE JSON line: `value` = whole-job samples/s with
inputs resident in HBM, `e2e` = the same through the public API with pinned host batches
(H2D inside the timed region and a D2H read of the loss every step), `roofline` for the
dominant entry point (CUDA-event timed per native call on the launching stream, in a second
identical K-step loop so that the event records do not slow the `value` loop), `cpu_baseline`
= the oracle's CPU train step timed on the host cores (rank 0, N=1 only).

`--dump-outputs DIR`: after the timed loop, rank 0 writes what the last timed step handed its
caller as DIR/<name>.npy (float32; see step_outputs).  Inputs, parameters and noise are seeded,
so two builds run with the same arguments can be compared output for output.

`--impl reference`: the CPU restatement of the reference train step (oracle/, torch CPU,
all host threads) on the same metric; under torchrun only rank 0 works.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
PKG = "autoencoded-vocal-analysis_b200"
METRIC = "vae_train_samples_per_sec"
UNIT = "samples/s"
DUMP_SAMPLE = 1 << 20     # positions kept of the 17.4 M-element parameter and gradient vectors

# (cin, cout, stride, h_in, transposed) for layers 0..13
LAYERS = [(1, 8, 1, 128, 0), (8, 8, 2, 128, 0), (8, 16, 1, 64, 0), (16, 16, 2, 64, 0),
          (16, 24, 1, 32, 0), (24, 24, 2, 32, 0), (24, 32, 1, 16, 0), (32, 24, 1, 16, 1),
          (24, 24, 2, 16, 1), (24, 16, 1, 32, 1), (16, 16, 2, 32, 1), (16, 8, 1, 64, 1),
          (8, 8, 2, 64, 1), (8, 1, 1, 128, 1)]


def layer_sizes(l):
    ci, co, s, h, tr = LAYERS[l]
    ho = h if s == 1 else (h * 2 if tr else h // 2)
    n_in, n_out = ci * h * h, co * ho * ho
    macs = 9 * ci * co * (ho * ho if not tr else h * h) if s == 2 else 9 * ci * co * h * h
    if s == 2 and not tr:
        macs = 9 * ci * co * ho * ho
    return n_in, n_out, macs


def algorithmic(key, args, B):
    """(bytes, flops) one launch of this native call must move / do (DESIGN.md,
    'Algorithmic bytes').  fp32 tensors; weights and statistics are negligible except
    for the dense layers."""
    name = key.split("[")[0]
    if name in ("ava_b200_bnconv_fwd", "ava_b200_bnconv_bwd_data", "ava_b200_bnconv_bwd_weight"):
        l = args[0]
        n_in, n_out, macs = layer_sizes(l)
        if name.endswith("fwd"):
            return 4.0 * B * (n_in + n_out), 2.0 * B * macs
        if name.endswith("bwd_data"):
            # reads dz (out-shaped) and x (in-shaped: BN backward + ReLU mask); writes the next dz
            return 4.0 * B * (n_out + 2 * n_in), 2.0 * B * macs
        return 4.0 * B * (n_out + n_in), 2.0 * B * macs   # reads dz, x
    if name == "ava_b200_linear_fwd":
        M, N, K, groups = args[6], args[7], args[8], args[10]
        return 4.0 * groups * (M * K + N * K + M * N), 2.0 * groups * M * N * K
    if name == "ava_b200_linear_bwd_data":
        M, N, K, groups = args[6], args[7], args[8], args[9]
        return 4.0 * groups * (2 * M * N + N * K + M * K), 2.0 * groups * M * N * K
    if name == "ava_b200_linear_bwd_weight":
        M, N, K, groups = args[7], args[8], args[9], args[10]
        return 4.0 * groups * (2 * M * N + M * K + N * K), 2.0 * groups * M * N * K
    if name in ("ava_b200_adam_step", "ava_b200_adam_step_dev"):
        n = args[4]
        return 4.0 * 7 * n, 12.0 * n
    if name == "ava_b200_recon":
        n = args[2]
        return 4.0 * 3 * n, 4.0 * n
    if name == "ava_b200_channel_stats":
        Bn, C, HW = args[1], args[2], args[3]
        return 4.0 * Bn * C * HW, 3.0 * Bn * C * HW
    if name == "ava_b200_dz_border_sums":
        Bn, C, H, W = args[1], args[2], args[3], args[4]
        return 4.0 * Bn * C * H * W, 2.0 * Bn * C * H * W
    if name == "ava_b200_bn_relu_bwd_apply":
        Bn, C, HW = args[5], args[6], args[7]
        return 4.0 * 3 * Bn * C * HW, 8.0 * Bn * C * HW
    return 0.0, 0.0


class EventProfiler:
    """Times every native call with a CUDA event pair on the launching stream."""

    def __init__(self, torch):
        self.torch = torch
        self.records = []   # (key, args, ev0, ev1)
        self._open = None

    def begin(self, name, args):
        key = name
        if name.startswith("ava_b200_bnconv"):
            key = "%s[%d]" % (name, args[0])
        elif name.startswith("ava_b200_linear_fwd"):
            key = "%s[%dx%dx%d]" % (name, args[6], args[7], args[8])
        elif name.startswith("ava_b200_linear_bwd_data"):
            key = "%s[%dx%dx%d]" % (name, args[6], args[7], args[8])
        elif name.startswith("ava_b200_linear_bwd_weight"):
            key = "%s[%dx%dx%d]" % (name, args[7], args[8], args[9])
        ev0 = self.torch.cuda.Event(enable_timing=True)
        ev0.record()
        self._open = (key, args, ev0)

    def end(self, name, args):
        key, a, ev0 = self._open
        ev1 = self.torch.cuda.Event(enable_timing=True)
        ev1.record()
        self.records.append((key, a, ev0, ev1))

    def summary(self, B, steps):
        agg = {}
        for key, args, e0, e1 in self.records:
            ms = e0.elapsed_time(e1)
            by, fl = algorithmic(key, args, B)
            d = agg.setdefault(key, {"ms": 0.0, "n": 0, "bytes": 0.0, "flops": 0.0})
            d["ms"] += ms
            d["n"] += 1
            d["bytes"] += by
            d["flops"] += fl
        return agg


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = False
        self.samples = []

    def _run_nvml(self):
        """Fast path: NVML through nvidia_ml_py (same counters as the nvidia-smi query below)."""
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        bits = {"hw_slowdown": pynvml.nvmlClocksEventReasonHwSlowdown,
                "hw_thermal_slowdown": pynvml.nvmlClocksEventReasonHwThermalSlowdown,
                "sw_thermal_slowdown": pynvml.nvmlClocksEventReasonSwThermalSlowdown,
                "sw_power_cap": pynvml.nvmlClocksEventReasonSwPowerCap}
        mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        while not self.stop_flag:
            sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
            self.samples.append([str(sm), str(mx)] + ["Active" if r & bits[n] else "Not Active" for n in
                                                     ("hw_slowdown", "hw_thermal_slowdown",
                                                      "sw_thermal_slowdown", "sw_power_cap")])
            time.sleep(0.01)

    def run(self):
        try:
            self._run_nvml()
            return
        except Exception:
            pass
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True,
                                     text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([f.strip() for f in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def result(self):
        sm = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = []
        for i, n in enumerate(names):
            if any(len(s) > 2 + i and s[2 + i].lower().startswith("active") for s in self.samples):
                reasons.append(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def cpu_train_samples_per_sec(batch, steps, warmup, seed=0, threads=None):
    """The oracle's restatement of the reference train step on the host CPU, on `threads`
    host threads (default: all cores -- torchrun exports OMP_NUM_THREADS=1, which is overridden
    here so that the figure is the box's, not one core's)."""
    import torch
    from oracle import vae_oracle
    torch.set_num_threads(threads if threads else (os.cpu_count() or 1))
    torch.manual_seed(seed)
    P = vae_oracle.make_params(seed)
    keys = [k for k, _ in vae_oracle.param_order()]
    st = {"step": 0, "m": {k: torch.zeros_like(P[k]) for k in keys},
          "v": {k: torch.zeros_like(P[k]) for k in keys}}
    x = torch.rand(batch, 128, 128)
    times = []
    for i in range(warmup + steps):
        ew, ed = torch.randn(batch, 1), torch.randn(batch, 32)
        t0 = time.perf_counter()
        vae_oracle.train_step_cpu(P, st, x, ew, ed)
        t1 = time.perf_counter()
        if i >= warmup:
            times.append(t1 - t0)
    total = sum(times)
    return batch * len(times) / total, 1e3 * total / len(times), torch.get_num_threads()


def step_outputs(model, loss):
    """What a train step hands its caller, as float32 host arrays: the loss it returns, the
    parameters its Adam update left, the gradient it computed (grad_dict) and the BatchNorm
    running statistics.  Parameters and gradients are concatenated in registration order (70 MB
    each) and cut to the same seeded sample of DUMP_SAMPLE positions."""
    import numpy as np
    import torch
    named = list(model.named_parameters())
    grads = model.grad_dict()
    params = torch.cat([p.detach().reshape(-1) for _, p in named])
    grad = torch.cat([grads[k].reshape(-1) for k, _ in named])
    idx = np.sort(np.random.default_rng(0).choice(params.numel(), DUMP_SAMPLE, replace=False))
    idx = torch.from_numpy(idx).to(params.device)
    running = torch.cat([b.reshape(-1) for _, b in model.named_buffers() if b.is_floating_point()])
    out = {"loss": loss.detach().reshape(1), "params_sample": params[idx], "grads_sample": grad[idx],
           "bn_running_stats": running}
    return {k: v.float().cpu().numpy() for k, v in out.items()}


def bind_to_gpu_numa_node(local_rank):
    """Multi-GPU runs: pin this rank's host threads (and so, by first touch, its pinned staging
    buffers) to the NUMA node its GPU hangs off -- 8 ranks x 64 MiB per step of host->device
    traffic otherwise cross the socket interconnect (round 1: e2e scaled 6.88x where the
    device-resident loop scaled 7.36x).  Returns a short description, or None if unavailable."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[local_rank]) if vis and vis.split(",")[local_rank].isdigit() else local_rank
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(idx)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.split(":", 1)
        path = "/sys/bus/pci/devices/%s:%s/numa_node" % (dom[-4:].lower(), rest.lower())
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return "rank threads bound to NUMA node %d (%d cpus) of GPU %s" % (node, len(cpus), bus)
    except Exception:      # noqa: BLE001  (no NVML / sysfs entry: leave the affinity alone)
        return None


def make_config(B, world, precision, graphs=None):
    return {"workload": "syllable VAE (z_dim=32) full train step (fwd+ELBO+bwd+Adam) on "
                        "128x128 synthetic specs, batch %d per GPU" % B,
            "batch_per_gpu": B, "global_batch": B * world, "precision": precision,
            "parallelism": "dp%d" % world, "cuda_graph": graphs,
            "l2": "per-step working set (%.1f GB activations + 0.49 GB optimizer "
                  "traffic) exceeds the 126 MB L2; two input batches alternate"
                  % (B * 2.42e-3 * 2)}


def run_reference(args, rank, world):
    """`--impl reference`: the reference's train step (its arithmetic restated in
    oracle/vae_oracle.py; the reference itself needs h5py/affinewarp/matplotlib at import and is
    not installable here) on the host CPU with all cores, on the SAME workload as our arm: one
    step = one optimizer step on a batch of `--batch` spectrograms.  If the box is too slow for
    K+W such steps to finish in ~4 minutes, the per-step batch is halved until they do and the
    line says so (`config.reference_sample_batch`); samples/s on the CPU is flat in the batch
    size, so the figure stays comparable."""
    if rank != 0:
        return
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    sample = args.batch
    budget_s = 240.0
    v1, ms1, cores = cpu_train_samples_per_sec(64, 1, 1)      # probe: one batch-64 step
    est = (ms1 * 1e-3) * (sample / 64.0) * (args.steps + args.warmup)
    while est > budget_s and sample > 64:
        sample //= 2
        est /= 2
    v, ms, cores = cpu_train_samples_per_sec(sample, args.steps, args.warmup)
    cfg = make_config(args.batch, max(world, 1), args.precision)
    cfg["reference_sample_batch"] = sample
    line = {
        "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
        "config": cfg,
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d timed train steps (after %d warm-up) of batch %d%s: the reference's "
                                   "arithmetic restated in oracle/vae_oracle.py, torch CPU, %d threads"
                                   % (args.steps, args.warmup, sample,
                                      "" if sample == args.batch else " (a sample of the %d-batch; the full "
                                      "batch would not finish in the time budget)" % args.batch, cores)},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def dp_check(model, vae_mod, dist, world, rank):
    """Numerical equivalence of the data-parallel step ON THE GPUS, before anything is timed
    (SURVEY section 4 test 9).  (a) every rank runs the same batch and noise: the all-reduced flat
    gradient must equal world x the local one.  (b) distinct shards: the all-reduced gradient and
    loss must equal what rank 0 gets by pushing every rank's shard through the model itself and
    summing (local-BatchNorm semantics: each rank == the reference on its shard; the loss is a
    batch SUM, so gradients add).  Parameters are untouched (no optimizer step); the BatchNorm
    running buffers are restored afterwards."""
    import torch
    Bc = 64
    keep_run, keep_nbt = model._flat_run.clone(), model._nbt.clone()
    gen = torch.Generator(device="cuda")
    res = {}

    def fwd_bwd(x, ew, ed, reduce):
        bufs = model._forward_native(x, (ew, ed), True, want_grad_seed=True)
        model._backward_native(bufs)
        if reduce:
            early, mid, late = model._grad_buckets()
            for w in model._allreduce(early + mid + late, async_op=True):
                w.wait()
        return bufs.loss.clone()

    def draw(seed):
        gen.manual_seed(seed)
        return (torch.rand(Bc, 128, 128, device="cuda", generator=gen),
                torch.randn(Bc, 1, device="cuda", generator=gen),
                torch.randn(Bc, 32, device="cuda", generator=gen))
    # (a) same batch everywhere
    x, ew, ed = draw(777)
    fwd_bwd(x, ew, ed, False)
    g_local = model._flat_g.clone()
    fwd_bwd(x, ew, ed, True)
    den = float(g_local.abs().max()) * world
    res["same_batch_max_rel_err"] = float((model._flat_g - world * g_local).abs().max()) / den
    # (b) distinct shards vs rank 0's own recomputation of every shard
    x, ew, ed = draw(1000 + rank)
    loss = fwd_bwd(x, ew, ed, True)
    g_dp = model._flat_g.clone()
    dist.all_reduce(loss, op=dist.ReduceOp.SUM)
    shards = [torch.empty_like(x) for _ in range(world)]
    dist.all_gather(shards, x)
    g_sum = torch.zeros_like(g_dp, dtype=torch.float64)
    loss_sum = 0.0
    for r in range(world):
        xr, ewr, edr = draw(1000 + r)
        assert torch.equal(xr, shards[r]), "dp_check: rank %d's shard differs from its seed" % r
        loss_sum += float(fwd_bwd(xr, ewr, edr, False))
        g_sum += model._flat_g.double()
    den = float(g_sum.abs().max())
    res["sharded_grad_max_rel_err"] = float((g_dp.double() - g_sum).abs().max()) / den
    res["sharded_loss_rel_err"] = abs(float(loss) - loss_sum) / abs(loss_sum)
    res["ok"] = bool(res["same_batch_max_rel_err"] < 1e-5 and res["sharded_grad_max_rel_err"] < 1e-5 and
                     res["sharded_loss_rel_err"] < 1e-6)
    res["what"] = ("batch %d per rank; (a) same batch on every rank: all-reduced gradient vs world x local; "
                   "(b) distinct shards: all-reduced gradient / loss vs this rank's recomputation of all %d "
                   "shards summed" % (Bc, world))
    model._flat_run.copy_(keep_run)
    model._nbt.copy_(keep_nbt)
    if getattr(model, "_dp_fused", None) is not None:
        # (c) the fused NVLink optimizer kernel (csrc/dp.cu) against bucketed NCCL all-reduce + Adam:
        # identical initial state, 3 steps on distinct shards, compare the parameters
        ends = []
        for fused in (True, False):
            torch.manual_seed(4321)
            mm = vae_mod.VAE(save_dir='', device_name='cuda', precision=model.precision, cuda_graphs=False)
            mm.enable_data_parallel(fused=fused)
            mm.train()
            for step in range(3):
                x, ew, ed = draw(2000 + 10 * step + rank)
                mm.train_step(x, noise=(ew, ed))
            mm.dp_check_status()
            torch.cuda.synchronize()
            ends.append(mm._flat_p.clone())
            del mm
        d = (ends[0] - ends[1]).abs()
        same = ends[0].clone()
        dist.broadcast(same, src=0)
        res["fused_vs_nccl_param_mean_abs"] = float(d.mean())
        res["fused_vs_nccl_param_max_abs"] = float(d.max())
        res["fused_replicas_identical"] = bool(torch.equal(same, ends[0]))
        # Adam's first steps are sign-like (|update| = lr = 1e-3 whatever the gradient's size): an
        # element whose gradient sum is ~0 can flip with the summation order, so the max is bounded
        # by steps x lr and the mean says how rare that is
        # (the NVSwitch's adder may round the sum differently in the last bit than NCCL's / a rank-order
        # sum: more near-zero gradients flip -- the multimem variant gets the wider bar; its data
        # path is pinned bit-exact against the peer-load variant in tests/test_gpu_dp.py)
        bar = 3e-5 if model._dp_fused["multimem"] else 2e-6
        res["ok"] = bool(res["ok"] and res["fused_replicas_identical"] and
                         res["fused_vs_nccl_param_mean_abs"] < bar and res["fused_vs_nccl_param_max_abs"] < 7e-3)
        res["what"] += "; (c) 3 steps of the fused NVLink reduce+Adam+broadcast kernel vs NCCL all-reduce + Adam"
    return res


FINCH_P = {  # examples/finch_window_mwe.py:29-49 (the shotgun VAE's preprocessing parameters)
    'fs': 32000, 'num_freq_bins': 128, 'num_time_bins': 128, 'nperseg': 512, 'noverlap': 256,
    'max_dur': 1e9, 'window_length': 0.12, 'min_freq': 400, 'max_freq': 10e3, 'spec_min_val': 2.0,
    'spec_max_val': 6.5, 'mel': True, 'time_stretch': False, 'within_syll_normalize': False,
}


def extra_get_latent(model, torch, dist, world, rank, n_total, B, peak):
    """BASELINE configs[4] / SURVEY 8(d) config 5: get_latent-style projection of `n_total`
    synthetic spectrograms sharded over the ranks in contiguous blocks, no collective on the data
    path.  Chunks are generated ON THE DEVICE inside the timed region (torch.rand, generator seeded
    per chunk: the corpus is never materialised -- 10 M specs would be 655 GB), encoded with
    eval-mode BatchNorm (stated; the reference's train-mode quirk F8 is covered by the parity
    tests), the latent means stay on the device and are downloaded once per rank, widened to
    float64 and gathered on rank 0's host as [n_total, 32]."""
    import numpy as np
    lo = (n_total * rank) // world
    hi = (n_total * (rank + 1)) // world
    n_mine = hi - lo
    model.eval()
    gen = torch.Generator(device="cuda")
    xbuf = torch.empty(B, 128, 128, device="cuda")
    lat = torch.empty(n_mine, model.z_dim, device="cuda")

    def run(n):
        done = 0
        with torch.no_grad():
            while done < n:
                b = min(B, n - done)
                gen.manual_seed(lo + done)
                xb = xbuf[:b]
                xb.uniform_(generator=gen)
                bufs = model._buffers_for(b)
                model._cur = bufs
                model._scratch_need = model._scratch_need_for(b)
                model._encode_native(xb, bufs, False)
                lat[done:done + b].copy_(bufs.heads[:, :model.z_dim])
                done += b
    run(min(n_mine, 4 * B))                        # warm-up
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run(n_mine)
    e1.record()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if world > 1:
        # results only: one gather of the fp32 latent means to rank 0 (blocks padded to equal size)
        n_max = (n_total + world - 1) // world
        pad = torch.zeros(n_max, model.z_dim, device="cuda")
        pad[:n_mine].copy_(lat)
        parts = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
        dist.gather(pad, parts, dst=0)
        host = None
        if rank == 0:
            sizes = [(n_total * (r + 1)) // world - (n_total * r) // world for r in range(world)]
            host = np.concatenate([p[:n].cpu().numpy() for p, n in zip(parts, sizes)]).astype(np.float64)
    else:
        host = lat.cpu().numpy().astype(np.float64)
    t_gather = time.perf_counter() - t0
    t = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    model.train()
    if rank != 0:
        return None
    assert host.shape == (n_total, model.z_dim) and np.isfinite(host).all()
    sps = n_total / (ms * 1e-3)
    return {"workload": "get_latent: %d synthetic specs generated on device in chunks of %d, sharded in "
                        "contiguous blocks over %d GPU(s), eval-mode BatchNorm, no collective on the data "
                        "path" % (n_total, B, world),
            "specs_per_s": sps, "device_ms": ms, "n_gpus": world,
            "hbm_frac_layer_granular": round(2.36e6 * sps / world / 1e9 / peak, 4),
            "algorithmic_bytes_per_spec": 2.36e6,
            "host_gather_s": round(t_gather, 3), "output": "float64 [%d, %d] on rank 0's host" % host.shape}


def extra_shotgun(model, torch, vae_mod, steps):
    """BASELINE configs[3] / SURVEY 8(d) config 4: synthetic corpus of 16 files x 600 s int16 audio
    @ 32 kHz, 2 ROIs per file, finch parameters; windows are sampled on the host with numpy's
    legacy RNG (bit-exact indices) and turned into 128x128 spectrograms by ONE launch of the GPU
    get_spec kernel per batch, feeding the train step.  "Training never waits" <=> the rate with
    on-the-fly windows equals the rate of the same step on a resident batch."""
    import numpy as np
    win_mod = importlib.import_module(PKG + ".models.window_vae_dataset")
    rng = np.random.default_rng(0)
    fs, n_files, dur = FINCH_P['fs'], 16, 600.0
    audio = [(3000 * rng.standard_normal(int(dur * fs), dtype=np.float32)).astype(np.int16)
             for _ in range(n_files)]
    rois = [np.array([[1.0, 250.0], [300.0, 598.0]]) for _ in range(n_files)]
    ds = win_mod.FixedWindowDataset(["f%02d.wav" % k for k in range(n_files)], None, dict(FINCH_P),
                                    audio=audio, fs=fs, rois=rois)
    out = {"workload": "shotgun VAE: random 0.12 s windows of 16 x 600 s synthetic int16 audio, finch "
                       "parameters, GPU get_spec on the fly"}

    def timed(fn, iters):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / iters
    for nb in (128, 1024):
        x = ds.sample_batch(nb)
        t_res = timed(lambda: model.train_step(x), steps)
        t_fly = timed(lambda: model.train_step(ds.sample_batch(nb)), steps)
        t_win = timed(lambda: ds.sample_batch(nb), steps)
        out["batch_%d" % nb] = {"train_samples_per_s_on_the_fly": nb / t_fly,
                                "train_samples_per_s_resident_batch": nb / t_res,
                                "ratio": t_res / t_fly, "windows_per_s_sampler_plus_get_spec": nb / t_win}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=1024, help="per-GPU batch")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="auto", choices=["auto", "fp32", "tf32x3", "tf32x3b", "tf32x3c", "tf32x3d", "tf32x3e", "tf32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--all-kernels", action="store_true", help="list every native call, not the top 12")
    ap.add_argument("--no-extra", action="store_true", help="skip the get_latent / shotgun blocks")
    ap.add_argument("--latent-specs", type=int, default=10_000_000,
                    help="corpus size of the get_latent block (BASELINE configs[4]: 10 M)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device"
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pkg = importlib.import_module(PKG)
    lib = importlib.import_module(PKG + "._lib")
    vae_mod = importlib.import_module(PKG + ".models.vae")

    B = args.batch
    torch.manual_seed(1234 + rank)
    # the public default (the whole step replayed as a CUDA graph when not data parallel) for the
    # `value` and `e2e` loops; eager launches for the per-call event profile
    model = vae_mod.VAE(save_dir='', device_name='cuda', precision=args.precision)
    dp = None
    if world > 1:
        model.enable_data_parallel()
        model.train()
        dp = dp_check(model, vae_mod, dist, world, rank)
        f = model._dp_fused
        dp_mode = ("bucketed NCCL all-reduce (3 buckets overlapped with the backward) + Adam on every rank"
                   if f is None else
                   "one fused kernel per rank over NVLink peer memory: reduce-scatter of the gradient (%s) + "
                   "Adam on the rank's 1/%d slice + parameter broadcast (%s); no NCCL on the step"
                   % (("multimem.ld_reduce in the NVSwitch", world, "multimem.st") if f["multimem"]
                      else ("peer loads", world, "peer stores")))
    model.train()
    # two resident synthetic batches (alternated) + pinned host copies for the e2e leg
    xs = [torch.rand(B, 128, 128, device="cuda") for _ in range(2)]
    xs_host = [x.cpu().pin_memory() for x in xs]

    align_t = torch.zeros(1, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def align():
        """After barrier(), right before a timed region starts: one more collective that is only
        ENQUEUED (no host sync), so the ranks' streams leave it at the same device time even when
        one host returns from the barrier milliseconds after the others (measured at N=2: the first
        timed step otherwise carried ~3 ms of exactly that skew)."""
        if world > 1:
            dist.all_reduce(align_t)

    # ---------------------------------------------------------------- device-resident
    # (the clock sampler starts before the warm-up: its NVML initialisation stays out of the timed region)
    sampler = ClockSampler(local_rank)
    sampler.start()
    for i in range(args.warmup):
        model.train_step(xs[i % 2])
    barrier()
    launches0 = lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    barrier()
    # the host-side barrier leaves the device idle for milliseconds and the first step after it ran
    # 0.2 ms (1 GPU) to 3.9 ms (8 GPUs) slow: two more untimed steps are enqueued behind the barrier so
    # that the timed region starts on a busy device, then the ranks' streams are aligned
    for i in range(2):
        model.train_step(xs[i % 2])
    align()
    ev0.record()
    for i in range(args.steps):
        loss = model.train_step(xs[i % 2])
        marks[i].record()        # per-step marks (diagnostic: `step_ms`); the value is ev0 -> ev1
    ev1.record()
    barrier()
    # taken before the loops below train the model further
    outputs = step_outputs(model, loss) if args.dump_outputs and rank == 0 else None
    per_step = [(ev0 if i == 0 else marks[i - 1]).elapsed_time(marks[i]) for i in range(args.steps)]
    launches = lib.launch_count() - launches0
    # the same K steps again with a CUDA-event pair around every native call (roofline /
    # kernel_families / kernels); the event records cost ~5 %, so `value` is taken from the
    # loop above and this loop's own time is reported as profiled_ms_per_step
    prof = None if args.no_profile else EventProfiler(torch)
    ms_prof = None
    if prof is not None:
        graphs_default = model.cuda_graphs
        model.cuda_graphs = False
        # per-call times are taken with every kernel alone on the device: the forked stream that
        # carries the dense weight / bias gradients beside the conv backward in the `value` and `e2e`
        # loops would lengthen whatever it overlaps (same kernels, same launch count)
        side_default = vae_mod._SIDE_STREAM
        vae_mod._SIDE_STREAM = False
        for i in range(2):
            model.train_step(xs[i % 2])
        launches_eager0 = lib.launch_count()
        lib.PROFILER = prof
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        align()
        p0.record()
        for i in range(args.steps):
            model.train_step(xs[i % 2])
        p1.record()
        barrier()
        lib.PROFILER = None
        model.cuda_graphs = graphs_default
        vae_mod._SIDE_STREAM = side_default
        ms_prof = p0.elapsed_time(p1) / args.steps
        if launches == 0:
            # the `value` loop replayed CUDA graphs (no host-side launch calls to count): the
            # graph holds exactly the kernels of an eager step, counted here over the same K steps
            launches = lib.launch_count() - launches_eager0
    if launches == 0:
        graphs_default = model.cuda_graphs
        model.cuda_graphs = False
        n0 = lib.launch_count()
        model.train_step(xs[0])
        launches = (lib.launch_count() - n0) * args.steps
        model.cuda_graphs = graphs_default
    ms_total = ev0.elapsed_time(ev1)
    t = torch.tensor([ms_total], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / args.steps
    value = world * B * args.steps / (ms_total * 1e-3)

    # ---------------------------------------------------------------- end to end
    # the public API a user script drives: pinned host batches, every batch copied host->device
    # inside the timed region (prefetch_to_device keeps the copy of batch i+1 in flight on a side
    # stream while step i runs, as VAE.train_epoch does) and loss.item() read back every step
    for xb in vae_mod.prefetch_to_device(xs_host):      # untimed warm-up of the same path
        float(model.train_step(xb).item())
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(2):          # (as above: a busy device behind the barrier)
        model.train_step(xs[i % 2])
    align()
    e0.record()
    host_batches = (xs_host[i % 2] for i in range(args.steps))
    # the reference reads loss.item() every step (vae.py:351).  Every step's loss is read here too
    # (4 bytes device->host per step, inside the timed region), but software-pipelined: the loss
    # of step i goes to a pinned slot with an event behind it and is read on the host while step
    # i+1 is already running, so the device never idles for a host round trip
    loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
    loss_ev = [torch.cuda.Event(), torch.cuda.Event()]
    losses_read = 0
    for i, xb in enumerate(vae_mod.prefetch_to_device(host_batches)):
        loss = model.train_step(xb)
        loss_host[i % 2:i % 2 + 1].copy_(loss.reshape(1), non_blocking=True)
        loss_ev[i % 2].record()
        if i > 0:
            loss_ev[(i - 1) % 2].synchronize()
            float(loss_host[(i - 1) % 2])
            losses_read += 1
    loss_ev[(args.steps - 1) % 2].synchronize()
    float(loss_host[(args.steps - 1) % 2])
    losses_read += 1
    assert losses_read == args.steps
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / (float(t.item()) * 1e-3)

    sampler.stop_flag = True      # sampled through both timed regions (device-resident and e2e)
    sampler.join(timeout=2)
    # ---------------------------------------------------------------- the other BASELINE configs
    extra = {}
    if world > 1:
        # where the multi-GPU step time goes: every rank runs the SAME step unsynchronised
        # (no data parallelism, all ranks at once) -- the slowest rank's free-running time is the
        # floor of the lock-stepped data-parallel step; the rest is the optimizer/collective kernel
        solo = vae_mod.VAE(save_dir='', device_name='cuda', precision=args.precision)
        solo.train()
        for i in range(4):
            solo.train_step(xs[i % 2])
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for i in range(args.steps):
            solo.train_step(xs[i % 2])
        s1.record()
        torch.cuda.synchronize()
        t = torch.tensor([s0.elapsed_time(s1) / args.steps], device="cuda")
        ts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(ts, t)
        extra["dp_diag"] = {"free_running_ms_per_step_by_rank": [round(float(v), 4) for v in ts],
                            "what": "the same step without data parallelism, all ranks running at once"}
        del solo
        if model._dp_fused is not None:
            # the fused optimizer/collective kernel on its own: 20 back-to-back calls, ranks in step
            model._flat_g.zero_()
            f = model._dp_fused
            variants = [("peer loads/stores", f["peers_p2p"])]
            if f["peers_mc"] is not None:
                variants.append(("multimem", f["peers_mc"]))
            keep = f["peers"]
            for name, peers in variants:
                f["peers"] = peers
                barrier()
                align()
                s0.record()
                for i in range(20):
                    model._adam_dp_native()
                s1.record()
                torch.cuda.synchronize()
                extra["dp_diag"]["adam_step_dp_us_back_to_back[%s]" % name] = round(1e3 * s0.elapsed_time(s1) / 20, 1)
            f["peers"] = keep
            model.dp_check_status()
    if not args.no_extra:
        # (secondary workloads never take the headline line down with them: a failure is reported)
        peak_x, _ = measured_peaks()
        try:
            lat_model = vae_mod.VAE(save_dir='', device_name='cuda', precision=args.precision)
            r = extra_get_latent(lat_model, torch, dist, world, rank, args.latent_specs, 1024, peak_x)
            if r is not None:
                extra["get_latent"] = r
            del lat_model
        except Exception as e:      # noqa: BLE001
            if world > 1:
                raise               # ranks must not diverge around a collective
            extra["get_latent"] = {"error": repr(e)}
        if world == 1:
            try:
                sg_model = vae_mod.VAE(save_dir='', device_name='cuda', precision=args.precision)
                sg_model.train()
                extra["shotgun"] = extra_shotgun(sg_model, torch, vae_mod, args.steps)
                del sg_model
            except Exception as e:  # noqa: BLE001
                extra["shotgun"] = {"error": repr(e)}
    if rank == 0:
        peak, peak_src = measured_peaks()
        roof, kernels, families = None, [], []
        if prof is not None:
            agg = prof.summary(B, args.steps)
            tot = sum(d["ms"] for d in agg.values())
            top = sorted(agg.items(), key=lambda kv: -kv[1]["ms"])
            for key, d in (top if args.all_kernels else top[:12]):
                gbs = d["bytes"] / (d["ms"] * 1e-3) / 1e9 if d["ms"] > 0 else 0.0
                tf = d["flops"] / (d["ms"] * 1e-3) / 1e12 if d["ms"] > 0 else 0.0
                kernels.append({"call": key.replace("ava_b200_", ""), "share": round(d["ms"] / tot, 4),
                                "us_per_launch": round(1e3 * d["ms"] / d["n"], 2),
                                "GBps": round(gbs, 1), "hbm_frac": round(gbs / peak, 4),
                                "fp32_TFLOPs": round(tf, 2)})
            # the dominant kernel = the native entry point (all its launches in the step, every
            # layer it serves) with the largest share of the step
            fam = {}
            for key, d in agg.items():
                f = fam.setdefault(key.split("[")[0], {"ms": 0.0, "n": 0, "bytes": 0.0, "flops": 0.0})
                for kk in ("ms", "n", "bytes", "flops"):
                    f[kk] += d[kk]
            ftop = sorted(fam.items(), key=lambda kv: -kv[1]["ms"])
            tpath = os.path.join(ROOT, "profiles", "r02_dram_traffic.json")
            tmap = {}
            if os.path.exists(tpath) and B == 1024:
                with open(tpath) as f:
                    tmap = json.load(f)
            for key, d in ftop[:8]:
                gbs = d["bytes"] / (d["ms"] * 1e-3) / 1e9
                families.append({"call": key.replace("ava_b200_", ""), "share": round(d["ms"] / tot, 4),
                                 "launches_per_step": d["n"] // args.steps,
                                 "us_per_step": round(1e3 * d["ms"] / args.steps, 1),
                                 "GBps": round(gbs, 1), "hbm_frac": round(gbs / peak, 4),
                                 "fp32_TFLOPs": round(d["flops"] / (d["ms"] * 1e-3) / 1e12, 2)})
            key, d = ftop[0]
            ach = d["bytes"] / (d["ms"] * 1e-3) / 1e9
            roof = {"kernel": key.replace("ava_b200_", ""), "bound": "hbm", "achieved": round(ach, 1),
                    "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": round(ach / peak, 4),
                    "traffic": tmap.get(key.replace("ava_b200_", "")),
                    "algorithmic_bytes_per_launch": d["bytes"] / d["n"],
                    "us_per_launch": round(1e3 * d["ms"] / d["n"], 2),
                    "launches_per_step": d["n"] // args.steps,
                    "fp32_TFLOPs": round(d["flops"] / (d["ms"] * 1e-3) / 1e12, 2),
                    "share_of_step": round(d["ms"] / tot, 4)}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            # SURVEY 8(d) config 1: batch 64, >= 3 warm-up and >= 10 timed steps on all host cores,
            # plus a 1-thread figure (about 15 s of CPU work in total)
            v, ms, cores = cpu_train_samples_per_sec(64, 10, 3)
            v1, _, _ = cpu_train_samples_per_sec(64, 3, 1, threads=1)
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "value_1_thread": v1,
                   "sample": "10 train steps of batch 64 after 3 warm-up (the reference's arithmetic "
                             "restated in oracle/vae_oracle.py, torch CPU, %d threads); value_1_thread: 3 "
                             "steps after 1 warm-up on one thread" % cores}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "profiled_ms_per_step": ms_prof,
            "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "dtype_note": "fp32 storage and accumulation everywhere; with precision auto/tf32x3 the "
                          "fc1/fc8 products (tcgen05) and the conv inner products of the layers with "
                          ">= 8 channels (mma.sync) are error-compensated 3xTF32 = fp32-level accuracy "
                          "(whole-model gradient parity equal to the fp32 FMA path); 'tf32' is the "
                          "opt-in reduced-precision mode (the reference's own GPU default)",
            "config": dict(make_config(B, world, args.precision, bool(model._graph_wanted(B))),
                           **({"dp_step": dp_mode, "host_numa": numa} if world > 1 else {})),
            "step_ms": {"median": round(sorted(per_step)[len(per_step) // 2], 4), "min": round(min(per_step), 4),
                        "max": round(max(per_step), 4), "argmax": per_step.index(max(per_step)),
                        "first": round(per_step[0], 4), "what": "rank 0's per-step device times inside the timed region"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * 128 * 128 * 4,
                    "d2h_bytes_per_step": 4},
            "gpu_launches": int(launches),
            "clocks": sampler.result(),
            "roofline": roof,
            "kernel_families": families,
            "kernels": kernels,
            "cpu_baseline": cpu,
            "dp_check": dp,
            "extra": extra,
        }
        if outputs is not None:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        print(json.dumps(line))
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
