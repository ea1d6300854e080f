"""LatentUMAP stage times on the device: kNN, graph (memberships, fuzzy union, schedule), initialisation
(spectral layout, expansion, noise, rescale), SGD and the total, with CUDA events, on Gaussian blobs
with D = 32 and AVA's arguments (n_neighbors=20, min_dist=0.1, random_state=42).

Prints one JSON line per N (and appends them to --out when given): kNN pairs/s and their share of the
card's FP32 FMA peak (each pair costs D subtractions and D FMAs on the FMA pipe; the peak is
148 SMs x 128 lanes x the maximum SM clock read from nvidia-smi in the same run), SGD edge-epochs/s,
and, at N = 10^4, the trustworthiness (n_neighbors 20) of the embedding.

    python bench_umap.py [--sizes 10000,100000,1000000] [--out FILE]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
lu = importlib.import_module("autoencoded-vocal-analysis_b200.data.latent_umap")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", "0"], capture_output=True, text=True, check=True).stdout.strip().split(",")
    return q[0].strip(), float(q[1]), float(q[2])


def blobs(n, d, centers=10, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    c = torch.randn(centers, d, generator=g, device="cuda", dtype=torch.float64) * 10.0
    lab = torch.randint(0, centers, (n,), generator=g, device="cuda")
    return (c[lab] + torch.randn(n, d, generator=g, device="cuda", dtype=torch.float64)).contiguous(), lab


def run(n, d, name, watts, clk_mhz):
    x, lab = blobs(n, d)
    k, seed = 20, 42
    a, b = lu.find_ab_params(1.0, 0.1)
    n_epochs = lu.default_n_epochs(n)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    torch.cuda.synchronize()
    ev[0].record()
    idx, dist = lu.knn(x, k)
    ev[1].record()
    g = lu.fuzzy_graph(idx, dist)
    sched = lu.edge_schedule(g, n_epochs)
    ev[2].record()
    lay, _ = lu.spectral_layout(x, g, 2, seed)
    emb = lu.init_embedding(lay, seed, True, x.device)
    ev[3].record()
    for ep in range(n_epochs):
        lu.sgd_epoch(emb, sched, ep, a, b, 1.0, 1.0 - ep / float(n_epochs), seed)
    ev[4].record()
    torch.cuda.synchronize()
    t = [ev[i].elapsed_time(ev[i + 1]) / 1e3 for i in range(4)]
    pairs = float(n) * n
    peak_fma = 148 * 128 * clk_mhz * 1e6
    n_edges = sched["head"].numel()
    e = emb.cpu().numpy()
    out = {"what": "LatentUMAP stages, %d x %d float64 blobs, n_neighbors=20, min_dist=0.1" % (n, d),
           "gpu": name, "power_limit_W": watts, "max_sm_clock_MHz": clk_mhz, "N": n, "D": d,
           "knn_s": t[0], "graph_s": t[1], "init_s": t[2], "sgd_s": t[3], "total_s": sum(t),
           "knn_pairs_per_s": pairs / t[0], "knn_fp32_fma_pipe_share": pairs * 2 * d / t[0] / peak_fma,
           "n_epochs": n_epochs, "edges": n_edges, "sgd_edge_epochs_per_s": n_edges * n_epochs / t[3],
           "finite": bool(np.isfinite(e).all())}
    if n <= 10000:
        from sklearn.manifold import trustworthiness
        out["trustworthiness"] = float(trustworthiness(x.cpu().numpy(), e, n_neighbors=20))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="10000,100000,1000000")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_umap.py needs a CUDA device")
    name, watts, clk = card()
    run(2000, 32, name, watts, clk)   # warm-up: module load, allocator
    for n in [int(s) for s in args.sizes.split(",")]:
        line = json.dumps(run(n, 32, name, watts, clk))
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
