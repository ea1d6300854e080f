"""Synchronised BatchNorm for data-parallel training (csrc/bnsync.cu, VAE.enable_data_parallel(sync_bn=True)).

1. The exchange kernel on one GPU: W virtual ranks whose slots and flags are sub-ranges of one
   allocation, each rank's calls on a stream of its own.
2. The model step on one GPU with virtual ranks (every rank a VAE of its own on its own stream, wired
   to one exchange allocation): against the float64 oracle on the concatenated batch, against one
   model on that batch, and the exact sequence of exchanges a step issues.
3. The model on two GPUs with NCCL and symmetric memory (skipped with fewer than two devices):
   graphs, both optimizer paths, empty shards through train_step, and one train_epoch.
4. CPU: sync_bn on a gloo group raises.
"""
import ctypes
import importlib
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import vae_oracle
from tests.helpers import gpu_relu_masks, masked_oracle_grads, rel_err, relu_flips

PKG = "autoencoded-vocal-analysis_b200"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
vae_mod = importlib.import_module(PKG + ".models.vae")
SLOT = vae_mod._BN_SYNC_SLOT
MOMENTUM = 0.1


def _lib():
    return importlib.import_module(PKG + "._lib")


class _Virtual:
    """W virtual ranks on the current device: slots | flag of rank r = row r of one allocation."""

    def __init__(self, W):
        self.W = W
        self.buf = torch.zeros(W, 2 * SLOT + 2, dtype=torch.float64, device="cuda")
        self.peers = vae_mod._BnSyncPeers()
        for r in range(W):
            self.peers.slots[r] = self.buf[r].data_ptr()
            self.peers.flags[r] = self.buf[r].data_ptr() + 8 * 2 * SLOT
        self.local = torch.zeros(W, 2, dtype=torch.int32, device="cuda")
        self.streams = [torch.cuda.Stream() for _ in range(W)]
        for s in self.streams:
            s.wait_stream(torch.cuda.current_stream())

    def raw(self, r, sums, channels, count, running=None, rm_off=0, rv_off=32, nbt=None, world=None, peers=None,
            local=True):
        """The raw call (status code), on rank r's stream."""
        L = _lib().lib()
        with torch.cuda.stream(self.streams[r]):
            return L.ava_b200_bn_stats_exchange(
                ctypes.byref(peers if peers is not None else self.peers), r, self.W if world is None else world,
                None if sums is None else sums.data_ptr(), channels, count,
                None if running is None else running.data_ptr(), rm_off, rv_off,
                None if nbt is None else nbt.data_ptr(), MOMENTUM,
                self.local[r].data_ptr() if local else None, self.streams[r].cuda_stream)

    def call(self, r, *args, **kw):
        rc = self.raw(r, *args, **kw)
        assert rc == 0, _lib().last_error()

    def join(self):
        for s in self.streams:
            torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()


def _restate(ins, counts, channels):
    """Host restatement of the kernel's fp64 expression: rank-order sums, then * (count_r / count_g)."""
    idx = [t for t in range(64) if t % 32 < channels]
    tot = ins[0].copy()
    n = float(counts[0])
    for a, c in zip(ins[1:], counts[1:]):
        tot = tot + a
        n = n + float(c)
    outs = []
    for a, c in zip(ins, counts):
        o = a.copy()
        o[idx] = tot[idx] * (float(c) / n) if n > 0 else 0.0
        outs.append(o)
    return outs, tot, n


def _bits(a):
    return np.asarray(a).view(np.uint64 if np.asarray(a).dtype == np.float64 else np.uint32)


# ------------------------------------------------------------------------------ 1. kernel
@pytest.mark.gpu
@pytest.mark.parametrize("W", [2, 3, 8])
def test_exchange_bits_and_running_update(W):
    rng = np.random.default_rng(W)
    v = _Virtual(W)
    cases = [(32, False), (24, False), (8, False), (1, False), (16, True)]
    # unequal counts, one empty rank, two ranks with the same count; last, a global count of 1
    for ci, (channels, single) in enumerate(cases):
        counts = [int(c) for c in rng.integers(1, 5000, size=W)]
        counts[W - 1] = 0
        if W > 2:
            counts[1] = counts[0]
        if single:
            counts = [0] * W
            counts[W // 2] = 1
        l = ci % 14
        ins = [rng.standard_normal(64) * 1e3 for _ in range(W)]
        for a, c in zip(ins, counts):
            a[32:] = np.abs(a[32:]) * 1e3 + (a[:32] ** 2) / max(c, 1)      # plausible sums of squares
        sums = [torch.from_numpy(a).cuda() for a in ins]
        run0 = torch.from_numpy(rng.random(14 * 64).astype(np.float32) + 0.5).cuda()
        runs = [run0.clone() for _ in range(W)]
        nbts = [torch.zeros(14, dtype=torch.int64, device="cuda") for _ in range(W)]
        for s in v.streams:
            s.wait_stream(torch.cuda.current_stream())
        for r in range(W):
            v.call(r, sums[r], channels, counts[r], running=runs[r], rm_off=64 * l, rv_off=64 * l + 32,
                   nbt=nbts[r][l:])
        v.join()
        want, tot, n = _restate(ins, counts, channels)
        got = [s.cpu().numpy() for s in sums]
        for r in range(W):
            assert np.array_equal(_bits(got[r]), _bits(want[r])), (W, channels, r)
        if W > 2 and not single:      # equal shares, equal bits
            idx = [t for t in range(64) if t % 32 < channels]
            assert np.array_equal(_bits(got[0][idx]), _bits(got[1][idx]))
        # running buffers: what ava_b200_bn_update_running makes of the global sums and count
        ref = run0.clone()
        ref_nbt = torch.zeros(14, dtype=torch.int64, device="cuda")
        block = torch.zeros(14 * 64, dtype=torch.float64, device="cuda")
        block[64 * l:64 * l + 64] = torch.from_numpy(tot)
        h_counts = (ctypes.c_longlong * 14)(*[int(n) if k == l else 0 for k in range(14)])
        h_ch = (ctypes.c_int * 14)(*([channels] * 14))
        h_rm = (ctypes.c_int * 14)(*[64 * k for k in range(14)])
        h_rv = (ctypes.c_int * 14)(*[64 * k + 32 for k in range(14)])
        _lib().call("ava_b200_bn_update_running", block.data_ptr(), h_ch, h_counts, ref.data_ptr(), h_rm, h_rv,
                    ref_nbt.data_ptr(), MOMENTUM, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert not torch.equal(ref, run0)
        for r in range(W):
            assert np.array_equal(_bits(runs[r].cpu().numpy()), _bits(ref.cpu().numpy())), (W, channels, r)
            assert torch.equal(nbts[r], ref_nbt)
    assert int(v.local[:, 1].abs().sum()) == 0
    assert v.local[:, 0].tolist() == [len(cases)] * W


@pytest.mark.gpu
@pytest.mark.parametrize("W", [2, 3, 8])
def test_exchange_back_to_back_never_reads_a_stale_slot(W):
    """200 exchanges per rank issued without a host synchronisation: ranks run up to one exchange
    apart, every input changes every time, and each output must still be the restatement of its own
    exchange's inputs, bit for bit."""
    K, channels = 200, 32
    rng = np.random.default_rng(100 + W)
    ins = rng.standard_normal((K, W, 64))
    counts = rng.integers(0, 3, size=(K, W)) * rng.integers(1, 1000, size=(K, W))
    counts[:, 0] += 1
    io = torch.from_numpy(ins).cuda()
    v = _Virtual(W)
    for k in range(K):
        for r in (range(W) if k % 2 == 0 else range(W - 1, -1, -1)):
            v.call(r, io[k, r], channels, int(counts[k, r]))
    v.join()
    got = io.cpu().numpy()
    for k in range(K):
        want, _, _ = _restate(list(ins[k]), list(counts[k]), channels)
        for r in range(W):
            assert np.array_equal(_bits(got[k, r]), _bits(want[r])), (k, r)
    assert v.local[:, 0].tolist() == [K] * W and int(v.local[:, 1].abs().sum()) == 0


@pytest.mark.gpu
def test_exchange_rejects_bad_arguments_and_writes_nothing():
    W = 3
    v = _Virtual(W)
    sums = torch.randn(64, dtype=torch.float64, device="cuda")
    run = torch.rand(14 * 64, device="cuda")
    nbt = torch.zeros(14, dtype=torch.int64, device="cuda")
    missing = vae_mod._BnSyncPeers()
    for r in range(W):
        missing.slots[r], missing.flags[r] = v.peers.slots[r], v.peers.flags[r]
    missing.flags[2] = None
    keep = [t.clone() for t in (sums, run, nbt, v.buf, v.local)]
    launches = _lib().launch_count()
    bad = [dict(world=9), dict(world=0), dict(channels=0), dict(channels=33), dict(count=-1),
           dict(sums=None), dict(local=False), dict(peers=missing), dict(running=run, nbt=None),
           dict(running=run, nbt=nbt, rm_off=-1)]
    for kw in bad:
        a = dict(sums=sums, channels=32, count=10, running=None, nbt=None)
        a.update(kw)
        rc = v.raw(0, a.pop("sums"), a.pop("channels"), a.pop("count"), **a)
        assert rc != 0, kw
        assert "bn_stats_exchange" in _lib().last_error(), kw
    v.join()
    for a, b in zip(keep, (sums, run, nbt, v.buf, v.local)):
        assert torch.equal(a, b)
    assert _lib().launch_count() == launches


# --------------------------------------------------------- 2. model, virtual ranks on one GPU
class _Recorder:
    def __init__(self):
        self.calls = []

    def begin(self, name, args):
        if name == "ava_b200_bn_stats_exchange":
            self.calls.append((args[7] // 64, args[6] is not None, args[5]))

    def end(self, name, args):
        pass


STEP_SEQUENCE = [(l, True) for l in range(14)] + [(l, False) for l in range(13, 0, -1)]


def _virtual_step(models, v, xs, noises, sync, record=False):
    """One forward + backward on every virtual rank (no optimizer step); returns the ranks' buffers
    (None for an empty shard) and, with `record`, each rank's exchange calls."""
    lib = _lib()
    out, seqs = [], []
    for s in v.streams:
        s.wait_stream(torch.cuda.current_stream())
    for r, m in enumerate(models):
        rec = _Recorder() if record else None
        lib.PROFILER = rec
        try:
            with torch.cuda.stream(v.streams[r]):
                m._bn_sync_on = sync
                if xs[r].shape[0] > 0:
                    bufs = m._forward_native(xs[r], noises[r], True, want_grad_seed=True)
                    m._backward_native(bufs)
                else:
                    bufs = None
                    if sync:
                        m._bn_exchange_empty()
                m._bn_sync_on = False
        finally:
            lib.PROFILER = None
        out.append(bufs)
        seqs.append(rec.calls if record else None)
    v.join()
    return out, seqs


def _make_models(shards, P):
    W = len(shards)
    v = _Virtual(W)
    models = []
    for r in range(W):
        m = vae_mod.VAE(save_dir='', device_name='cuda', cuda_graphs=False)
        m.load_flat_state(P)
        m.train()
        m._dp_world, m._dp_rank = W, r
        m._bn_sync = {"peers": v.peers, "local": v.local[r],
                      "zeros": torch.zeros(2 * 14 * 64, dtype=torch.float64, device="cuda")}
        models.append(m)
    return models, v


def _shard_inputs(shards, seed):
    Bg = sum(shards)
    x = vae_oracle.make_input(seed, Bg)
    ew, ed = vae_oracle.make_noise(seed, Bg)          # noise fixed per row of the global batch
    xs, noises, o = [], [], 0
    for b in shards:
        xs.append(x[o:o + b].cuda())
        noises.append((ew[o:o + b].cuda(), ed[o:o + b].cuda()))
        o += b
    return x, ew, ed, xs, noises


@pytest.mark.gpu
@pytest.mark.parametrize("shards", [(64, 64), (5, 11), (7, 0)])
def test_virtual_ranks_step_equals_global_batch(shards):
    P = vae_oracle.make_params(3)
    W, Bg = len(shards), sum(shards)
    x, ew, ed, xs, noises = _shard_inputs(shards, 40 + Bg)
    models, v = _make_models(shards, P)
    # one local-statistics pass first: allocates every buffer, so that nothing on the host waits for
    # the device while a rank's exchange waits for the next rank's launches
    keep = [(m._flat_run.clone(), m._nbt.clone()) for m in models]
    local_bufs, _ = _virtual_step(models, v, xs, noises, sync=False)
    local_g = sum(m._flat_g.clone() for m, b in zip(models, local_bufs) if b is not None)
    local_masks = [gpu_relu_masks(b) for b in local_bufs if b is not None]
    for m, (run, nbt) in zip(models, keep):
        m._flat_run.copy_(run)
        m._nbt.copy_(nbt)
    bufs, seqs = _virtual_step(models, v, xs, noises, sync=True, record=True)
    # the exchange sequence of a step, on the empty-shard rank too
    for r, seq in enumerate(seqs):
        assert [(l, f) for l, f, _ in seq] == STEP_SEQUENCE, (r, seq)
        assert all(c == shards[r] * vae_mod._LAYERS[l][4] ** 2 for l, _, c in seq)
    g_sum = sum(m._flat_g.clone() for m, b in zip(models, bufs) if b is not None)
    full = [r for r, b in enumerate(bufs) if b is not None]
    loss = sum(float(bufs[r].loss[0]) for r in full) - (len(full) - 1) * models[0].loss_constant()

    # against the float64 oracle on the concatenated batch, ReLU pattern forced to the ranks' own
    def cat_masks(per_rank):
        return {k: torch.cat([mk[k] for mk in per_rank]) for k in per_rank[0]}
    masks = cat_masks([gpu_relu_masks(bufs[r]) for r in full])
    ref, grads, _, acts64, err32 = masked_oracle_grads(P, x, ew, ed, 10.0, masks)
    flips, flips32 = relu_flips(masks, acts64), err32.pop("__flips32__")
    assert abs(loss - float(ref["loss"])) <= 1e-4 * abs(float(ref["loss"])), (loss, float(ref["loss"]))
    assert flips <= max(16, 4 * flips32), (flips, flips32)
    m0 = models[0]
    worst = {}
    for k, off in m0._off.items():
        n = grads[k].numel()
        worst[k] = rel_err(g_sum[off:off + n].double().cpu().numpy().reshape(grads[k].shape), grads[k].numpy())
        assert worst[k] <= max(1e-4, 3 * err32[k]), (k, worst[k], err32[k])
    print("shards %s: worst gradient error %.1e (%s), %d flips (float32 oracle %d)"
          % (shards, max(worst.values()), max(worst, key=worst.get), flips, flips32))
    # the same shards with per-rank statistics miss that bar (an empty shard makes them the same)
    if 0 not in shards:
        lmasks = cat_masks(local_masks)
        _, lgrads, _, _, lerr32 = masked_oracle_grads(P, x, ew, ed, 10.0, lmasks)
        lerr32.pop("__flips32__")
        missed = [k for k, off in m0._off.items()
                  if rel_err(local_g[off:off + lgrads[k].numel()].double().cpu().numpy().reshape(lgrads[k].shape),
                             lgrads[k].numpy()) > max(1e-4, 3 * lerr32[k])]
        assert missed, "local BatchNorm statistics pass the global-batch bar: the test does not discriminate"

    # against one model on the concatenated batch: statistics blocks, running buffers, nbt
    one = vae_mod.VAE(save_dir='', device_name='cuda', cuda_graphs=False)
    one.load_flat_state(P)
    one.train()
    ob = one._forward_native(x.cuda(), (ew.cuda(), ed.cuda()), True, want_grad_seed=True)
    one._backward_native(ob)
    torch.cuda.synchronize()
    # After the exchange every rank holds the same global sums, scaled to its share.
    for name in ("stats", "dstats"):
        norm = [getattr(bufs[r], name).double().cpu().numpy() * (Bg / shards[r]) for r in full]
        for l in range(1 if name == "dstats" else 0, 14):       # layer 0's dstats stay local
            blk = [a[64 * l:64 * l + 64] for a in norm]
            for a in blk[1:]:
                e = np.abs(a - blk[0]).max() / max(np.abs(blk[0]).max(), 1e-300)
                assert e <= 1e-14, (shards, name, l, e)
    # Against one model on the whole batch.  Layer 0's statistics are sums over the same input rows:
    # they agree to the rounding of the in-CTA fp32 partials.  Every later block also sees the rank's
    # dense layers run at the rank's batch size, which can select another GEMM path than the whole
    # batch does (the tensor-core path needs a multiple of 128 rows): fp32-level differences.  For the
    # forward statistics those stay fp32-sized.  The backward sums (sum g, sum g*(x - mean)) cancel
    # heavily, so the same fp32 differences are large relative to their result; they are held to the
    # float64 oracle instead, through the BatchNorm affine gradients above (dbeta is the sum over ranks
    # of dstats[c], dgamma of invstd * dstats[32 + c]).
    worst = {"stats": 0.0, "dstats": 0.0}
    for r in full:
        scale = Bg / shards[r]
        for name, a, b in (("stats", bufs[r].stats, ob.stats), ("dstats", bufs[r].dstats, ob.dstats)):
            for l in range(1 if name == "dstats" else 0, 14):
                got = (a[64 * l:64 * l + 64] * scale).cpu().numpy()
                want = b[64 * l:64 * l + 64].cpu().numpy()
                e = np.abs(got - want).max() / max(np.abs(want).max(), 1e-300)
                worst[name] = max(worst[name], e)
                if name == "stats":
                    assert e <= (1e-7 if l == 0 else 1e-4), (shards, r, name, l, e)
    for _ in range(2):       # three steps in all: running buffers follow the single-GPU recursion
        _virtual_step(models, v, xs, noises, sync=True)
        ob = one._forward_native(x.cuda(), (ew.cuda(), ed.cuda()), True, want_grad_seed=True)
        one._backward_native(ob)
    torch.cuda.synchronize()
    for m in models[1:]:
        assert torch.equal(m._flat_run, models[0]._flat_run)
        assert torch.equal(m._nbt, models[0]._nbt)
    assert torch.equal(models[0]._nbt, one._nbt)
    d = ((models[0]._flat_run - one._flat_run).abs() / one._flat_run.abs().clamp(min=1.0)).max().item()
    print("shards %s: against one model: stats %.1e, dstats %.1e, running buffers %.1e after 3 steps"
          % (shards, worst["stats"], worst["dstats"], d))
    assert d <= 1e-6, d
    assert int(v.local[:, 1].abs().sum()) == 0


# ------------------------------------------------------------------------ 3. two GPUs, NCCL
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _two_gpu_worker(rank, world, port, tmp):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    sys.path.insert(0, ROOT)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    vm = importlib.import_module(PKG + ".models.vae")
    ds_mod = importlib.import_module(PKG + ".models.vae_dataset")
    P = vae_oracle.make_params(3)

    def model(graphs, fused, sync=True):
        m = vm.VAE(save_dir='', device_name='cuda', cuda_graphs=graphs)
        m.load_flat_state(P)
        m.enable_data_parallel(fused=fused, sync_bn=sync)
        m.train()
        assert (m._bn_sync is not None) == sync
        return m

    # (a) 6 steps: graphs on / off, fused / NCCL optimizer; every run ends where the eager NCCL run ends
    shards = (5, 11)
    runs = {}
    for key in ((False, False), (True, False), (False, True), (True, True)):
        m = model(*key)
        losses = []
        for step in range(6):
            x, ew, ed, xs, noises = _shard_inputs(shards, 60 + step)
            losses.append(float(m.train_step(xs[rank], noise=noises[rank])))
        if key[0]:
            assert m._graphs[shards[rank]]["graph"] is not None
        m.dp_check_status()
        torch.cuda.synchronize()
        mine, other = m._flat_p.clone(), m._flat_p.clone()
        dist.broadcast(other, src=0)
        assert torch.equal(mine, other), key
        run, other = m._flat_run.clone(), m._flat_run.clone()
        dist.broadcast(other, src=0)
        assert torch.equal(run, other), key
        runs[key] = (losses, mine)
    ref_loss, ref_p = runs[(False, False)]
    for key, (losses, p) in runs.items():
        for a, b in zip(losses, ref_loss):
            assert abs(a - b) <= 2e-4 * abs(b), (key, losses, ref_loss)
        assert (p - ref_p).abs().max().item() <= 6 * 2.5e-3, key
        assert (p - ref_p).abs().mean().item() <= 2e-6, key
    # (b) an empty shard through train_step: 3 steps against one GPU on the whole batch
    for fused in (False, True):
        m = model(False, fused)
        one = vm.VAE(save_dir='', device_name='cuda', cuda_graphs=False)
        one.load_flat_state(P)
        one.train()
        for step in range(3):
            x, ew, ed, xs, noises = _shard_inputs((7, 0), 80 + step)
            m.train_step(xs[rank], noise=noises[rank] if rank == 0 else None)
            one.train_step(x.cuda(), noise=(ew.cuda(), ed.cuda()))
        m.dp_check_status()
        torch.cuda.synchronize()
        assert torch.equal(m._nbt, one._nbt)
        assert (m._flat_run - one._flat_run).abs().max().item() <= 1e-6
        assert (m._flat_p - one._flat_p).abs().max().item() <= 3 * 2.5e-3
        assert (m._flat_p - one._flat_p).abs().mean().item() <= 2e-6
    # (c) one epoch over a seeded syllable set: world 2 + sync_bn == world 1 (noise fixed per syllable)
    N, Z = 40, 32
    files = [os.path.join(tmp, "sylls%d.npy" % i) for i in range(2)]
    if rank == 0:
        rng = np.random.default_rng(5)
        for i, fn in enumerate(files):
            a = rng.random((N // 2, 128, 128))
            a[:, 0, 0] = (np.arange(N // 2) + i * N // 2 + 0.5) / 64.0     # the syllable's id, exact in fp32
            np.save(fn, a)
    dist.barrier()
    gen = torch.Generator().manual_seed(9)
    table = torch.randn(N, 1 + Z, generator=gen)

    def fixed_noise(m):
        step = m.train_step

        def train_step(data, noise=None):
            idx = (data[:, 0, 0].float().cpu() * 64.0).long()
            t = table[idx].cuda()
            return step(data, noise=(t[:, :1].contiguous(), t[:, 1:].contiguous()) if len(idx) else None)
        m.train_step = train_step
        return m

    def epoch(m, r, w):
        loader = ds_mod.get_syllable_data_loaders({'train': files, 'test': []}, batch_size=12,
                                                  shuffle=(False, False), rank=r, world_size=w)['train']
        return m.train_epoch(loader)
    m = fixed_noise(model(False, True))
    got = epoch(m, rank, world)
    m.dp_check_status()
    if rank == 0:
        one = vm.VAE(save_dir='', device_name='cuda', cuda_graphs=False)
        one.load_flat_state(P)
        want = epoch(fixed_noise(one), 0, 1)
        torch.cuda.synchronize()
        assert abs(got - want) <= 1e-6 * abs(want), (got, want)
        assert (m._flat_p - one._flat_p).abs().max().item() <= 4 * 2.5e-3
        assert (m._flat_p - one._flat_p).abs().mean().item() <= 2e-6
        assert torch.equal(m._nbt, one._nbt)
        assert (m._flat_run - one._flat_run).abs().max().item() <= 1e-6
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_sync_bn_on_two_gpus(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    mp.spawn(_two_gpu_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)


# ----------------------------------------------------------------------------------- 4. CPU
def _gloo_worker(rank, world, port):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    vm = importlib.import_module(PKG + ".models.vae")
    m = vm.VAE(save_dir='', device_name='cpu')
    with pytest.raises(RuntimeError, match="synchronised BatchNorm needs CUDA ranks of one NCCL group"):
        m.enable_data_parallel(sync_bn=True)
    assert m._bn_sync is None and m._dp_world == 1        # nothing was set up
    m.enable_data_parallel()                              # the default still works on gloo
    assert m._bn_sync is None and m._dp_world == world
    dist.destroy_process_group()


def test_sync_bn_on_gloo_raises():
    mp.spawn(_gloo_worker, args=(2, _free_port()), nprocs=2, join=True)
