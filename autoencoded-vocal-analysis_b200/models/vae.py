"""
B200-native VAE for 128x128 spectrograms: drop-in for ``ava.models.vae``.

Mirrors the reference module surface (ava/models/vae.py:33-547): ``X_SHAPE``,
``X_DIM`` and ``class VAE`` with the same constructor arguments, attributes,
sub-module names (so checkpoints interchange) and methods ``encode``, ``decode``,
``forward``, ``train_epoch``, ``test_epoch``, ``train_loop``, ``save_state``,
``load_state``, ``visualize``, ``get_latent``.

Underneath, every tensor operation runs in hand-written sm_100a kernels reached
through the C ABI in include/ava_b200.h (ctypes, see _lib.py).  torch is used for
device memory, streams, RNG draws, the nn.Module/optimizer *containers* and
checkpoint (de)serialisation.  There is no CPU fallback: compute methods raise
if the model is not on a CUDA device or the native library is missing.

Additions over the reference API (keyword-only / new methods, defaults preserve
behaviour): ``precision=`` constructor argument, ``train_step``, ``compute_loss``,
``grad_dict``, ``load_flat_state``.  ``encode``, ``decode`` and ``forward`` are differentiable
as the reference's autograd graphs are, in train and eval mode, w.r.t. their input and the
parameters they touch (native backward kernels; no double backward).
"""
import ctypes
import math
import os
import warnings

import numpy as np
import torch
import torch.nn as nn
from torch.optim import Adam

from .. import _lib
from .._lib import call, ptr

X_SHAPE = (128, 128)
"""Processed spectrogram shape: ``[freq_bins, time_bins]``"""
X_DIM = int(np.prod(X_SHAPE))
"""Processed spectrogram dimension: ``freq_bins * time_bins``"""

# (name, in channels, out channels, stride, in height) -- ava/models/vae.py:128-134,155-161
_CONV = [("conv1", 1, 8, 1, 128), ("conv2", 8, 8, 2, 128), ("conv3", 8, 16, 1, 64),
         ("conv4", 16, 16, 2, 64), ("conv5", 16, 24, 1, 32), ("conv6", 24, 24, 2, 32),
         ("conv7", 24, 32, 1, 16)]
_CONVT = [("convt1", 32, 24, 1, 16), ("convt2", 24, 24, 2, 16), ("convt3", 24, 16, 1, 32),
          ("convt4", 16, 16, 2, 32), ("convt5", 16, 8, 1, 64), ("convt6", 8, 8, 2, 64),
          ("convt7", 8, 1, 1, 128)]
_LAYERS = _CONV + _CONVT           # layer id 0..13 of the C ABI
_BN_MOMENTUM = 0.1
# what precision='auto' means for the conv layers (ava_b200_set_conv_precision): 2 = 3xTF32;
# 3 / 5 / 6 / 4 = BF16 correction terms in the weight-gradient / + backward-data / + decoder-forward /
# + all forward kernels.  Measured at batch 1024 (gpurun_out s18-s25 -> profiles/r02_summary.md):
# worst gradient error vs float64 4.2e-5 / 4.4e-5 / 4.0e-5 / 7.2e-5 and 191 / 191 / 260 / 403 ReLU units on
# the other side of zero (the float32 reference itself: 129; bar: 4x that).  6 costs nothing in gradient
# accuracy; 4 ('tf32x3c') holds the 1e-4 bar with 1.4x margin and stays opt-in.
_AUTO_CONV_MODE = 6
_DP_MULTIMEM_MIN_WORLD = 4
_DP_MAX_WORLD = 8          # AVA_DP_MAX_WORLD, include/ava_b200.h


class _BiasJob(ctypes.Structure):
    """ava_b200_bias_job (include/ava_b200.h)."""
    _fields_ = [("dy", ctypes.c_void_p), ("mask", ctypes.c_void_p), ("db", ctypes.c_void_p),
                ("ld", ctypes.c_int), ("M", ctypes.c_int), ("N", ctypes.c_int)]


class _DpPeers(ctypes.Structure):
    """ava_b200_dp_peers (include/ava_b200.h): per-rank device pointers into symmetric memory."""
    _fields_ = [("grad", ctypes.c_void_p * _DP_MAX_WORLD), ("param", ctypes.c_void_p * _DP_MAX_WORLD),
                ("flags", ctypes.c_void_p * _DP_MAX_WORLD), ("grad_mc", ctypes.c_void_p),
                ("param_mc", ctypes.c_void_p)]


class _BnSyncPeers(ctypes.Structure):
    """ava_b200_bn_sync_peers (include/ava_b200.h): per-rank slot and flag pointers, symmetric memory."""
    _fields_ = [("slots", ctypes.c_void_p * _DP_MAX_WORLD), ("flags", ctypes.c_void_p * _DP_MAX_WORLD)]
_BN_SYNC_SLOT = 65         # AVA_BN_SYNC_SLOT, include/ava_b200.h

# The dense layers' weight and bias gradients are off the backward pass's critical path (only the
# data gradients feed the next layer): they are issued on a second stream that forks where their
# inputs are complete and joins before a gradient bucket is declared final / before the optimizer
# step, with a scratch buffer of its own.  Captured like everything else (a fork / join inside the
# CUDA graph).  AVA_B200_SIDE_STREAM=0: everything on one stream.
_SIDE_STREAM = os.environ.get("AVA_B200_SIDE_STREAM", "1") != "0"


def _out_hw(layer):
    _, _, _, s, h = _LAYERS[layer]
    if s == 1:
        return h
    return h // 2 if layer < 7 else h * 2


def _set_conv_precision(mode):
    """Process-wide conv arithmetic of the native library (0 fp32 FMA, 1 TF32, 2 3xTF32); the
    reference-side analogue is torch.backends.cudnn.allow_tf32.  A host-side switch, no launch."""
    if _lib.lib().ava_b200_set_conv_precision(mode) != 0:
        raise _lib.AvaB200Error(_lib.last_error())


def _stream():
    return torch.cuda.current_stream().cuda_stream


class _Buffers:
    """Activation / gradient workspace for one batch size (all torch-owned)."""

    def __init__(self, B, z_dim, device):
        f32 = dict(dtype=torch.float32, device=device)
        self.B = B
        self.act = []      # outputs of layers 0..13
        for l, (_, _, co, _, _) in enumerate(_LAYERS):
            hw = _out_hw(l)
            self.act.append(torch.empty(B, co, hw, hw, **f32))
        self.h1 = torch.empty(B, 1024, **f32)
        self.h2 = torch.empty(B, 256, **f32)
        self.h3 = torch.empty(B, 192, **f32)
        self.heads = torch.empty(B, 3 * z_dim, **f32)
        self.z = torch.empty(B, z_dim, **f32)
        self.d = torch.empty(B, z_dim, **f32)
        self.t5 = torch.empty(B, 64, **f32)
        self.t6 = torch.empty(B, 256, **f32)
        self.t7 = torch.empty(B, 1024, **f32)
        self.t8 = torch.empty(B, 8192, **f32)
        # fp64 accumulators: stats[14][64] | dstats[14][64] | acc[4] | tsums[14][288]
        self.accum = torch.zeros(2 * 14 * 64 + 4 + 14 * 288, dtype=torch.float64, device=device)
        self.stats = self.accum[:14 * 64]
        self.dstats = self.accum[14 * 64:2 * 14 * 64]
        self.acc = self.accum[2 * 14 * 64:2 * 14 * 64 + 4]
        self.tsums = self.accum[2 * 14 * 64 + 4:]
        self.loss = torch.zeros(1, **f32)
        # backward scratch (allocated lazily)
        self.g = None
        # eval-mode autograd: the running buffers the forward normalised with ([14][64] as
        # VAE._flat_run), which the backward must use even if a train-mode call moves the live ones;
        # None for train mode (batch statistics)
        self.run = None
        self._run_store = None

    def snapshot_running(self, flat_run, train):
        if train:
            self.run = None
            return
        if self._run_store is None:
            self._run_store = torch.empty_like(flat_run)
        self._run_store.copy_(flat_run)
        self.run = self._run_store

    def alloc_backward(self, z_dim):
        if self.g is not None:
            return
        B = self.B
        f32 = dict(dtype=torch.float32, device=self.h1.device)
        big = B * 8 * 128 * 128
        self.g = [torch.empty(big, **f32), torch.empty(big, **f32)]   # ping-pong
        self.dt8 = torch.empty(B, 8192, **f32)
        self.dt7 = torch.empty(B, 1024, **f32)
        self.dt6 = torch.empty(B, 256, **f32)
        self.dt5 = torch.empty(B, 64, **f32)
        self.gz = torch.empty(B, z_dim, **f32)
        self.gheads = torch.empty(B, 3 * z_dim, **f32)
        self.dh3 = torch.empty(B, 192, **f32)
        self.dh2 = torch.empty(B, 256, **f32)
        self.dh1 = torch.empty(B, 1024, **f32)
        self.da6 = torch.empty(B, 8192, **f32)


_PREFETCH_STATE = {}


def prefetch_to_device(batches, device=None, depth=1):
    """Iterate over host batches with the host->device copy of batch i+1 in flight on a side
    stream while batch i is being consumed (the reference copies synchronously inside the step,
    ava/models/vae.py:349).  Batches that are already on the device pass through.  Copies land
    in a small ring of preallocated device buffers (no allocator traffic in the loop); pageable
    CPU tensors are staged through pinned memory so that the copy is asynchronous."""
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    nslots = depth + 1
    # the side stream and the staging ring persist across calls (one set per device): epochs
    # after the first allocate nothing
    state = _PREFETCH_STATE.setdefault((device.index, nslots), {"stream": None, "ring": {}})
    if state["stream"] is None:
        state["stream"] = torch.cuda.Stream(device=device)
    copy_stream, ring = state["stream"], state["ring"]
    done = [None] * nslots          # consumer-finished events per slot
    copy_stream.wait_stream(torch.cuda.current_stream(device))   # earlier readers of the ring
    queue = []
    count = 0

    def enqueue(b):
        nonlocal count
        if not torch.is_tensor(b):
            b = torch.as_tensor(b)
        if b.is_cuda:
            queue.append((b, None, -1))
            return
        if b.dtype != torch.float32:
            b = b.float()
        if not b.is_pinned():
            b = b.pin_memory()
        slot = count % nslots
        count += 1
        bufs = ring.setdefault(tuple(b.shape), [None] * nslots)
        if bufs[slot] is None:
            bufs[slot] = torch.empty(b.shape, dtype=torch.float32, device=device)
        if done[slot] is not None:
            copy_stream.wait_event(done[slot])      # the step that read this slot has been issued
        with torch.cuda.stream(copy_stream):
            bufs[slot].copy_(b, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        queue.append((bufs[slot], ev, slot))

    def pop():
        d, ev, slot = queue.pop(0)
        if ev is not None:
            torch.cuda.current_stream(device).wait_event(ev)
        return d, slot

    def release(slot):
        if slot >= 0:
            done[slot] = torch.cuda.Event()
            done[slot].record(torch.cuda.current_stream(device))

    for b in batches:
        enqueue(b)
        if len(queue) > depth:
            d, slot = pop()
            yield d
            release(slot)
    while queue:
        d, slot = pop()
        yield d
        release(slot)


class VAE(nn.Module):
    """Variational Autoencoder class for single-channel images (B200-native).

    Attributes
    ----------
    save_dir, lr, z_dim, model_precision, device, optimizer, epoch, loss :
        as in the reference (ava/models/vae.py:43-122).
    precision : {'auto', 'fp32', 'tf32x3', 'tf32x3b', 'tf32x3d', 'tf32x3e', 'tf32x3c', 'tf32'}
        Arithmetic of the inner products (storage and accumulation are fp32 in every mode).
        'fp32': fp32 FMA everywhere.  'tf32x3': error-compensated 3xTF32 on the tensor cores
        (tcgen05 for fc1/fc8 at batch % 128 == 0, mma.sync for the conv layers with >= 8
        channels on both sides): fp32-level parity (rtol 1e-4 vs float64).  'tf32x3b' /
        'tf32x3d' / 'tf32x3e' / 'tf32x3c': as 'tf32x3' with the two correction terms of the conv
        products as half-rate BF16 instructions in the weight-gradient kernels / also the
        backward-data kernels / also the decoder's forward kernels / all three conv kernel
        families (include/ava_b200.h, ava_b200_set_conv_precision modes 3 / 5 / 6 / 4; all hold
        rtol 1e-4, with decreasing margin).  'tf32': single-pass TF32, the opt-in reduced-precision mode (stated
        tolerance 1e-2 forward).  'auto' (default): 'tf32x3' dense layers and 'tf32x3e' conv
        layers (mode 6, chosen by measurement: see _AUTO_CONV_MODE).
    """

    def __init__(self, save_dir='', lr=1e-3, z_dim=32, model_precision=10.0,
                 device_name="auto", *, precision='auto', cuda_graphs='auto'):
        super(VAE, self).__init__()
        self.save_dir = save_dir
        self.lr = lr
        self.z_dim = z_dim
        self.model_precision = model_precision
        assert device_name != "cuda" or torch.cuda.is_available()
        if device_name == "auto":
            device_name = "cuda" if torch.cuda.is_available() else "cpu"
        self.device = torch.device(device_name)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        assert precision in ('auto', 'fp32', 'tf32x3', 'tf32x3b', 'tf32x3c', 'tf32x3d', 'tf32x3e', 'tf32')
        self.precision = precision
        # dense layers: 0 fp32 FMA, 1 TF32, 2 3xTF32; conv layers additionally 3 / 4 = 3-term product
        # with the two correction terms as half-rate BF16 instructions (csrc/conv.cu, cv_pack_bf16)
        # in the weight-gradient kernels / in all three kernel families
        self._tc = {'auto': 2, 'fp32': 0, 'tf32x3': 2, 'tf32x3b': 2, 'tf32x3c': 2, 'tf32x3d': 2, 'tf32x3e': 2, 'tf32': 1}[precision]
        self._tc_conv = {'auto': _AUTO_CONV_MODE, 'tf32x3b': 3, 'tf32x3c': 4, 'tf32x3d': 5, 'tf32x3e': 6}.get(precision, self._tc)
        # CUDA graphs for the train step: 'auto' = when the step is host-bound (batch <= 256)
        assert cuda_graphs in ('auto', True, False)
        self.cuda_graphs = cuda_graphs
        if self.save_dir != '' and not os.path.exists(self.save_dir):
            os.makedirs(self.save_dir)
        self._flat_ready = False
        self._build_network()
        self.optimizer = Adam(self.parameters(), lr=self.lr)
        self.epoch = 0
        self.loss = {'train': {}, 'test': {}}
        self._bufs = {}
        self._grad_pool = {}       # free activation sets of the autograd paths, see _grad_buffers
        self._scratch = None
        self._step_host = 0
        self._graphs = {}
        self._dp_group = None
        self._dp_world = 1
        self._bn_sync = None       # synchronised BatchNorm state (enable_data_parallel(sync_bn=True))
        self._bn_sync_on = False   # set by train_step only: the exchanges run inside a training step
        self.to(self.device)

    # ------------------------------------------------------------------ network
    def _build_network(self):
        """Define all the network layers (containers only; ava/models/vae.py:125-168)."""
        z = self.z_dim
        for name, ci, co, s, _ in _CONV:
            setattr(self, name, nn.Conv2d(ci, co, 3, s, padding=1))
        for i, (_, ci, _, _, _) in enumerate(_CONV):
            setattr(self, "bn%d" % (i + 1), nn.BatchNorm2d(ci))
        self.fc1 = nn.Linear(8192, 1024)
        self.fc2 = nn.Linear(1024, 256)
        self.fc31 = nn.Linear(256, 64)
        self.fc32 = nn.Linear(256, 64)
        self.fc33 = nn.Linear(256, 64)
        self.fc41 = nn.Linear(64, z)
        self.fc42 = nn.Linear(64, z)
        self.fc43 = nn.Linear(64, z)
        self.fc5 = nn.Linear(z, 64)
        self.fc6 = nn.Linear(64, 256)
        self.fc7 = nn.Linear(256, 1024)
        self.fc8 = nn.Linear(1024, 8192)
        for name, ci, co, s, _ in _CONVT:
            if s == 1:
                setattr(self, name, nn.ConvTranspose2d(ci, co, 3, 1, padding=1))
            else:
                setattr(self, name, nn.ConvTranspose2d(ci, co, 3, 2, padding=1,
                                                       output_padding=1))
        for i, (_, ci, _, _, _) in enumerate(_CONVT):
            setattr(self, "bn%d" % (i + 8), nn.BatchNorm2d(ci))

    def _get_layers(self):
        """Return a dictionary mapping names to network layers (vae.py:171-186)."""
        names = ['fc1', 'fc2', 'fc31', 'fc32', 'fc33', 'fc41', 'fc42', 'fc43', 'fc5',
                 'fc6', 'fc7', 'fc8'] + ['bn%d' % i for i in range(1, 15)] + \
                ['conv%d' % i for i in range(1, 8)] + ['convt%d' % i for i in range(1, 8)]
        return {n: getattr(self, n) for n in names}

    # --------------------------------------------------------- flat storage
    def _memory_order(self):
        """Order of tensors inside the flat parameter buffer.  Independent of the
        registration order (which fixes the optimizer's positional state_dict);
        the three posterior heads are made contiguous so they run as one GEMM."""
        names = []
        for n, *_ in _CONV:
            names += [n + ".weight", n + ".bias"]
        names += ["fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias"]
        names += ["fc31.weight", "fc32.weight", "fc33.weight", "fc31.bias", "fc32.bias",
                  "fc33.bias", "fc41.weight", "fc42.weight", "fc43.weight", "fc41.bias",
                  "fc42.bias", "fc43.bias"]
        for n in ("fc5", "fc6", "fc7", "fc8"):
            names += [n + ".weight", n + ".bias"]
        for n, *_ in _CONVT:
            names += [n + ".weight", n + ".bias"]
        for i in range(1, 15):
            names += ["bn%d.weight" % i, "bn%d.bias" % i]
        return names

    def _flatten(self):
        """(Re)build the flat parameter / gradient / Adam-moment / BN-buffer storage
        on the module's current device and re-point every nn.Parameter and buffer
        to a view of it."""
        params = dict(self.named_parameters())
        dev = next(iter(params.values())).device
        order = self._memory_order()
        assert sorted(order) == sorted(params.keys())
        off, self._off = 0, {}
        for k in order:
            self._off[k] = off
            n = params[k].numel()
            # 16-byte aligned tensors; the z-dependent head blocks stay contiguous
            off += n if k.startswith(("fc3", "fc4")) else (n + 3) // 4 * 4
        self._n_flat = (off + 3) // 4 * 4
        f32 = dict(dtype=torch.float32, device=dev)
        old_m = getattr(self, "_flat_m", None)
        old_views_m = getattr(self, "_views_m", None)
        flat_p = torch.zeros(self._n_flat, **f32)
        flat_g = torch.zeros(self._n_flat, **f32)
        flat_m = torch.zeros(self._n_flat, **f32)
        flat_v = torch.zeros(self._n_flat, **f32)
        if old_m is not None and old_m.numel() == self._n_flat:
            flat_m.copy_(old_m)
            flat_v.copy_(self._flat_v)
        self._views_g, self._views_m, self._views_v = {}, {}, {}
        for k in order:
            p = params[k]
            o, n = self._off[k], p.numel()
            flat_p[o:o + n].copy_(p.detach().reshape(-1).to(torch.float32))
            p.data = flat_p[o:o + n].view(p.shape)
            self._views_g[k] = flat_g[o:o + n].view(p.shape)
            self._views_m[k] = flat_m[o:o + n].view(p.shape)
            self._views_v[k] = flat_v[o:o + n].view(p.shape)
            p.grad = None
        self._flat_p, self._flat_g, self._flat_m, self._flat_v = flat_p, flat_g, flat_m, flat_v
        self._dp_fused = None      # (a re-flatten leaves the symmetric-memory buffers of the fused DP path)
        # optimizer state that aliased the previous flat moment buffers follows them (model.to(),
        # .cuda(), .float() after training); the step count is kept, not re-adopted
        opt = getattr(self, "optimizer", None)
        if opt is not None and old_m is not None and old_m.numel() == self._n_flat:
            for k in order:
                st = opt.state.get(params[k])
                if st is not None and 'exp_avg' in st and old_views_m is not None and \
                        st['exp_avg'].data_ptr() == old_views_m[k].data_ptr():
                    st['exp_avg'], st['exp_avg_sq'] = self._views_m[k], self._views_v[k]
        # BN running buffers: [rm_1 | rv_1 | rm_2 | rv_2 ...], 32 floats each
        run = torch.zeros(14 * 64, **f32)
        nbt = torch.zeros(14, dtype=torch.int64, device=dev)
        self._bn_channels = []
        for i in range(14):
            bn = getattr(self, "bn%d" % (i + 1))
            c = bn.num_features
            self._bn_channels.append(c)
            run[i * 64:i * 64 + c].copy_(bn.running_mean)
            run[i * 64 + 32:i * 64 + 32 + c].copy_(bn.running_var)
            nbt[i] = int(bn.num_batches_tracked)
            bn._buffers['running_mean'] = run[i * 64:i * 64 + c]
            bn._buffers['running_var'] = run[i * 64 + 32:i * 64 + 32 + c]
            bn._buffers['num_batches_tracked'] = nbt[i]
        self._flat_run, self._nbt = run, nbt
        self._step_dev = torch.full((1,), float(self._step_host), **f32)
        self._hyper_dev = torch.zeros(4, dtype=torch.float64, device=dev)
        self._hyper_host = None
        self._loss_sum = torch.zeros(1, dtype=torch.float64, device=dev)
        self._bufs, self._scratch, self._graphs = {}, None, {}
        self._grad_pool = {}
        # host-side tables for the two BN bookkeeping kernels
        self._h_channels = (ctypes.c_int * 14)(*self._bn_channels)
        self._h_rm_off = (ctypes.c_int * 14)(*[i * 64 for i in range(14)])
        self._h_rv_off = (ctypes.c_int * 14)(*[i * 64 + 32 for i in range(14)])
        self._h_dg_off = (ctypes.c_int * 14)(*[self._off["bn%d.weight" % (i + 1)] for i in range(14)])
        self._h_db_off = (ctypes.c_int * 14)(*[self._off["bn%d.bias" % (i + 1)] for i in range(14)])
        self._flat_ready = True

    def _apply(self, fn, *args, **kwargs):
        # .to()/.cuda()/.float() re-allocate every tensor separately: re-flatten.
        out = super(VAE, self)._apply(fn, *args, **kwargs)
        if getattr(self, "_flat_ready", None) is not None and hasattr(self, "fc8"):
            self._flatten()
            try:
                self.device = self._flat_p.device
            except AttributeError:
                pass
            # the forked stream and its scratch belong to the device the model was on
            self._side_stream, self._scratch_side, self._side_dirty = None, None, False
        return out

    def _p(self, key):
        o = self._off[key]
        return self._flat_p.data_ptr() + 4 * o

    def _g(self, key):
        o = self._off[key]
        return self._flat_g.data_ptr() + 4 * o

    def _rm(self, bn_index):   # bn_index 0..13
        return self._flat_run.data_ptr() + 4 * (bn_index * 64)

    def _rv(self, bn_index):
        return self._flat_run.data_ptr() + 4 * (bn_index * 64 + 32)

    def _require_cuda(self):
        if self._flat_p.device.type != "cuda":
            raise RuntimeError(
                "ava_b200 VAE: compute requires a CUDA device (model is on %s); there is "
                "no CPU fallback" % self._flat_p.device)
        _lib.lib()

    _MAX_BATCH_SIZES = 4

    def _buffers_for(self, B):
        """Activation workspace for batch size B.  The least recently used sizes are dropped
        beyond _MAX_BATCH_SIZES (a default train_loop sees four: the regular batch, the ragged
        train and test tails and visualize's 5).  A captured CUDA graph holds raw pointers into
        its workspace, so a graph never outlives it: evicting a size drops its graph too."""
        b = self._bufs.pop(B, None)
        if b is None:
            while len(self._bufs) >= self._MAX_BATCH_SIZES:
                old = next(iter(self._bufs))
                self._bufs.pop(old)
                self._graphs.pop(old, None)
            b = _Buffers(B, self.z_dim, self._flat_p.device)
        self._bufs[B] = b          # most recently used last
        return b

    def _grad_buffers(self, B):
        """Activation workspace for a call that records an autograd graph.  The graph owns it until
        its backward has run or it is freed (_Lease): such sets never come from the _buffers_for cache,
        so neither a later call nor a captured train_step graph writes into them.  Sets come back to a
        small per-size free list, so a forward/backward loop allocates nothing after warm-up."""
        free = self._grad_pool.get(B)
        if free:
            return free.pop()
        return _Buffers(B, self.z_dim, self._flat_p.device)

    def _release_grad_buffers(self, bufs):
        if bufs.h1.device != self._flat_p.device:
            return                 # (the model moved while the graph was alive)
        free = self._grad_pool.pop(bufs.B, [])
        if len(free) < 2:
            free.append(bufs)
        self._grad_pool[bufs.B] = free         # most recently used last
        while len(self._grad_pool) > self._MAX_BATCH_SIZES:
            self._grad_pool.pop(next(iter(self._grad_pool)))

    def _side_fork(self):
        """The second stream, waiting for everything issued so far on the current one."""
        side = getattr(self, "_side_stream", None)
        if side is None:
            side = self._side_stream = torch.cuda.Stream(device=self._flat_p.device)
        side.wait_stream(torch.cuda.current_stream())
        self._side_dirty = True
        return side

    def _side_join(self):
        """The current stream waits for the work issued on the second one."""
        if getattr(self, "_side_dirty", False):
            torch.cuda.current_stream().wait_stream(self._side_stream)
            self._side_dirty = False

    def _ws_side(self, nbytes):
        ws = getattr(self, "_scratch_side", None)
        if ws is None or ws.numel() < nbytes:
            if ws is not None:
                self._graphs = {}
            ws = self._scratch_side = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8,
                                                  device=self._flat_p.device)
        return ws

    def _ws(self, nbytes):
        if self._scratch is None or self._scratch.numel() < nbytes:
            if self._scratch is not None:
                # captured graphs point into the old scratch buffer: they go with it
                self._graphs = {}
            self._scratch = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8,
                                        device=self._flat_p.device)
        return self._scratch

    def _scratch_bytes(self, B):
        L = _lib.lib()
        need = 0
        for l in range(14):
            need = max(need, L.ava_b200_bnconv_bwd_weight_ws(l, B))
        for (n, k) in [(1024, 8192), (256, 1024), (192, 256), (self.z_dim, 64), (64, self.z_dim),
                       (256, 64), (1024, 256), (8192, 1024)]:
            need = max(need, L.ava_b200_linear_ws_bytes(B, n, k))
        need = max(need, 64 * 4 * (8192 + 1024 + 256 + 64))      # ava_b200_bias_grads, decoder segment
        return int(need)

    # ------------------------------------------------------------- native passes
    def _linear(self, x, ldx, wkey, bkey, y, ldy, M, N, K, act, groups=1, x_gs=0, w_gs=0,
                b_gs=0, y_gs=0, tc=0):
        ws = self._ws(self._scratch_need)
        call("ava_b200_linear_fwd", ptr(x), ldx, self._p(wkey), self._p(bkey), ptr(y), ldy, M, N,
             K, act, groups, x_gs, w_gs, b_gs, y_gs, tc, ptr(ws), ws.numel(), _stream())

    def _linear_bwd(self, dy, lddy, ymask, x, ldx, wkey, bkey, dx, lddx, M, N, K, groups=1,
                    dy_gs=0, x_gs=0, w_gs=0, b_gs=0, dx_gs=0, tc=0, bias_jobs=None):
        """dW, db into the flat gradient buffer; dx (if not None) = (dy*mask) W.  With `bias_jobs`
        the bias gradient is not computed here but queued for one batched ava_b200_bias_grads call
        per backward segment (_flush_bias; the groups of a grouped layer are adjacent column blocks
        of dy and adjacent biases, i.e. one job)."""
        ws = self._ws(self._scratch_need)
        s = _stream()
        gb = self._g(bkey)
        if bias_jobs is not None:
            assert groups == 1 or (dy_gs == N and b_gs == N)
            bias_jobs.append((ptr(dy), ptr(ymask), gb, lddy, M, N * groups))
            gb = None
        if _SIDE_STREAM and gb is None:
            side = self._side_fork()
            ws2 = self._ws_side(self._scratch_need)
            with torch.cuda.stream(side):
                call("ava_b200_linear_bwd_weight", ptr(dy), lddy, ptr(ymask), ptr(x), ldx, self._g(wkey),
                     None, M, N, K, groups, dy_gs, x_gs, w_gs, b_gs, tc, ptr(ws2), ws2.numel(), _stream())
        else:
            call("ava_b200_linear_bwd_weight", ptr(dy), lddy, ptr(ymask), ptr(x), ldx, self._g(wkey),
                 gb, M, N, K, groups, dy_gs, x_gs, w_gs, b_gs, tc, ptr(ws), ws.numel(), s)
        if dx is not None:
            call("ava_b200_linear_bwd_data", ptr(dy), lddy, ptr(ymask), self._p(wkey), ptr(dx), lddx,
                 M, N, K, groups, dy_gs, w_gs, dx_gs, 0, tc, ptr(ws), ws.numel(), s)

    def _flush_bias(self, jobs):
        """All queued bias gradients of a backward segment in two launches."""
        arr = (_BiasJob * len(jobs))()
        for a, (dy, mask, db, ld, M, N) in zip(arr, jobs):
            a.dy, a.mask, a.db, a.ld, a.M, a.N = dy, mask, db, ld, M, N
        if _SIDE_STREAM:
            side = self._side_fork()
            ws2 = self._ws_side(self._scratch_need)
            with torch.cuda.stream(side):
                call("ava_b200_bias_grads", arr, len(jobs), ptr(ws2), ws2.numel(), _stream())
            return
        ws = self._ws(self._scratch_need)
        call("ava_b200_bias_grads", arr, len(jobs), ptr(ws), ws.numel(), _stream())

    def _conv_fwd(self, l, B, x, y, bufs, train, want_stats_out):
        name = _LAYERS[l][0]
        st = bufs.stats.data_ptr()
        _set_conv_precision(self._tc_conv)
        call("ava_b200_bnconv_fwd", l, B, ptr(x), ptr(y), self._p(name + ".weight"),
             self._p(name + ".bias"), self._p("bn%d.weight" % (l + 1)), self._p("bn%d.bias" % (l + 1)),
             st + 8 * 64 * l, self._rm(l), self._rv(l), 1 if train else 0,
             (st + 8 * 64 * (l + 1)) if want_stats_out else None, _stream())

    def _encode_native(self, x, bufs, train):
        """x [B,128,128] -> bufs.heads (mu | u | log d).  ava/models/vae.py:216-232."""
        B, Z, s = bufs.B, self.z_dim, _stream()
        if train:
            call("ava_b200_channel_stats", ptr(x), B, 1, X_DIM, bufs.stats.data_ptr(), s)
        h = x
        for l in range(7):
            if train and self._bn_sync_on:
                self._bn_exchange(l, B, bufs.stats, forward=True)
            self._conv_fwd(l, B, h, bufs.act[l], bufs, train, train and l < 6)
            h = bufs.act[l]
        tc = self._tc
        self._linear(h, 8192, "fc1.weight", "fc1.bias", bufs.h1, 1024, B, 1024, 8192, 1, tc=tc)
        self._linear(bufs.h1, 1024, "fc2.weight", "fc2.bias", bufs.h2, 256, B, 256, 1024, 1, tc=tc)
        # fc31|fc32|fc33 share their input: one [192,256] layer
        self._linear(bufs.h2, 256, "fc31.weight", "fc31.bias", bufs.h3, 192, B, 192, 256, 1)
        # fc41|fc42|fc43: three [Z,64] layers on the three 64-wide slices (strided batch)
        self._linear(bufs.h3, 192, "fc41.weight", "fc41.bias", bufs.heads, 3 * Z, B, Z, 64, 0,
                     groups=3, x_gs=64, w_gs=Z * 64, b_gs=Z, y_gs=Z)

    def _decode_native(self, z, bufs, train):
        """z [B,Z] -> bufs.act[13] = x_rec [B,1,128,128].  ava/models/vae.py:258-270."""
        B, Z, s = bufs.B, self.z_dim, _stream()
        tc = self._tc
        self._linear(z, Z, "fc5.weight", "fc5.bias", bufs.t5, 64, B, 64, Z, 1)
        self._linear(bufs.t5, 64, "fc6.weight", "fc6.bias", bufs.t6, 256, B, 256, 64, 1)
        self._linear(bufs.t6, 256, "fc7.weight", "fc7.bias", bufs.t7, 1024, B, 1024, 256, 1, tc=tc)
        self._linear(bufs.t7, 1024, "fc8.weight", "fc8.bias", bufs.t8, 8192, B, 8192, 1024, 1, tc=tc)
        if train:
            call("ava_b200_channel_stats", ptr(bufs.t8), B, 32, 256,
                 bufs.stats.data_ptr() + 8 * 64 * 7, s)
        h = bufs.t8
        for l in range(7, 14):
            if train and self._bn_sync_on:
                self._bn_exchange(l, B, bufs.stats, forward=True)
            self._conv_fwd(l, B, h, bufs.act[l], bufs, train, train and l < 13)
            h = bufs.act[l]

    def _update_running(self, B, first, last):
        """BN running buffers of layers first..last-1 (train-mode side effect)."""
        counts = [0] * 14
        for l in range(first, last):
            h = _LAYERS[l][4]
            counts[l] = B * h * h
        h_counts = (ctypes.c_longlong * 14)(*counts)
        call("ava_b200_bn_update_running", self._cur.stats.data_ptr(), self._h_channels, h_counts,
             ptr(self._flat_run), self._h_rm_off, self._h_rv_off, ptr(self._nbt), _BN_MOMENTUM, _stream())

    def _draw_noise(self, B):
        # Same draw order as LowRankMultivariateNormal.rsample: eps_W [B,1] then eps_D [B,Z].
        dev = self._flat_p.device
        ew = torch.randn(B, 1, dtype=torch.float32, device=dev)
        ed = torch.randn(B, self.z_dim, dtype=torch.float32, device=dev)
        return ew, ed

    def _forward_native(self, x, noise, train, want_grad_seed, bufs=None):
        """Full forward pass; returns the _Buffers holding every intermediate (`bufs`, or the
        cached set of this batch size).  Loss (fp32) lands in bufs.loss; if want_grad_seed,
        dL/dx_rec in bufs.g[0]."""
        self._require_cuda()
        x = self._as_input(x)
        B = x.shape[0]
        if bufs is None:
            bufs = self._buffers_for(B)
        self._cur = bufs
        self._scratch_need = self._scratch_need_for(B)
        s = _stream()
        bufs.accum.zero_()
        self._encode_native(x, bufs, train)
        ew, ed = noise if noise is not None else self._draw_noise(B)
        ew = ew.to(torch.float32).contiguous()
        ed = ed.to(torch.float32).contiguous()
        bufs.eps_w, bufs.eps_d = ew, ed
        call("ava_b200_latent_fwd", ptr(bufs.heads), ptr(ew), ptr(ed), B, self.z_dim, ptr(bufs.z),
             ptr(bufs.d), bufs.acc.data_ptr(), s)
        self._decode_native(bufs.z, bufs, train)
        g = None
        if want_grad_seed:
            bufs.alloc_backward(self.z_dim)
            g = bufs.g[0]
        # (the gradient written here is convt7's dz: its nine border sums are accumulated on the way)
        ts13 = (bufs.tsums.data_ptr() + 8 * 288 * 13) if g is not None else None
        call("ava_b200_recon", ptr(x), ptr(bufs.act[13]), B * X_DIM, float(self.model_precision),
             ptr(g), bufs.acc.data_ptr(), ts13, X_SHAPE[0], X_SHAPE[1], s)
        call("ava_b200_elbo_finalize", bufs.acc.data_ptr(), self.z_dim, X_DIM,
             float(self.model_precision), ptr(bufs.loss), ptr(self._loss_sum), s)
        if train and not self._bn_sync_on:      # (synchronised BatchNorm: done by the exchanges)
            self._update_running(B, 0, 14)
        bufs.x = x
        return bufs

    def _scratch_need_for(self, B):
        cache = getattr(self, "_scratch_cache", None)
        if cache is None:
            cache = self._scratch_cache = {}
        if B not in cache:
            cache[B] = self._scratch_bytes(B)
        return cache[B]

    def _conv_bwd(self, l, bufs, dz, x, dz_prev, relu_mask=1):
        """Backward of fused layer l given dz = the gradient w.r.t. its pre-activation output,
        whose nine border sums the kernel that wrote dz has already accumulated into tsums[l].
        (1) weight / bias gradients into the flat gradient buffer AND this layer's
        BatchNorm-backward reductions dstats[l] (both from the same centred raw product, see
        include/ava_b200.h); (2) the data gradient, pushed through this layer's BatchNorm backward
        and the previous layer's ReLU in the kernel's epilogue, lands in dz_prev as the previous
        layer's dz -- the gradient w.r.t. the BatchNorm output never goes to memory.
        bufs.run set: eval-mode BatchNorm with those running buffers.  relu_mask=0: no ReLU factor
        (layer 0's data gradient is the gradient w.r.t. the input spectrogram)."""
        B = bufs.B
        name = _LAYERS[l][0]
        st, ds, ts = bufs.stats.data_ptr(), bufs.dstats.data_ptr(), bufs.tsums.data_ptr()
        s = _stream()
        gamma, beta = self._p("bn%d.weight" % (l + 1)), self._p("bn%d.bias" % (l + 1))
        train, rm, rv = 1, None, None
        if bufs.run is not None:
            train, rm = 0, bufs.run.data_ptr() + 4 * 64 * l
            rv = rm + 4 * 32
        ws = self._ws(self._scratch_need)
        _set_conv_precision(self._tc_conv)
        call("ava_b200_bnconv_bwd_weight_ex", l, B, ptr(dz), ptr(x), self._p(name + ".weight"), gamma, beta,
             st + 8 * 64 * l, rm, rv, train, ts + 8 * 288 * l, self._g(name + ".weight"),
             self._g(name + ".bias"), ds + 8 * 64 * l, ptr(ws), s)
        if dz_prev is not None:
            if self._bn_sync_on:
                self._bn_exchange(l, B, bufs.dstats, forward=False)
            # the epilogue also accumulates the border sums of the dz it writes (layer l-1's; layer
            # 7 writes fc8's output gradient and layer 0 the input's, which need none)
            call("ava_b200_bnconv_bwd_data_ex", l, B, ptr(dz), self._p(name + ".weight"), ptr(x), gamma,
                 st + 8 * 64 * l, rv, train, ds + 8 * 64 * l, relu_mask, ptr(dz_prev),
                 (ts + 8 * 288 * (l - 1)) if l not in (0, 7) else None, s)

    def _bwd_decoder(self, bufs):
        """Backward segment 1: decoder conv stack (layers 13..7) and fc8..fc5.  Afterwards the
        gradients of fc5..fc8 and convt1..7 are final."""
        B, Z = bufs.B, self.z_dim
        bufs.alloc_backward(Z)
        g_cur, g_nxt = bufs.g[0], bufs.g[1]      # g[0] holds dL/dx_rec = convt7's dz (recon kernel)
        # layer 7 writes the gradient w.r.t. fc8's pre-activation output (bn8 backward + fc8's
        # ReLU) straight into dt8
        for l in range(13, 6, -1):
            xin = bufs.act[l - 1] if l > 7 else bufs.t8
            out = g_nxt if l > 7 else bufs.dt8
            self._conv_bwd(l, bufs, g_cur, xin, out)
            g_cur, g_nxt = g_nxt, g_cur
        jobs = []
        self._linear_bwd(bufs.dt8, 8192, None, bufs.t7, 1024, "fc8.weight", "fc8.bias", bufs.dt7, 1024,
                         B, 8192, 1024, tc=self._tc, bias_jobs=jobs)
        self._linear_bwd(bufs.dt7, 1024, bufs.t7, bufs.t6, 256, "fc7.weight", "fc7.bias", bufs.dt6, 256,
                         B, 1024, 256, tc=self._tc, bias_jobs=jobs)
        self._linear_bwd(bufs.dt6, 256, bufs.t6, bufs.t5, 64, "fc6.weight", "fc6.bias", bufs.dt5, 64,
                         B, 256, 64, bias_jobs=jobs)
        self._linear_bwd(bufs.dt5, 64, bufs.t5, bufs.z, Z, "fc5.weight", "fc5.bias", bufs.gz, Z,
                         B, 64, Z, bias_jobs=jobs)
        self._flush_bias(jobs)

    def _bwd_dense_encoder(self, bufs, latent=True):
        """Backward segment 2: latent (analytic gradients of sample + prior + entropy) and the
        encoder's dense layers.  Afterwards the gradients of fc1..fc43 are final (fc1.weight is
        half of all parameters).  latent=False: bufs.gheads already holds the heads' gradient
        (encode's backward)."""
        B, Z, s = bufs.B, self.z_dim, _stream()
        if latent:
            call("ava_b200_latent_bwd", ptr(bufs.heads), ptr(bufs.eps_w), ptr(bufs.eps_d), ptr(bufs.z),
                 ptr(bufs.gz), B, Z, ptr(bufs.gheads), s)
        jobs = []
        self._linear_bwd(bufs.gheads, 3 * Z, None, bufs.h3, 192, "fc41.weight", "fc41.bias", bufs.dh3, 192,
                         B, Z, 64, groups=3, dy_gs=Z, x_gs=64, w_gs=Z * 64, b_gs=Z, dx_gs=64, bias_jobs=jobs)
        self._linear_bwd(bufs.dh3, 192, bufs.h3, bufs.h2, 256, "fc31.weight", "fc31.bias", bufs.dh2, 256,
                         B, 192, 256, bias_jobs=jobs)
        self._linear_bwd(bufs.dh2, 256, bufs.h2, bufs.h1, 1024, "fc2.weight", "fc2.bias", bufs.dh1, 1024,
                         B, 256, 1024, tc=self._tc, bias_jobs=jobs)
        self._linear_bwd(bufs.dh1, 1024, bufs.h1, bufs.act[6], 8192, "fc1.weight", "fc1.bias",
                         bufs.da6, 8192, B, 1024, 8192, tc=self._tc, bias_jobs=jobs)
        self._flush_bias(jobs)

    def _bwd_conv_encoder(self, bufs, dx=None, n_bn=14):
        """Backward segment 3: encoder conv stack (layers 6..0) and the BatchNorm affine
        parameter gradients of layers 0..n_bn-1.  dx (optional): the gradient w.r.t. the input
        spectrogram, layer 0's data gradient."""
        B, s = bufs.B, _stream()
        # conv7's ReLU on the gradient arriving from fc1 (no BatchNorm at this seam)
        # (and the nine border sums of the dz it writes, conv7's)
        call("ava_b200_bn_relu_bwd_apply", ptr(bufs.da6), ptr(bufs.act[6]), None, None, None, B, 32, 256,
             1, ptr(bufs.da6), bufs.tsums.data_ptr() + 8 * 288 * 6, 16, s)
        g_cur = bufs.da6
        free = [bufs.g[0], bufs.g[1]]
        for l in range(6, -1, -1):          # (layer 0's data gradient only for dx)
            xin = bufs.act[l - 1] if l > 0 else bufs.x
            out = free[0] if l > 0 else dx
            self._conv_bwd(l, bufs, g_cur, xin, out, relu_mask=1 if l > 0 else 0)
            g_cur, free = out, [free[1], free[0]]
        self._bn_param_grads(bufs, 0, n_bn)

    def _bn_param_grads(self, bufs, first, last):
        """BatchNorm affine parameter gradients of layers first..last-1 from their dstats (one launch;
        eval mode with the running buffers in bufs.run)."""
        counts = [bufs.B * _LAYERS[l][4] ** 2 if first <= l < last else 0 for l in range(14)]
        h_counts = (ctypes.c_longlong * 14)(*counts)
        call("ava_b200_bn_param_grads_ex", bufs.stats.data_ptr(), bufs.dstats.data_ptr(), self._h_channels,
             h_counts, ptr(self._flat_g), self._h_dg_off, self._h_db_off, ptr(bufs.run), self._h_rv_off,
             1 if bufs.run is None else 0, _stream())

    def _backward_native(self, bufs, after_decoder=None, after_dense=None, dx=None):
        """Backward of the whole loss; leaves every parameter gradient in the flat
        gradient buffer (overwritten, not accumulated).  Replaces loss.backward(),
        ava/models/vae.py:352.  The two callbacks fire where a gradient bucket becomes final.
        dx (optional): the encoder's part of the input gradient, see _bwd_conv_encoder."""
        self._bwd_decoder(bufs)
        if after_decoder is not None:
            self._side_join()
            after_decoder()
        self._bwd_dense_encoder(bufs)
        if after_dense is not None:
            self._side_join()
            after_dense()
        self._bwd_conv_encoder(bufs, dx=dx)
        self._side_join()

    def _sync_hyper(self):
        """lr / betas / eps as torch.optim.Adam holds them (optimizer.param_groups[0]: what
        load_state restores from a checkpoint, ava/models/vae.py:470, and what LR schedulers
        change), mirrored into a device buffer the Adam kernel reads -- so a captured CUDA graph
        of the step follows them too."""
        grp = self.optimizer.param_groups[0]
        if grp.get('weight_decay', 0) != 0 or grp.get('amsgrad', False) or grp.get('maximize', False):
            raise NotImplementedError("ava_b200: Adam with weight_decay/amsgrad/maximize is not implemented")
        hyper = (float(grp['lr']), float(grp['betas'][0]), float(grp['betas'][1]), float(grp['eps']))
        if hyper != self._hyper_host:
            self._hyper_dev.copy_(torch.tensor(hyper, dtype=torch.float64))
            self._hyper_host = hyper

    def _adam_native(self):
        call("ava_b200_adam_step_dev", ptr(self._flat_p), ptr(self._flat_g), ptr(self._flat_m),
             ptr(self._flat_v), self._n_flat, ptr(self._step_dev), ptr(self._hyper_dev), 1.0, _stream())
        self._step_host += 1

    def _as_input(self, x):
        if not torch.is_tensor(x):
            x = torch.as_tensor(x)
        x = x.to(device=self._flat_p.device, dtype=torch.float32, non_blocking=True)
        if x.dim() != 3 or tuple(x.shape[1:]) != X_SHAPE:
            raise ValueError("expected input of shape [batch,128,128], got %s" % (tuple(x.shape),))
        return x.contiguous()

    # ------------------------------------------------------------------ public API
    def _grad_wanted(self, x, params):
        return torch.is_grad_enabled() and (
            (torch.is_tensor(x) and x.requires_grad) or any(p.requires_grad for p in params))

    def _params_of(self, part):
        """The parameters a call touches: 'encoder' (conv1-7, bn1-7, fc1-fc43), 'decoder' (fc5-8,
        convt1-7, bn8-14) or 'all', in registration order."""
        def is_enc(name):
            layer = name.split(".")[0]
            if layer.startswith("bn"):
                return int(layer[2:]) <= 7
            return (layer.startswith("conv") and not layer.startswith("convt")) or \
                layer in ("fc1", "fc2", "fc31", "fc32", "fc33", "fc41", "fc42", "fc43")
        return [(n, p) for n, p in self.named_parameters()
                if part == "all" or is_enc(n) == (part == "encoder")]

    def encode(self, x):
        """Compute q(z|x) = N(mu, u u^T + diag(d)).  ava/models/vae.py:189-233.

        Returns mu [B,z], u [B,z,1], d [B,z].  BatchNorm follows ``self.training``
        exactly as in the reference (batch statistics + running-buffer update in
        train mode).  Differentiable, in train and eval mode, w.r.t. `x` and the encoder's
        parameters (conv1-7, bn1-7, fc1, fc2, fc31-33, fc41-43) when grad mode is on and one of
        them requires grad; the backward is native (_EncodeFn)."""
        enc = self._params_of("encoder")
        if self._grad_wanted(x, [p for _, p in enc]):
            return _EncodeFn.apply(self, x, [n for n, _ in enc], *[p for _, p in enc])
        self._require_cuda()
        x = self._as_input(x)
        B, Z = x.shape[0], self.z_dim
        bufs = self._buffers_for(B)
        self._cur = bufs
        self._scratch_need = self._scratch_need_for(B)
        if self.training:
            bufs.accum.zero_()
        self._encode_native(x, bufs, self.training)
        if self.training:
            self._update_running(B, 0, 7)
        # d = exp(fc43(.)): same layer once more with the exp epilogue
        self._linear(bufs.h3[:, 128:], 192, "fc43.weight", "fc43.bias", bufs.d, Z, B, Z, 64, 2)
        heads = bufs.heads
        mu = heads[:, :Z].clone()
        u = heads[:, Z:2 * Z].clone().unsqueeze(-1)
        return mu, u, bufs.d.clone()

    def decode(self, z):
        """Compute the mean of p(x|z).  ava/models/vae.py:236-270.  Returns [B,16384].
        Differentiable, in train and eval mode, w.r.t. `z` and the decoder's parameters (fc5-8,
        convt1-7, bn8-14) when grad mode is on and one of them requires grad (_DecodeFn)."""
        dec = self._params_of("decoder")
        if self._grad_wanted(z, [p for _, p in dec]):
            return _DecodeFn.apply(self, z, [n for n, _ in dec], *[p for _, p in dec])
        self._require_cuda()
        z = z.to(device=self._flat_p.device, dtype=torch.float32).contiguous()
        B = z.shape[0]
        bufs = self._buffers_for(B)
        self._cur = bufs
        self._scratch_need = self._scratch_need_for(B)
        if self.training:
            bufs.accum.zero_()
        self._decode_native(z, bufs, self.training)
        if self.training:
            self._update_running(B, 7, 14)
        return bufs.act[13].reshape(B, X_DIM).clone()

    def forward(self, x, return_latent_rec=False, noise=None):
        """Send `x` round trip and compute the loss (negative ELBO summed over the
        batch; ava/models/vae.py:273-327).  The returned loss supports
        ``.backward()`` in train and eval mode (eval: BatchNorm with the running buffers, which the
        backward leaves unchanged): gradients w.r.t. every parameter and, if `x` requires grad, the
        input come from the native backward pass.

        `noise` (optional, addition): (eps_W [B,1], eps_D [B,z]) to use instead of
        drawing them with torch.randn.

        Under ``enable_data_parallel`` this, ``encode`` and ``decode`` and their backward passes
        stay local to the rank: no collectives and no BatchNorm statistics exchange."""
        params = self._params_of("all")
        if self._grad_wanted(x, [p for _, p in params]):
            loss, z, x_rec = _LossFn.apply(self, x, noise, [n for n, _ in params], *[p for _, p in params])
        else:
            bufs = self._forward_native(x, noise, self.training, want_grad_seed=False)
            loss = bufs.loss[0].clone()
            z, x_rec = bufs.z, bufs.act[13]
        if return_latent_rec:
            return loss, z.detach().cpu().numpy(), \
                x_rec.view(-1, X_SHAPE[0], X_SHAPE[1]).detach().cpu().numpy()
        return loss

    def compute_loss(self, x, noise=None):
        """Alias for ``forward(x)`` (named in the north-star API; the reference has
        no such method)."""
        return self.forward(x, noise=noise)

    # ------------------------------------------------------------ data parallel
    def enable_data_parallel(self, process_group=None, fused=None, sync_bn=False):
        """Shard batches over the ranks of `process_group` (default: WORLD), one process
        per GPU.  Semantics (SURVEY.md section 5): the loss is a batch SUM, so rank
        gradients are SUMMED (not averaged) -- the update equals the reference's at the
        global batch; BatchNorm uses each rank's local batch statistics (every rank ==
        the reference run on its shard) and the running buffers are averaged across ranks
        at epoch boundaries (exactly what per-step averaging would give, since the
        running-average recursion is linear).  Parameters are broadcast from rank 0.

        `fused` (default: on for CUDA ranks of one NCCL node with <= 8 ranks; environment
        AVA_B200_DP_FUSED=0 turns it off): the optimizer step and its two collectives run as
        ONE kernel per rank over NVLink peer memory (csrc/dp.cu: each rank sums its 1/world
        slice of everybody's gradient, applies Adam to that slice, stores the new parameters
        into every rank's buffer); gradients, parameters and flags then live in symmetric
        memory.  Otherwise: bucketed NCCL all-reduces overlapped with the backward pass.

        `sync_bn=True`: synchronised BatchNorm.  Every BatchNorm layer of a training step
        (``train_step``, and so ``train_epoch`` / ``train_loop``) normalises with the statistics of
        the GLOBAL batch -- the concatenation of the ranks' shards, which is what the reference's
        single process sees -- so loss, summed gradients, update and running buffers are the
        reference's at the global batch (up to rounding), for any split of the batch over the ranks,
        empty shards included.  Each step exchanges 14 forward and 13 backward statistics blocks
        over NVLink peer memory (csrc/bnsync.cu); the running buffers are updated from the global
        statistics, identically on every rank, and are not re-averaged at epoch ends.  Works with
        both optimizer paths.  Needs CUDA ranks of one NCCL group with at most 8 ranks and symmetric
        memory; otherwise this raises.  ``encode``, ``decode``, ``forward``, ``test_epoch`` and
        ``get_latent`` keep per-rank statistics (they are not collectives: ranks need not call them
        in lockstep)."""
        import torch.distributed as dist
        group = process_group if process_group is not None else dist.group.WORLD
        if sync_bn and not (self._flat_p.is_cuda and dist.get_backend(group) == "nccl"
                            and dist.get_world_size(group) <= _DP_MAX_WORLD):
            raise RuntimeError("ava_b200: synchronised BatchNorm needs CUDA ranks of one NCCL group with at "
                               "most %d ranks (got backend %r, %d ranks, model on %s)"
                               % (_DP_MAX_WORLD, dist.get_backend(group), dist.get_world_size(group),
                                  self._flat_p.device))
        self._dp_group = group
        self._dp_world = dist.get_world_size(self._dp_group)
        self._dp_rank = dist.get_rank(self._dp_group)
        for t in (self._flat_p, self._flat_run, self._nbt, self._flat_m, self._flat_v):
            dist.broadcast(t, src=dist.get_global_rank(self._dp_group, 0), group=self._dp_group)
        self._dp_fused = None
        want = fused if fused is not None else os.environ.get("AVA_B200_DP_FUSED", "1") != "0"
        if want and self._dp_world > 1:
            ok = (self._flat_p.is_cuda and dist.get_backend(self._dp_group) == "nccl"
                  and self._dp_world <= _DP_MAX_WORLD)
            if ok:
                try:
                    self._enable_fused_dp()
                except Exception as e:          # no symmetric memory / no peer access on this box
                    if fused:
                        raise
                    warnings.warn("ava_b200: fused NVLink data-parallel step unavailable (%s: %s); "
                                  "using bucketed NCCL all-reduces" % (type(e).__name__, e))
                    self._dp_fused = None
            elif fused:
                raise RuntimeError("ava_b200: fused data parallelism needs CUDA ranks of one NCCL group "
                                   "with at most %d ranks" % _DP_MAX_WORLD)
        self._bn_sync = None
        if sync_bn and self._dp_world > 1:
            try:
                self._enable_sync_bn()
            except Exception as e:
                raise RuntimeError("ava_b200: synchronised BatchNorm could not set up its symmetric-memory "
                                   "exchange buffer (%s: %s)" % (type(e).__name__, e)) from e
        return self

    def _enable_sync_bn(self):
        """Each rank's two exchange slots and its flag in one small symmetric-memory allocation of
        its own (independent of the fused optimizer's); the table of peer pointers for
        csrc/bnsync.cu."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        dev, W = self._flat_p.device, self._dp_world
        buf = symm.empty(2 * _BN_SYNC_SLOT + 1, dtype=torch.float64, device=dev)   # slots | flag
        buf.zero_()
        hdl = symm.rendezvous(buf, self._dp_group)
        ptrs = [int(a) for a in hdl.buffer_ptrs]
        assert len(ptrs) == W and ptrs[self._dp_rank] == buf.data_ptr()
        peers = _BnSyncPeers()
        for r in range(W):
            peers.slots[r] = ptrs[r]
            peers.flags[r] = ptrs[r] + 8 * 2 * _BN_SYNC_SLOT
        local = torch.zeros(2, dtype=torch.int32, device=dev)
        zeros = torch.zeros(2 * 14 * 64, dtype=torch.float64, device=dev)   # an empty shard's stats | dstats
        torch.cuda.synchronize(dev)
        dist.barrier(group=self._dp_group)       # every rank's flag is zero before anyone signals
        self._bn_sync = {"buf": buf, "hdl": hdl, "peers": peers, "local": local, "zeros": zeros}
        self._graphs = {}

    def _bn_exchange(self, l, B, block, forward):
        """Synchronised BatchNorm: layer l's sums in `block` (the stats or dstats of a _Buffers) become
        the global sums scaled by B / global batch (csrc/bnsync.cu); a forward exchange also applies the
        layer's running-buffer update from the global statistics."""
        f = self._bn_sync
        call("ava_b200_bn_stats_exchange", ctypes.byref(f["peers"]), self._dp_rank, self._dp_world,
             block.data_ptr() + 8 * 64 * l, self._bn_channels[l], B * _LAYERS[l][4] ** 2,
             ptr(self._flat_run) if forward else None, 64 * l, 64 * l + 32,
             (self._nbt.data_ptr() + 8 * l) if forward else None, _BN_MOMENTUM, ptr(f["local"]), _stream())

    def _bn_exchange_empty(self):
        """An empty shard's part of a step's 27 exchanges, in the order a step issues them: it
        contributes zero sums and a zero count, and still applies the running-buffer updates."""
        zeros = self._bn_sync["zeros"]
        zeros.zero_()
        for l in range(14):
            self._bn_exchange(l, 0, zeros, forward=True)
        for l in range(13, 0, -1):
            self._bn_exchange(l, 0, zeros[14 * 64:], forward=False)

    def _rebind_flat(self, flat_p, flat_g):
        """Move the flat parameter / gradient storage into the given buffers (same layout) and
        re-point every nn.Parameter and gradient view; captured graphs point at the old ones."""
        flat_p.copy_(self._flat_p)
        flat_g.zero_()
        params = dict(self.named_parameters())
        for k, o in self._off.items():
            p = params[k]
            n = p.numel()
            p.data = flat_p[o:o + n].view(p.shape)
            self._views_g[k] = flat_g[o:o + n].view(p.shape)
        self._flat_p, self._flat_g = flat_p, flat_g
        self._graphs = {}

    def _enable_fused_dp(self):
        """Gradients | parameters | flags in ONE symmetric-memory allocation, peer-mapped on every
        rank (torch.distributed._symmetric_memory); the table of peer pointers for csrc/dp.cu."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        n, dev, W = self._n_flat, self._flat_p.device, self._dp_world
        buf = symm.empty(2 * n + 64, dtype=torch.float32, device=dev)
        buf.zero_()
        hdl = symm.rendezvous(buf, self._dp_group)
        ptrs = [int(a) for a in hdl.buffer_ptrs]
        assert len(ptrs) == W and ptrs[self._dp_rank] == buf.data_ptr()
        self._rebind_flat(buf[n:2 * n], buf[:n])
        def table(mc):
            peers = _DpPeers()
            for r in range(W):
                peers.grad[r] = ptrs[r]
                peers.param[r] = ptrs[r] + 4 * n
                peers.flags[r] = ptrs[r] + 8 * n
            peers.grad_mc = mc if mc else None
            peers.param_mc = (mc + 4 * n) if mc else None
            return peers
        mc = 0
        try:
            mc = int(hdl.multicast_ptr) if hdl.has_multicast_support else 0
        except Exception:
            mc = 0
        peers_p2p, peers_mc = table(0), (table(mc) if mc else None)
        # Which variant: AVA_B200_DP_MULTIMEM=1/0 forces it; default by measurement (bench.py
        # dp_diag, profiles/r02_summary.md): plain peer loads/stores win on 2 GPUs (every byte
        # crosses one link either way and the switch reduction adds latency), the in-switch
        # reduction wins from 4 GPUs on (a rank reads its slice once instead of world times)
        env = os.environ.get("AVA_B200_DP_MULTIMEM")
        use_mc = bool(mc) and (env == "1" if env in ("0", "1") else W >= _DP_MULTIMEM_MIN_WORLD)
        peers = peers_mc if use_mc else peers_p2p
        local = torch.zeros(4, dtype=torch.int32, device=dev)
        torch.cuda.synchronize(dev)
        dist.barrier(group=self._dp_group)       # every rank's flags are zero before anyone signals
        self._dp_fused = {"buf": buf, "hdl": hdl, "peers": peers, "peers_p2p": peers_p2p, "peers_mc": peers_mc,
                          "local": local, "multimem": use_mc, "multimem_available": bool(mc)}

    def _adam_dp_native(self):
        """The fused data-parallel optimizer step (csrc/dp.cu)."""
        f = self._dp_fused
        call("ava_b200_adam_step_dp", ctypes.byref(f["peers"]), self._dp_rank, self._dp_world,
             ptr(self._flat_m), ptr(self._flat_v), self._n_flat, ptr(self._step_dev), ptr(self._hyper_dev),
             1.0, ptr(f["local"]), _stream())
        self._step_host += 1

    def dp_check_status(self):
        """Raise if a peer ever failed to arrive at a fused data-parallel step (one device read)."""
        f = getattr(self, "_dp_fused", None)
        if f is not None and int(f["local"][2].item()) != 0:
            raise RuntimeError("ava_b200: a data-parallel peer did not arrive within the kernel's timeout; "
                               "the replicas are out of step")
        b = getattr(self, "_bn_sync", None)
        if b is not None and int(b["local"][1].item()) != 0:
            raise RuntimeError("ava_b200: a data-parallel peer did not arrive at a BatchNorm statistics "
                               "exchange within the kernel's timeout; the replicas are out of step")

    def _gather_moment_shards(self):
        """Fused data parallelism shards the Adam moments (rank r keeps slice r current): bring every
        slice to every rank (checkpoints are written by rank 0 and must hold them all)."""
        if getattr(self, "_dp_fused", None) is None:
            return
        import torch.distributed as dist
        n4, W = self._n_flat // 4, self._dp_world
        for r in range(W):
            lo, hi = 4 * (n4 * r // W), 4 * (n4 * (r + 1) // W)
            src = dist.get_global_rank(self._dp_group, r)
            dist.broadcast(self._flat_m[lo:hi], src=src, group=self._dp_group)
            dist.broadcast(self._flat_v[lo:hi], src=src, group=self._dp_group)

    def _grad_buckets(self):
        """(early, mid, late) slices of the flat gradient buffer, in the order the backward pass
        completes them (SURVEY section 5 item 2):
        `early` = fc5..fc8 + convt1..7 (36 MB incl. fc8.weight), final after the decoder half;
        `mid`   = fc1..fc43 (34 MB incl. fc1.weight), final after the encoder's dense layers --
                  its all-reduce overlaps the encoder conv backward (a third of the backward);
        `late`  = conv1..7 and the 14 BatchNorm affine pairs (0.1 MB), final at the very end."""
        a0 = self._off["fc1.weight"]
        a1 = self._off["fc5.weight"]
        a2 = self._off["bn1.weight"]
        return [(a1, a2)], [(a0, a1)], [(0, a0), (a2, self._n_flat)]

    def _allreduce(self, slices, async_op):
        import torch.distributed as dist
        return [dist.all_reduce(self._flat_g[lo:hi], op=dist.ReduceOp.SUM, group=self._dp_group,
                                async_op=async_op) for lo, hi in slices if hi > lo]

    def _sync_bn_buffers(self):
        """Average the BatchNorm running buffers over the ranks."""
        if self._dp_world > 1:
            import torch.distributed as dist
            dist.all_reduce(self._flat_run, op=dist.ReduceOp.SUM, group=self._dp_group)
            self._flat_run.div_(self._dp_world)

    def loss_constant(self):
        """The two Gaussian normalising constants the reference adds ONCE PER BATCH
        (quirk F6, ava/models/vae.py:316-318)."""
        return 0.5 * self.z_dim * math.log(2 * math.pi) + \
            0.5 * X_DIM * math.log(2 * math.pi / self.model_precision)

    def _graph_wanted(self, B):
        if self._flat_p.device.type != "cuda":
            return False
        if self.cuda_graphs == 'auto':
            return True     # measured: 1.41 vs 1.68 ms at batch 64, 8.13 vs 8.46 ms at batch 1024
        return bool(self.cuda_graphs)

    def _train_step_graph(self, x, noise):
        """The whole step (~160 launches) replayed as one CUDA graph per batch size (data
        parallel: four graphs with the collectives between them, _capture_dp_segments): at
        batch 64 the step is otherwise bound by host launch overhead, and even at batch 1024
        the launch gaps between the many small kernels cost 4 %.  The first two steps
        at a new batch size run eagerly (they also warm up lazy initialisation), the third
        is captured.  Inputs and noise are copied into static buffers before each replay."""
        B = x.shape[0]
        st = self._graphs.get(B)
        if st is None:
            dev = self._flat_p.device
            st = self._graphs[B] = {
                "count": 0, "graph": None,
                "x": torch.empty(B, X_SHAPE[0], X_SHAPE[1], dtype=torch.float32, device=dev),
                "ew": torch.empty(B, 1, dtype=torch.float32, device=dev),
                "ed": torch.empty(B, self.z_dim, dtype=torch.float32, device=dev)}
        st["x"].copy_(x, non_blocking=True)
        if noise is not None:
            st["ew"].copy_(noise[0].reshape(B, 1))
            st["ed"].copy_(noise[1].reshape(B, self.z_dim))
        else:
            st["ew"].normal_()     # same draw order as rsample: eps_W first, then eps_D
            st["ed"].normal_()
        if st["graph"] is None:
            st["count"] += 1
            if st["count"] <= 2:
                return self._train_step_eager(st["x"], (st["ew"], st["ed"]))
            try:
                host_step = self._step_host
                if self._dp_world > 1 and self._dp_fused is None:
                    st["graph"] = self._capture_dp_segments(st)
                else:
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        st["loss"] = self._train_step_eager(st["x"], (st["ew"], st["ed"]))
                    st["graph"] = [g]
                self._step_host = host_step      # capture records, it does not execute
                # the graph owns references to everything it points into
                st["bufs"], st["scratch"] = self._bufs[B], (self._scratch, getattr(self, "_scratch_side", None))
            except Exception:
                self.cuda_graphs = False
                st["graph"] = None
                torch.cuda.synchronize()
                return self._train_step_eager(st["x"], (st["ew"], st["ed"]))
        self._buffers_for(B)             # keep this size most recently used
        self._cur = st["bufs"]
        graphs = st["graph"]
        if len(graphs) == 1:
            graphs[0].replay()
        else:
            # data parallel: the collectives stay OUTSIDE the graphs (NCCL kernels captured into a
            # graph ran slower than eager ones here and the process hung at teardown); each is
            # launched right after the segment that completes its bucket and overlaps the next
            early, mid, late = self._grad_buckets()
            graphs[0].replay()
            works = self._allreduce(early, async_op=True)
            graphs[1].replay()
            works += self._allreduce(mid, async_op=True)
            graphs[2].replay()
            works += self._allreduce(late, async_op=True)
            for w in works:
                w.wait()
            graphs[3].replay()
        self._step_host += 1
        return st["loss"]

    def _capture_dp_segments(self, st):
        """The data-parallel step as four CUDA graphs -- forward + decoder backward | dense encoder
        backward | encoder conv backward | Adam -- with the three gradient all-reduces between
        them.  All four share one memory pool (they run strictly in this order)."""
        x, noise = st["x"], (st["ew"], st["ed"])
        graphs = [torch.cuda.CUDAGraph() for _ in range(4)]
        pool = torch.cuda.graph_pool_handle()
        with torch.cuda.graph(graphs[0], pool=pool):
            bufs = self._forward_native(x, noise, True, want_grad_seed=True)
            self._bwd_decoder(bufs)
            self._side_join()        # (a capture ends with every forked stream joined)
        with torch.cuda.graph(graphs[1], pool=pool):
            self._bwd_dense_encoder(bufs)
            self._side_join()
        with torch.cuda.graph(graphs[2], pool=pool):
            self._bwd_conv_encoder(bufs)
            self._side_join()
        with torch.cuda.graph(graphs[3], pool=pool):
            self._adam_native()
        st["loss"] = bufs.loss[0]
        return graphs

    def train_step(self, x, noise=None):
        """zero_grad + forward + backward + Adam for one batch, entirely native
        (the body of the loop at ava/models/vae.py:347-353).  Returns the loss as a
        0-dim device tensor (no host sync).  Under data parallelism `x` is this rank's
        shard and the gradient all-reduce overlaps the encoder half of the backward."""
        self._ensure_optimizer_state()
        self._require_cuda()
        self._sync_hyper()
        x = self._as_input(x)
        self._bn_sync_on = self._bn_sync is not None
        try:
            if x.shape[0] == 0:
                return self._train_step_empty()
            if self._graph_wanted(x.shape[0]):
                return self._train_step_graph(x, noise)
            return self._train_step_eager(x, noise)
        finally:
            self._bn_sync_on = False

    def _train_step_empty(self):
        """This rank's shard of the global batch is empty (a ragged last batch smaller than the
        world size): contribute zero gradients to the same all-reduces as the other ranks and
        apply the same update.  The per-batch loss constants are booked as on every other rank
        (_epoch_loss counts them once per global batch)."""
        if self._dp_world <= 1:
            raise ValueError("train_step: empty batch")
        if self._bn_sync is not None:
            self._bn_exchange_empty()
        self._flat_g.zero_()
        if self._dp_fused is not None:
            self._adam_dp_native()
        else:
            early, mid, late = self._grad_buckets()
            for w in self._allreduce(early + mid + late, async_op=True):
                w.wait()
            self._adam_native()
        self._loss_sum += self.loss_constant()
        return torch.full((), self.loss_constant(), dtype=torch.float32, device=self._flat_p.device)

    def _train_step_eager(self, x, noise):
        bufs = self._forward_native(x, noise, True, want_grad_seed=True)
        if self._dp_world > 1 and self._dp_fused is not None:
            # gradients stay local: the optimizer kernel does the reduction over NVLink itself
            self._backward_native(bufs)
            self._adam_dp_native()
            return bufs.loss[0]
        if self._dp_world > 1:
            early, mid, late = self._grad_buckets()
            works = []
            self._backward_native(
                bufs, after_decoder=lambda: works.extend(self._allreduce(early, async_op=True)),
                after_dense=lambda: works.extend(self._allreduce(mid, async_op=True)))
            works += self._allreduce(late, async_op=True)
            for w in works:
                w.wait()
        else:
            self._backward_native(bufs)
        self._adam_native()
        return bufs.loss[0]

    def grad_dict(self):
        """name -> gradient view, as left by the last backward pass."""
        return dict(self._views_g)

    def train_epoch(self, train_loader):
        """Train the model for a single epoch (ava/models/vae.py:330-358)."""
        self.train()
        self._require_cuda()
        self._loss_sum.zero_()
        n_steps = 0
        for batch_idx, data in enumerate(prefetch_to_device(train_loader, self._flat_p.device)):
            self.train_step(data)
            n_steps += 1
        # one device->host read per epoch instead of loss.item() per step
        train_loss = self._epoch_loss(n_steps)
        train_loss /= len(train_loader.dataset)
        print('Epoch: {} Average loss: {:.4f}'.format(self.epoch, train_loss))
        self.epoch += 1
        return train_loss

    def test_epoch(self, test_loader):
        """Test the model on a held-out test set (ava/models/vae.py:361-385)."""
        self.eval()
        self._require_cuda()
        self._loss_sum.zero_()
        n_steps = 0
        with torch.no_grad():
            for i, data in enumerate(prefetch_to_device(test_loader, self._flat_p.device)):
                if len(data) == 0 and self._dp_world > 1:    # empty shard of a small last batch
                    self._loss_sum += self.loss_constant()
                else:
                    self._forward_native(data, None, False, want_grad_seed=False)
                n_steps += 1
        test_loss = self._epoch_loss(n_steps)
        test_loss /= len(test_loader.dataset)
        print('Test loss: {:.4f}'.format(test_loss))
        return test_loss

    def _epoch_loss(self, n_steps):
        """Sum of the per-batch losses of this epoch (one device->host read).  Under data
        parallelism: summed over ranks, with the per-batch constants counted once per
        GLOBAL batch as the reference would, and the BN running buffers re-averaged (not under
        synchronised BatchNorm: there they are already identical on every rank)."""
        if self._dp_world > 1:
            import torch.distributed as dist
            dist.all_reduce(self._loss_sum, op=dist.ReduceOp.SUM, group=self._dp_group)
            if self._bn_sync is None:
                self._sync_bn_buffers()
            return float(self._loss_sum.item()) - (self._dp_world - 1) * n_steps * self.loss_constant()
        return float(self._loss_sum.item())

    def train_loop(self, loaders, epochs=100, test_freq=2, save_freq=10, vis_freq=1):
        """Train the model for multiple epochs, testing and saving along the way
        (ava/models/vae.py:388-430)."""
        print("=" * 40)
        print("Training: epochs", self.epoch, "to", self.epoch + epochs - 1)
        print("Training set:", len(loaders['train'].dataset))
        print("Test set:", len(loaders['test'].dataset))
        print("=" * 40)
        for epoch in range(self.epoch, self.epoch + epochs):
            loss = self.train_epoch(loaders['train'])
            self.loss['train'][epoch] = loss
            if (test_freq is not None) and (epoch % test_freq == 0):
                loss = self.test_epoch(loaders['test'])
                self.loss['test'][epoch] = loss
            if (save_freq is not None) and (epoch % save_freq == 0) and (epoch > 0):
                filename = "checkpoint_" + str(epoch).zfill(3) + '.tar'
                self.save_state(filename)
            if (vis_freq is not None) and (epoch % vis_freq == 0):
                self.visualize(loaders['test'])

    # ------------------------------------------------------------- checkpointing
    def _ensure_optimizer_state(self):
        """Make torch.optim.Adam's per-parameter state alias the flat moment buffers
        (torch creates that state lazily at the first step; so do we)."""
        params = dict(self.named_parameters())
        first = next(iter(params.values()))
        st = self.optimizer.state.get(first)
        if st is not None and 'exp_avg' in st and \
                st['exp_avg'].data_ptr() == self._views_m[next(iter(params))].data_ptr():
            return
        adopted_step = None
        for k, p in params.items():
            st = self.optimizer.state.get(p)
            if st is not None and 'exp_avg' in st and \
                    st['exp_avg'].data_ptr() != self._views_m[k].data_ptr():
                # state created by torch (load_state_dict or a user-driven optimizer.step()):
                # its moments and step count win.  State that already aliases the flat buffers
                # is ours: its `step` entry is only published at save_state (the live count is
                # self._step_host / self._step_dev) and must not be re-adopted.
                self._views_m[k].copy_(st['exp_avg'])
                self._views_v[k].copy_(st['exp_avg_sq'])
                adopted_step = float(st['step'])
            self.optimizer.state[p] = {'step': torch.tensor(float(self._step_host)),
                                       'exp_avg': self._views_m[k], 'exp_avg_sq': self._views_v[k]}
        if adopted_step is not None:
            self._step_host = int(adopted_step)
            self._step_dev.fill_(float(self._step_host))
            self._publish_optimizer_steps()

    def _publish_optimizer_steps(self):
        for p in self.parameters():
            st = self.optimizer.state.get(p)
            if st is not None:
                st['step'] = torch.tensor(float(self._step_host))

    def save_state(self, filename):
        """Save all the model parameters to the given file (vae.py:433-446); the file
        is readable by the reference's load_state and vice versa."""
        self._gather_moment_shards()     # (fused data parallelism: a collective -- every rank calls save_state)
        if self._step_host > 0:
            self._ensure_optimizer_state()
            self._publish_optimizer_steps()
        layers = self._get_layers()
        state = {}
        for layer_name in layers:
            state[layer_name] = layers[layer_name].state_dict()
        state['optimizer_state'] = self.optimizer.state_dict()
        state['loss'] = self.loss
        state['z_dim'] = self.z_dim
        state['epoch'] = self.epoch
        state['lr'] = self.lr
        state['save_dir'] = self.save_dir
        filename = os.path.join(self.save_dir, filename)
        if self._dp_world > 1 and self._dp_rank != 0:
            return  # only rank 0 writes
        torch.save(state, filename)

    def load_state(self, filename):
        """Load all the model parameters from the given ``.tar`` file
        (vae.py:449-472).  `self.lr`, `self.save_dir`, `self.z_dim` are not loaded."""
        checkpoint = torch.load(filename, map_location=self.device)
        assert checkpoint['z_dim'] == self.z_dim
        layers = self._get_layers()
        for layer_name in layers:
            layer = layers[layer_name]
            layer.load_state_dict(checkpoint[layer_name])
        self.optimizer.load_state_dict(checkpoint['optimizer_state'])
        self._step_host = 0
        self._step_dev.zero_()
        self._flat_m.zero_()
        self._flat_v.zero_()
        self._ensure_optimizer_state()
        self.loss = checkpoint['loss']
        self.epoch = checkpoint['epoch']

    def load_flat_state(self, state):
        """Copy a {state_dict-style key: tensor} mapping (parameters and BN buffers)
        into the model (used by tests/bench to install seeded weights)."""
        own = dict(self.named_parameters())
        own.update(dict(self.named_buffers()))
        with torch.no_grad():
            for k, v in state.items():
                own[k].copy_(torch.as_tensor(v).to(own[k].dtype))

    # ---------------------------------------------------------------- inspection
    def visualize(self, loader, num_specs=5, gap=(2, 6), save_filename='reconstruction.pdf'):
        """Plot spectrograms and their reconstructions (vae.py:475-516).  Plotting
        needs matplotlib; without it the arrays are still returned."""
        assert num_specs <= len(loader.dataset) and num_specs >= 1
        indices = np.random.choice(np.arange(len(loader.dataset)), size=num_specs, replace=False)
        specs = torch.stack(loader.dataset[indices]).to(self.device)
        with torch.no_grad():
            _, _, rec_specs = self.forward(specs, return_latent_rec=True)
        specs = specs.detach().cpu().numpy()
        all_specs = np.stack([specs, rec_specs])
        save_filename = os.path.join(self.save_dir, save_filename)
        try:
            from ..plotting import grid_plot
            grid_plot(all_specs, gap=gap, filename=save_filename)
        except ImportError:
            pass
        return specs, rec_specs

    def get_latent(self, loader):
        """Get latent means for all syllables in the given loader (vae.py:519-547).
        As in the reference the module's train/eval mode is NOT changed here."""
        self._require_cuda()
        n = len(loader.dataset)
        Z = self.z_dim
        dev_latent = torch.zeros(n, Z, dtype=torch.float32, device=self._flat_p.device)
        i = 0
        with torch.no_grad():
            for data in prefetch_to_device(loader, self._flat_p.device):
                x = self._as_input(data)
                B = x.shape[0]
                if B == 0:
                    continue
                bufs = self._buffers_for(B)
                self._cur = bufs
                self._scratch_need = self._scratch_need_for(B)
                if self.training:
                    bufs.accum.zero_()
                self._encode_native(x, bufs, self.training)
                if self.training:
                    self._update_running(B, 0, 7)
                dev_latent[i:i + B].copy_(bufs.heads[:, :Z])
                i += B
        # single device->host transfer, widened to the reference's float64
        return dev_latent.cpu().numpy().astype(np.float64)


class _Lease:
    """An activation set checked out by a call that recorded an autograd graph (VAE._grad_buffers).
    It goes back to the model's free list when the graph's backward has run (a second backward of
    the same graph raises) or when the graph is freed without one."""

    def __init__(self, model, bufs):
        self.model, self.bufs = model, bufs

    def release(self):
        if self.bufs is not None:
            self.model._release_grad_buffers(self.bufs)
            self.bufs = None

    __del__ = release


def _checkout(ctx, model, B, train):
    """Start of a recording forward: an owned activation set (running buffers snapshotted in eval
    mode), made the model's current one."""
    bufs = model._grad_buffers(B)
    bufs.snapshot_running(model._flat_run, train)
    ctx.lease = _Lease(model, bufs)
    model._cur = bufs
    model._scratch_need = model._scratch_need_for(B)
    return bufs


def _begin_backward(ctx):
    bufs = ctx.lease.bufs
    if bufs is None:
        raise RuntimeError("ava_b200: this graph's backward has already run; its activations are released "
                           "(a second backward through the same VAE call is not supported)")
    ctx.lease.model._scratch_need = ctx.lease.model._scratch_need_for(bufs.B)
    bufs.alloc_backward(ctx.lease.model.z_dim)
    return ctx.lease.model, bufs


def _param_grads(ctx, model, names, scale=None):
    """The flat gradient buffer's entries for the call's parameters, copied out (the buffer is
    shared with every other backward and with train_step); None where no gradient is wanted."""
    out = []
    for i, n in enumerate(names):          # (ctx.first: index of the first parameter among the inputs)
        if not ctx.needs_input_grad[ctx.first + i]:
            out.append(None)
        else:
            g = model._views_g[n]
            out.append(g * scale if scale is not None else g.clone())
    return tuple(out)


class _EncodeFn(torch.autograd.Function):
    """encode(x) -> (mu, u, d) with the native backward: latent_heads_grad, the dense encoder
    backward and the conv encoder backward (+ layer 0's data gradient when x requires grad)."""

    @staticmethod
    def forward(ctx, model, x, names, *params):
        model._require_cuda()
        ctx.x_meta = (x.device, x.dtype) if torch.is_tensor(x) else None
        x = model._as_input(x)
        B, Z, train = x.shape[0], model.z_dim, model.training
        bufs = _checkout(ctx, model, B, train)
        bufs.accum.zero_()
        model._encode_native(x, bufs, train)
        if train:
            model._update_running(B, 0, 7)
        model._linear(bufs.h3[:, 128:], 192, "fc43.weight", "fc43.bias", bufs.d, Z, B, Z, 64, 2)
        bufs.x = x
        ctx.names, ctx.first = names, 3
        ctx.set_materialize_grads(False)
        heads = bufs.heads
        return heads[:, :Z].clone(), heads[:, Z:2 * Z].clone().unsqueeze(-1), bufs.d.clone()

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dmu, du, dd):
        model, bufs = _begin_backward(ctx)
        B, Z, s = bufs.B, model.z_dim, _stream()
        seeds = [None if t is None else t.to(torch.float32).reshape(B, Z).contiguous() for t in (dmu, du, dd)]
        bufs.dstats[:7 * 64].zero_()
        bufs.tsums[:7 * 288].zero_()
        call("ava_b200_latent_heads_grad", ptr(seeds[0]), ptr(seeds[1]), ptr(seeds[2]), ptr(bufs.d), B, Z,
             ptr(bufs.gheads), s)
        model._bwd_dense_encoder(bufs, latent=False)
        dx = torch.empty_like(bufs.x) if ctx.needs_input_grad[1] else None
        model._bwd_conv_encoder(bufs, dx=dx, n_bn=7)
        model._side_join()
        grads = _param_grads(ctx, model, ctx.names)
        ctx.lease.release()
        if dx is not None:
            dx = dx.to(device=ctx.x_meta[0], dtype=ctx.x_meta[1])
        return (None, dx, None) + grads


class _DecodeFn(torch.autograd.Function):
    """decode(z) -> x_rec [B,16384] with the native backward: the seed's border sums
    (ava_b200_dz_border_sums) and the decoder backward, whose fc5 data gradient is dL/dz."""

    @staticmethod
    def forward(ctx, model, z, names, *params):
        model._require_cuda()
        ctx.z_meta = (z.device, z.dtype)
        B, train = z.shape[0], model.training
        bufs = _checkout(ctx, model, B, train)
        bufs.z.copy_(z.detach().reshape(B, model.z_dim))      # fc5's input, kept for its weight gradient
        bufs.accum.zero_()
        model._decode_native(bufs.z, bufs, train)
        if train:
            model._update_running(B, 7, 14)
        ctx.names, ctx.first = names, 3
        ctx.set_materialize_grads(False)
        return bufs.act[13].reshape(B, X_DIM).clone()

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gx):
        if gx is None:
            ctx.lease.release()
            return (None,) * (3 + len(ctx.names))
        model, bufs = _begin_backward(ctx)
        B, s = bufs.B, _stream()
        bufs.dstats[7 * 64:].zero_()
        bufs.tsums[7 * 288:].zero_()
        seed = bufs.g[0][:B * X_DIM]          # convt7's dz (no ReLU after it): the seed itself
        seed.copy_(gx.reshape(-1))
        call("ava_b200_dz_border_sums", ptr(seed), B, 1, X_SHAPE[0], X_SHAPE[1], 0,
             bufs.tsums.data_ptr() + 8 * 288 * 13, s)
        model._bwd_decoder(bufs)
        model._bn_param_grads(bufs, 7, 14)
        model._side_join()
        grads = _param_grads(ctx, model, ctx.names)
        gz = bufs.gz.to(device=ctx.z_meta[0], dtype=ctx.z_meta[1], copy=True) if ctx.needs_input_grad[1] else None
        ctx.lease.release()
        return (None, gz, None) + grads


class _LossFn(torch.autograd.Function):
    """Autograd glue: loss = VAE.forward(x) with the native backward pass (train or eval mode;
    the input gradient when x requires grad)."""

    @staticmethod
    def forward(ctx, model, x, noise, names, *params):
        model._require_cuda()
        ctx.x_meta = (x.device, x.dtype) if torch.is_tensor(x) else None
        x = model._as_input(x)
        train = model.training
        bufs = _checkout(ctx, model, x.shape[0], train)
        model._forward_native(x, noise, train, want_grad_seed=True, bufs=bufs)
        ctx.names, ctx.first = names, 4
        ctx.mark_non_differentiable(bufs.z, bufs.act[13])
        return bufs.loss[0].clone(), bufs.z, bufs.act[13]

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_loss, _gz, _gx):
        model, bufs = _begin_backward(ctx)
        dx = torch.empty_like(bufs.x) if ctx.needs_input_grad[1] else None
        model._backward_native(bufs, dx=dx)
        if dx is not None:
            # (the reconstruction seed in g[0] is gone by now: recomputed from x and x_rec)
            call("ava_b200_recon_input_grad", ptr(dx), ptr(bufs.x), ptr(bufs.act[13]), bufs.B * X_DIM,
                 float(model.model_precision), ptr(dx), _stream())
            dx = (dx * grad_loss).to(device=ctx.x_meta[0], dtype=ctx.x_meta[1])
        grads = _param_grads(ctx, model, ctx.names, scale=grad_loss)
        ctx.lease.release()
        return (None, dx, None, None) + grads


if __name__ == '__main__':
    pass
