"""Conformance of the spectrogram kernels (csrc/spec.cu) across the parameter space the entry points
accept, not only the two production parameter sets of oracle/spec_oracle.py.

  * `ava_b200_get_spec_batch` at every power-of-two nperseg from 16 to 4096 (all nine template
    instantiations, packing factors G = 8, 4, 2, 1), hops N/2, N/4, N, N/2 + 3 and 1, int16 /
    float32 / float64 samples with and without DC removal, target frequencies that read the DC and
    Nyquist bins, rows and columns of fill, n_f up to 129 and n_t up to 1000 (several output passes,
    odd row counts), single-run windows (nperseg <= 256) and windows of ~86 overlapping slot runs
    (nperseg >= 2048).
  * Every output ELEMENT is held to an extended-precision reference: a direct DFT in long double
    (80-bit on x86-64) of the needed frames and bins, with twiddles from the exact integer phase
    (j*b) mod N, log(scale*|X| + 1e-12), the kernel's own float64 interpolation weights, normalise
    and clip.  The bound is
        |got - ref| <= (TAU * log2(N) * kappa + 2^-45) / |spec_max - spec_min|,
        kappa = max over the four corners of A / (scale*|X| + 1e-12),
    A = scale * sum_j |s_j| w_j over the raw samples of the frame and of its neighbours in the list
    of needed frames (two frames share one packed complex FFT, so each one's rounding error scales
    with its partner's amplitude too).  kappa is the condition number of the log magnitude; where it
    is huge (spectral nulls at the 1e-12 floor) the bound says nothing, elsewhere it is tight.
    Every configuration runs at spec range [-28, 12], where nothing in range is clipped, at the
    production range [2, 6.5], and at that range inverted (fill value 1).
  * Outputs sit inside NaN guard bands: every element written, nothing outside; out == out64 in
    float32; calls with one output only and repeated calls are bit-identical.
  * `ava_b200_quantile_normalize` bit for bit against numpy, `ava_b200_window_time_tables` bit for
    bit against the host `bracket`, and the argument checks of all three entries.

The long-double reference is validated without a GPU by test_reference_matches_scipy_and_oracle.
Run with -s for the worst err/bound ratio per nperseg."""
import functools
import importlib
import math

import numpy as np
import pytest
import torch

from oracle import spec_oracle

PKG = "autoencoded-vocal-analysis_b200"
pre = importlib.import_module(PKG + ".preprocessing.utils")
_lib = importlib.import_module(PKG + "._lib")

TAU = 2.0 ** -48
FLOOR = 2.0 ** -45
LD = np.longdouble
EPS_LOG = LD(1e-12)           # the float64 constant the kernel adds, held exactly
PI_LD = 4 * np.arctan(LD(1))
WIDE = (-28.0, 12.0)          # log(1e-12) = -27.6: nothing in range is clipped
PROD = (2.0, 6.5)
RANGES = (WIDE, PROD, PROD[::-1])
SMEM_LIMIT = 227 * 1024
GUARD = 4096                  # 32-bit words of guard band on each side of every output
SENT = 0x7FF8DEAD             # a NaN as float32, and two of them a NaN as float64

SIGNALS = ("synth", "dc", "nyquist", "const", "bintone", "zeros")
TIMES = ("lin", "over", "rand", "onframe", "out")
FREQS = ("lin0", "mel", "wide", "randf")
N_FS = (128, 129, 37)
N_TS = (2, 128, 129, 300, 1000)
FSS = (32000, 44100, 250000)
DTYPES = (np.int16, np.float32, np.float64)
IS_F32 = {np.dtype(np.int16): 0, np.dtype(np.float32): 1, np.dtype(np.float64): 2}


def stream():
    return torch.cuda.current_stream().cuda_stream


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ------------------------------------------------------------------------------ configurations
def _config_list():
    """Every nperseg with each hop (the other axes rotate through their values), then eight edge
    configurations each at nperseg 16, 512, 1024 and 4096 that between them take every signal,
    target-time set, target-frequency set, n_f and n_t, and two long windows of >= 256 frames."""
    out = []

    def add(**c):
        c.setdefault("seed", len(out))
        out.append(c)

    i = 0
    for lg in range(4, 13):
        N = 1 << lg
        hops = [N // 2, N // 4, N, N // 2 + 3] + ([1] if N <= 32 else [])
        for h in hops:
            add(N=N, hop=h, fs=FSS[i % 3], dtype=DTYPES[(i // 3) % 3], dc=(i // 2) % 2 == 0,
                sig=SIGNALS[(5 * i) % 6 if h != 1 else 0], times=TIMES[(3 * i) % 5 if h != 1 else 0],
                freqs=FREQS[i % 4], n_f=N_FS[(i // 4) % 3], n_t=N_TS[(2 * i + 1) % 5 if h != 1 else 4])
            i += 1
    for N in (16, 512, 1024, 4096):
        hops = [N // 2, N // 4, N, N // 2 + 3]
        s = N.bit_length()
        for e in range(8):
            add(N=N, hop=hops[(e + s) % 4], fs=FSS[(e + s) % 3], dtype=DTYPES[(e // 2 + s) % 3],
                dc=(e + s) % 2 == 0, sig=SIGNALS[e % 6], times=TIMES[(e + s) % 5], freqs=FREQS[(e + 2 * s) % 4],
                n_f=N_FS[(e + s) % 3], n_t=N_TS[(2 * e + s) % 5])
    # ~86 runs of 3 new frames each (CF = 4 at nperseg >= 2048)
    add(N=4096, hop=1024, fs=250000, dtype=np.int16, dc=True, sig="synth", times="lin", freqs="lin0",
        n_f=128, n_t=1000, seg_frames=258)
    add(N=2048, hop=1024, fs=44100, dtype=np.float32, dc=False, sig="dc", times="rand", freqs="randf",
        n_f=37, n_t=1000, seg_frames=300)
    return out


CONFIGS = {}
for _c in _config_list():
    _c["id"] = "N%d-h%d-%s-%s-%s-%s-%s-f%d-t%d-%d" % (
        _c["N"], _c["hop"], np.dtype(_c["dtype"]).name, "dc" if _c["dc"] else "nodc", _c["sig"], _c["times"],
        _c["freqs"], _c["n_f"], _c["n_t"], _c["fs"])
    CONFIGS[_c["id"]] = _c
CONFIG_IDS = list(CONFIGS)


def make_signal(kind, n, fs, N, rng):
    if kind in ("synth", "dc"):
        y = spec_oracle.synth_audio(int(rng.integers(1 << 30)), n, fs, dtype=np.float64)
        return y + 1.2e4 if kind == "dc" else y
    if kind == "nyquist":
        return 32767.0 * (1 - 2 * (np.arange(n) % 2))
    if kind == "const":
        return np.full(n, 12345.0)
    if kind == "bintone":
        j = np.arange(n)
        return 8000 * np.cos(2 * np.pi * (N // 8) * j / N) + 5000 * np.cos(2 * np.pi * (3 * N // 8) * j / N + 0.3)
    assert kind == "zeros"
    return np.zeros(n)


def to_dtype(y, dtype):
    if np.dtype(dtype) == np.int16:
        return np.clip(np.round(y), -32768, 32767).astype(np.int16)
    return y.astype(dtype)


def segment_tables(N, hop, fs, flen, t1, t2):
    """SpecEngine._segments for one segment: (lo, seg_len (0 = too short), K, base frame times)."""
    s1, s2 = int(np.rint(t1 * fs)), int(np.rint(t2 * fs))
    lo, hi = max(0, s1), min(flen, s2)
    seg_len = hi - lo
    if seg_len < N or s2 <= 0 or s1 >= flen:
        seg_len, K = 0, 3
    else:
        K = int(pre.num_frames(seg_len, N, hop))
    base = np.arange(N / 2, N / 2 + K * hop, hop) / float(fs)
    base = base - (N / 2) / fs
    return lo, seg_len, K, base


@functools.lru_cache(maxsize=None)
def build_case(cid):
    """Audio of one file, the segment [t1, t2], targets and the kernel's tables."""
    c = CONFIGS[cid]
    N, hop, fs = c["N"], c["hop"], c["fs"]
    rng = np.random.default_rng(1000 + c["seed"])
    seg_n = c.get("seg_frames", 0) * hop or max(8 * N, 40 * hop, 2400)
    pad = 0 if c["times"] == "over" else N + 37
    body = make_signal(c["sig"], seg_n, fs, N, rng)
    # loud samples around the segment: a read outside [lo, lo + seg_len) would show
    loud = 20000.0 * np.sign(rng.standard_normal(pad))
    audio = to_dtype(np.concatenate([loud, body, loud[::-1]]), c["dtype"])
    flen = len(audio)
    if c["times"] == "over":
        t1, t2 = -0.3 * flen / fs, 1.3 * flen / fs
    else:
        t1, t2 = (pad + 0.25) / fs, (pad + seg_n + 0.25) / fs
    lo, seg_len, K, base = segment_tables(N, hop, fs, flen, t1, t2)
    assert seg_len == seg_n
    grid0 = max(0.0, t1)
    g = base[:K] + grid0
    n_t, n_f, d = c["n_t"], c["n_f"], t2 - t1
    kind = c["times"]
    if kind == "lin":
        tt = np.linspace(t1 + 0.05 * d, t2 - 0.05 * d, n_t)
    elif kind == "over":
        tt = np.linspace(t1, t2, n_t)
    elif kind == "rand":
        tt = rng.uniform(t1 - 0.1 * d, t2 + 0.1 * d, n_t)
        tt[1::5] = tt[0]                                   # duplicates, as the warped dataset makes
    elif kind == "onframe":
        tt = g[rng.integers(0, K, n_t)]
        tt[0], tt[-1] = g[0], g[K - 1]
    else:
        tt = np.linspace(g[K - 1] + 1e-3, g[K - 1] + 2e-3, n_t)
    fgrid = np.fft.rfftfreq(N, 1 / fs)
    kind = c["freqs"]
    if kind == "lin0":
        tf = np.linspace(0.0, fgrid[-1], n_f)              # bin 0 with weight 0, bin N/2 with weight 1
    elif kind == "mel":
        tf = pre._inv_mel(np.linspace(pre._mel(400.0), pre._mel(10e3), n_f))
    elif kind == "wide":
        tf = np.linspace(-0.05 * fs, 0.55 * fs, n_f)
    else:
        tf = rng.uniform(0.0, fs / 2, n_f)
    t_idx, t_frac = pre.bracket(np.array([grid0]), base, np.array([K]), tt[None, :])
    f_idx, f_frac = pre.bracket_1d(fgrid, tf)
    window = pre._hann_window(N)
    return dict(c=c, audio=audio, t1=t1, t2=t2, tt=tt, tf=tf, lo=lo, seg_len=seg_len, K=K, kmax=K,
                t_idx=t_idx[0], t_frac=t_frac[0], f_idx=f_idx, f_frac=f_frac, window=window,
                scale=float(1.0 / window.sum()))


# ------------------------------------------------------------------ extended-precision reference
@functools.lru_cache(maxsize=None)
def unit_circle(N):
    ph = 2 * PI_LD * np.arange(N, dtype=LD) / N
    return np.cos(ph), np.sin(ph)


def ld_spectrum(seg, N, hop, remove_dc, window, scale, frames, bins):
    """Direct DFT in long double of the given frames and bins of one segment (scipy.signal.stft
    framing: nperseg/2 zeros of boundary extension, zero padding).  Returns log(scale|X| + 1e-12),
    scale|X| [frames, bins] and A = scale * sum_j |s_j| w_j [frames] over the raw samples."""
    x = np.asarray(seg).astype(LD)
    L = len(x)
    mean = x.sum() / L if remove_dc else LD(0)
    j = np.arange(N)
    idx = frames[:, None] * hop + j[None, :] - N // 2
    inside = (idx >= 0) & (idx < L)
    raw = np.where(inside, x[np.clip(idx, 0, L - 1)], LD(0))
    w = window.astype(LD)
    v = np.where(inside, raw - mean, LD(0)) * w
    cos, sin = unit_circle(N)
    ph = (j[:, None] * bins[None, :]) % N
    re, im = v @ cos[ph], v @ sin[ph]
    sc = LD(scale)
    M = sc * np.sqrt(re * re + im * im)
    A = sc * (np.abs(raw) * w).sum(axis=1)
    return np.log(M + EPS_LOG), M, A


def ld_needed(seg, N, hop, remove_dc, window, scale, K, t_idx, f_idx):
    """The long-double log spectrum of the frames and bins that the tables bracket, with A widened
    to the neighbours in the needed-frame list (a frame's packed-FFT partner is one of them)."""
    vt = (t_idx >= 0) & (t_idx + 1 < K)
    vf = f_idx >= 0
    frames = np.unique(np.concatenate([t_idx[vt], t_idx[vt] + 1])).astype(np.int64)
    bins = np.unique(np.concatenate([f_idx[vf], f_idx[vf] + 1])).astype(np.int64)
    if len(frames) and len(bins):
        LS, M, A = ld_spectrum(seg, N, hop, remove_dc, window, scale, frames, bins)
    else:
        LS = M = np.zeros((len(frames), len(bins)), LD)
        A = np.zeros(len(frames), LD)
    Aeff = A.copy()
    if len(A) > 1:
        Aeff[1:] = np.maximum(Aeff[1:], A[:-1])
        Aeff[:-1] = np.maximum(Aeff[:-1], A[1:])
    return dict(frames=frames, bins=bins, LS=LS, M=M, Aeff=Aeff)


def fill_value(smin, smax):
    return float(np.clip((-1 / 1e-12 - smin) / (smax - smin), 0.0, 1.0))


def ld_interp(R, N, K, t_idx, t_frac, f_idx, f_frac, smin, smax):
    """(reference [n_f, n_t] long double, elementwise bound [n_f, n_t]; 0 where exact)."""
    ref = np.full((len(f_idx), len(t_idx)), LD(fill_value(smin, smax)))
    bound = np.zeros(ref.shape)
    vt = (t_idx >= 0) & (t_idx + 1 < K)
    vf = f_idx >= 0
    if not vt.any() or not vf.any():
        return ref, bound
    r0 = np.searchsorted(R["frames"], t_idx[vt])[None, :]
    c0 = np.searchsorted(R["bins"], f_idx[vf])[:, None]
    LS, M, Ae = R["LS"], R["M"], R["Aeff"]
    wx = t_frac[vt].astype(LD)[None, :]
    wy = f_frac[vf].astype(LD)[:, None]
    s00, s01, s10, s11 = LS[r0, c0], LS[r0 + 1, c0], LS[r0, c0 + 1], LS[r0 + 1, c0 + 1]
    v = (1 - wy) * ((1 - wx) * s00 + wx * s01) + wy * ((1 - wx) * s10 + wx * s11)
    v = np.clip((v - LD(smin)) / (LD(smax) - LD(smin)), LD(0), LD(1))
    kappa = np.zeros(v.shape, LD)
    for r in (r0, r0 + 1):
        for cc in (c0, c0 + 1):
            kappa = np.maximum(kappa, Ae[r] / (M[r, cc] + EPS_LOG))
    ref[np.ix_(vf, vt)] = v
    bound[np.ix_(vf, vt)] = ((TAU * math.log2(N) * kappa + FLOOR) / abs(smax - smin)).astype(np.float64)
    return ref, bound


@functools.lru_cache(maxsize=None)
def reference(cid):
    b = build_case(cid)
    c = b["c"]
    seg = b["audio"][b["lo"]:b["lo"] + b["seg_len"]]
    return ld_needed(seg, c["N"], c["hop"], c["dc"], b["window"], b["scale"], b["K"], b["t_idx"], b["f_idx"])


def ld_output(cid, smin, smax):
    b = build_case(cid)
    return ld_interp(reference(cid), b["c"]["N"], b["K"], b["t_idx"], b["t_frac"], b["f_idx"], b["f_frac"],
                     smin, smax)


def oracle_params(c, n_f, n_t, smin, smax):
    return {'nperseg': c["N"], 'noverlap': c["N"] - c["hop"], 'spec_min_val': smin, 'spec_max_val': smax,
            'num_freq_bins': n_f, 'num_time_bins': n_t, 'max_dur': 1e9, 'mel': False, 'time_stretch': False,
            'within_syll_normalize': False}


# -------------------------------------------------------------- CPU self-check of the reference
@pytest.mark.parametrize("cid", CONFIG_IDS)
def test_reference_matches_scipy_and_oracle(cid):
    """The long-double reference against scipy.signal.stft (log magnitude of every needed frame and
    bin) and against spec_oracle.get_spec (the whole output, all three ranges), to 1e-10 plus the
    same kappa term: both are float64 FFTs, exact only where the log magnitude is well conditioned.
    float32 audio goes to both as float64, the kernel's documented semantics."""
    from scipy.signal import stft
    b, R = build_case(cid), reference(cid)
    c = b["c"]
    N = c["N"]
    seg = b["audio"][b["lo"]:b["lo"] + b["seg_len"]].astype(np.float64)
    if c["dc"]:
        seg = seg - np.mean(seg)
    _, _, Z = stft(seg, c["fs"], nperseg=N, noverlap=N - c["hop"])
    assert Z.shape == (N // 2 + 1, b["K"])
    if c["freqs"] == "lin0":
        assert (b["f_idx"][0], b["f_frac"][0]) == (0, 0.0)
        assert (b["f_idx"][-1], b["f_frac"][-1]) == (N // 2 - 1, 1.0)
    if c["times"] == "onframe":
        assert (b["t_frac"] == 0.0).any()
    if len(R["frames"]) and len(R["bins"]):
        ls = np.log(np.abs(Z[np.ix_(R["bins"], R["frames"])].T) + 1e-12)
        kap = (R["Aeff"][:, None] / (R["M"] + EPS_LOG)).astype(np.float64)
        err = np.abs(ls - R["LS"].astype(np.float64))
        assert (err <= 1e-10 + TAU * math.log2(N) * kap).all(), err.max()
        # the needed frames really are the ones scipy puts at the frame times
        assert np.all(R["frames"] < b["K"])
    audio64 = b["audio"].astype(np.float64)
    for smin, smax in RANGES:
        ref, bound = ld_output(cid, smin, smax)
        p = oracle_params(c, len(b["tf"]), len(b["tt"]), smin, smax)
        o, _ = spec_oracle.get_spec(b["t1"], b["t2"], audio64, p, fs=c["fs"], target_freqs=b["tf"],
                                    target_times=b["tt"], remove_dc_offset=c["dc"])
        err = np.abs(o - ref.astype(np.float64))
        assert (err <= 1e-10 + bound).all(), (smin, smax, err.max())


# ------------------------------------------------------------------------------- GPU plumbing
class Guarded:
    """A [shape] tensor of `dtype` inside GUARD words of NaN sentinel on each side, itself NaN."""

    def __init__(self, shape, dtype):
        n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size() // 4
        self.n = n
        self.raw = torch.full((2 * GUARD + n,), SENT, dtype=torch.int32, device="cuda")
        self.t = self.raw[GUARD:GUARD + n].view(dtype).view(shape)

    def guards_ok(self):
        return bool((self.raw[:GUARD] == SENT).all()) and bool((self.raw[GUARD + self.n:] == SENT).all())

    def untouched(self):
        return bool((self.raw == SENT).all())


class Launch:
    """Device copies of one batch's audio and tables; run() calls ava_b200_get_spec_batch."""

    def __init__(self, audio, seg_start, seg_len, N, hop, remove_dc, t_idx, t_frac, f_idx, f_frac, max_frames):
        audio = np.asarray(audio)
        self.is_f32 = IS_F32[audio.dtype]
        self.audio = dev(audio)
        self.seg_start = dev(np.asarray(seg_start, np.int64))
        self.seg_len = dev(np.asarray(seg_len, np.int32))
        self.n, self.n_t = t_idx.shape
        self.n_f = len(f_idx)
        self.N, self.hop, self.remove_dc = N, hop, int(remove_dc)
        win = pre._hann_window(N)
        self.window, self.scale = dev(win), float(1.0 / win.sum())
        self.t_idx, self.t_frac = dev(t_idx.astype(np.int32)), dev(t_frac)
        self.f_idx, self.f_frac = dev(f_idx.astype(np.int32)), dev(f_frac)
        self.max_frames = max_frames

    @classmethod
    def of_case(cls, b):
        c = b["c"]
        return cls(b["audio"], [b["lo"]], [b["seg_len"]], c["N"], c["hop"], c["dc"], b["t_idx"][None, :],
                   b["t_frac"][None, :], b["f_idx"], b["f_frac"], b["kmax"] + 1)

    def call(self, out_ptr, out64_ptr, smin, smax, max_frames=None, w0=0, n=None):
        """Windows [w0, w0 + n) of the batch (pointers into the same tables)."""
        n = self.n if n is None else n
        _lib.call("ava_b200_get_spec_batch", self.audio.data_ptr(), self.is_f32,
                  self.seg_start.data_ptr() + 8 * w0, self.seg_len.data_ptr() + 4 * w0, n, self.N,
                  self.N - self.hop, self.remove_dc, self.window.data_ptr(), self.scale,
                  self.t_idx.data_ptr() + 4 * w0 * self.n_t, self.t_frac.data_ptr() + 8 * w0 * self.n_t, self.n_t,
                  self.f_idx.data_ptr(), self.f_frac.data_ptr(), self.n_f,
                  self.max_frames if max_frames is None else max_frames, smin, smax, out_ptr, out64_ptr, stream())

    def run(self, smin, smax, want32=True, want64=True, max_frames=None):
        shape = (self.n, self.n_f, self.n_t)
        o32 = Guarded(shape, torch.float32) if want32 else None
        o64 = Guarded(shape, torch.float64) if want64 else None
        self.call(o32.t.data_ptr() if o32 else None, o64.t.data_ptr() if o64 else None, smin, smax, max_frames)
        torch.cuda.synchronize()
        for o in (o32, o64):
            if o is not None:
                assert o.guards_ok(), "write outside the output"
                assert not bool(torch.isnan(o.t).any()), "output element never written"
        return o32, o64


@pytest.fixture(scope="module")
def worst():
    """Worst err/bound ratio per nperseg over the file's get_spec tests, printed at the end."""
    table = {}
    yield table
    if table:
        name = torch.cuda.get_device_name(0) if torch.cuda.is_available() else "?"
        print("\nworst |got - ref| / bound per nperseg (%s):" % name)
        for N in sorted(table):
            print("  nperseg %4d: %.3g" % (N, table[N]))


def check_against_reference(cid, o64, smin, smax, worst, what=""):
    ref, bound = ld_output(cid, smin, smax)
    got = o64.t.cpu().numpy()[0]
    err = np.abs(got.astype(LD) - ref).astype(np.float64)
    exact = bound == 0
    assert (err[exact] == 0).all(), ("fill / exact cells differ", what, err[exact].max())
    ratio = float((err[~exact] / bound[~exact]).max()) if (~exact).any() else 0.0
    N = build_case(cid)["c"]["N"]
    worst[N] = max(worst.get(N, 0.0), ratio)
    bad = np.argwhere(err > bound)
    assert len(bad) == 0, ("outside the bound", what, smin, smax, ratio, bad[:5].tolist())
    return ratio


# ------------------------------------------------------------------------- get_spec, per config
@pytest.mark.gpu
@pytest.mark.parametrize("cid", CONFIG_IDS)
def test_get_spec_elementwise(cid, worst):
    """One window of configuration `cid` at three spec ranges: every element within the bound (the
    fill cells exact), written exactly once inside guard bands, out == out64 in float32, the same
    bits with one output only and when called again; and get_spec itself returns the same array."""
    b = build_case(cid)
    c = b["c"]
    L = Launch.of_case(b)
    ratios = []
    for smin, smax in RANGES:
        o32, o64 = L.run(smin, smax)
        assert torch.equal(o32.t, o64.t.float())
        ratios.append(check_against_reference(cid, o64, smin, smax, worst))
        a32, _ = L.run(smin, smax, want64=False)
        _, a64 = L.run(smin, smax, want32=False)
        r32, r64 = L.run(smin, smax)
        for x, y in ((a32, o32), (a64, o64), (r32, o32), (r64, o64)):
            assert torch.equal(x.t.view(torch.int32), y.t.view(torch.int32))
        if c["sig"] == "zeros":
            # an all-zero segment: every in-range cell is log(1e-12) normalised (exact when clipped)
            v = float(np.clip((np.log(1e-12) - smin) / (smax - smin), 0.0, 1.0))
            got = o64.t.cpu().numpy()[0]
            inr = np.ix_(b["f_idx"] >= 0, (b["t_idx"] >= 0) & (b["t_idx"] + 1 < b["K"]))
            tol = 0.0 if v in (0.0, 1.0) else FLOOR / abs(smax - smin)
            assert np.abs(got[inr] - v).max(initial=0.0) <= tol
    p = oracle_params(c, len(b["tf"]), len(b["tt"]), *WIDE)
    spec, _ = pre.get_spec(b["t1"], b["t2"], b["audio"], p, fs=c["fs"], target_freqs=b["tf"],
                           target_times=b["tt"], remove_dc_offset=c["dc"])
    o32, o64 = L.run(*WIDE)
    assert np.array_equal(spec, o64.t.cpu().numpy()[0])
    print("%s: worst err/bound %s" % (cid, " ".join("%.3g" % r for r in ratios)))


@pytest.mark.gpu
def test_get_spec_larger_max_frames_changes_runs_not_result(worst):
    """A larger max_frames shrinks the slot count CF (more, shorter runs; a different pairing of
    frames into packed FFTs): still within the bound, out == out64 in float32."""
    cid = next(k for k, c in CONFIGS.items() if c["N"] == 512 and c["n_t"] >= 300 and c["times"] in ("lin", "rand"))
    b = build_case(cid)
    L = Launch.of_case(b)
    for extra in (0, 3000, 20000):
        for smin, smax in (WIDE, PROD):
            o32, o64 = L.run(smin, smax, max_frames=b["kmax"] + 1 + extra)
            assert torch.equal(o32.t, o64.t.float())
            check_against_reference(cid, o64, smin, smax, worst, "max_frames +%d" % extra)


def spec_smem(N, max_frames, n_f):
    """The launcher's shared-memory size (csrc/spec.cu, ava_b200_get_spec_batch)."""
    G = min(8, max(1, 2048 // N))
    NBP = N // 2 + 2
    fixed = G * N * 16 + N * 16 + 64 + 2 * (max_frames + 1) * 4 + 16 + (n_f + 2) * 12 + 16
    cf = (96 * 1024 - fixed) // (NBP * 8) if fixed < 96 * 1024 else 0
    cf = max(2, min(max(cf, 4), max_frames + 1))
    return -(-(fixed + cf * NBP * 8) // 16) * 16


@pytest.mark.gpu
def test_get_spec_largest_max_frames_at_4096(worst):
    """nperseg 4096: the largest max_frames whose shared memory fits runs a window of max_frames - 1
    frames within the bound; one frame more, and 10000, are rejected with nothing written."""
    N, hop, fs, n_f = 4096, 1024, 250000, 128
    mf = 10000
    while spec_smem(N, mf, n_f) > SMEM_LIMIT:
        mf -= 1
    assert spec_smem(N, 10000, n_f) > 270 * 1024
    rng = np.random.default_rng(5)
    seg_n = (mf - 2) * hop
    audio = to_dtype(spec_oracle.synth_audio(77, seg_n, fs, dtype=np.float64), np.int16)
    K = int(pre.num_frames(seg_n, N, hop))
    assert K == mf - 1
    base = (np.arange(N / 2, N / 2 + K * hop, hop) / float(fs)) - (N / 2) / fs
    tt = np.sort(np.concatenate([rng.uniform(0, 0.2, 12), rng.uniform(base[K - 1] - 0.1, base[K - 1], 12),
                                 rng.uniform(0, base[K - 1], 8)]))
    t_idx, t_frac = pre.bracket(np.zeros(1), base, np.array([K]), tt[None, :])
    fgrid = np.fft.rfftfreq(N, 1 / fs)
    f_idx, f_frac = pre.bracket_1d(fgrid, np.linspace(0.0, fgrid[-1], n_f))
    assert (t_idx >= 0).all() and (f_idx >= 0).all()
    L = Launch(audio, [0], [seg_n], N, hop, True, t_idx, t_frac, f_idx, f_frac, mf)
    o32, o64 = L.run(*WIDE)
    R = ld_needed(audio, N, hop, True, pre._hann_window(N), L.scale, K, t_idx[0], f_idx)
    ref, bound = ld_interp(R, N, K, t_idx[0], t_frac[0], f_idx, f_frac, *WIDE)
    err = np.abs(o64.t.cpu().numpy()[0].astype(LD) - ref).astype(np.float64)
    assert (err <= bound).all(), (err / bound).max()
    worst[N] = max(worst.get(N, 0.0), float((err / bound).max()))
    for bad in (mf + 1, 10000):
        o = Guarded((1, n_f, len(tt)), torch.float32)
        n0 = _lib.launch_count()
        with pytest.raises(_lib.AvaB200Error, match="shared memory"):
            L.call(o.t.data_ptr(), None, *WIDE, max_frames=bad)
        torch.cuda.synchronize()
        assert o.untouched() and _lib.launch_count() == n0


# --------------------------------------------------------------------- batch of mixed windows
@pytest.mark.gpu
def test_get_spec_batch_of_2048_mixed_windows():
    """2048 windows at nperseg 512 over three files in one launch (several waves over the SMs):
    segment lengths 0, < nperseg (zeros), exactly nperseg and long.  Each window matches
    spec_oracle at 1e-9 and is bit-identical to the same window run as a batch of one with the same
    max_frames."""
    p = dict(spec_oracle.FINCH_P)
    fs, N, hop = p['fs'], p['nperseg'], p['nperseg'] - p['noverlap']
    audio = [spec_oracle.synth_audio(40 + i, int((1.0 + 0.5 * i) * fs), fs) for i in range(3)]
    lengths = np.array([len(a) for a in audio])
    offsets = np.concatenate([[0], np.cumsum(lengths)[:-1]])
    n = 2048
    rng = np.random.default_rng(21)
    files = rng.integers(0, 3, n)
    kind = np.arange(n) % 8
    t1 = rng.uniform(-0.05, lengths[files] / fs - 0.05)
    dur = rng.uniform(0.02, 0.4, n)
    s1 = rng.integers(0, lengths[files] - N)
    t1 = np.where(kind == 1, s1 / fs, t1)                                   # exactly nperseg samples
    dur = np.where(kind == 1, N / fs, dur)
    dur = np.where(kind == 2, 300 / fs, dur)                                # shorter than nperseg
    t1 = np.where(kind == 3, -0.5, t1)                                      # ends before the file
    dur = np.where(kind == 3, 0.3, dur)
    t1 = np.where(kind == 4, lengths[files] / fs + 0.01, t1)                # starts after its end
    t2 = t1 + dur
    n_t = 128
    tt = np.linspace(t1 - 0.01, t2 + 0.01, n_t, axis=-1)
    segs = [segment_tables(N, hop, fs, lengths[f], a, z) for f, a, z in zip(files, t1, t2)]
    lo = np.array([s[0] for s in segs])
    seg_len = np.array([s[1] for s in segs])
    K = np.array([s[2] for s in segs])
    kmax = int(K.max())
    base = (np.arange(N / 2, N / 2 + kmax * hop, hop) / float(fs)) - (N / 2) / fs
    t_idx, t_frac = pre.bracket(np.maximum(0.0, t1), base, K, tt)
    f_idx, f_frac = pre.bracket_1d(np.fft.rfftfreq(N, 1 / fs), pre.target_freqs_for(p))
    assert (seg_len == 0).sum() >= 3 * n // 8 and (seg_len == N).sum() >= n // 8 - 2
    L = Launch(np.concatenate(audio), offsets[files] + lo, seg_len, N, hop, True, t_idx, t_frac, f_idx, f_frac,
               kmax + 1)
    smin, smax = p['spec_min_val'], p['spec_max_val']
    o32, o64 = L.run(smin, smax)
    assert torch.equal(o32.t, o64.t.float())
    one = torch.full((n, 128, n_t), float("nan"), dtype=torch.float64, device="cuda")
    for i in range(n):
        L.call(None, one.data_ptr() + 8 * i * 128 * n_t, smin, smax, w0=i, n=1)
    torch.cuda.synchronize()
    assert torch.equal(one.view(torch.int64), o64.t.view(torch.int64))
    got = o64.t.cpu().numpy()
    for i in range(n):
        ref, _ = spec_oracle.get_spec(t1[i], t2[i], audio[files[i]], p, fs=fs, target_times=tt[i])
        assert np.abs(got[i] - ref).max() <= 1e-9, i
        if seg_len[i] == 0:
            assert not got[i].any()


# ----------------------------------------------------------------------- quantile normalisation
Q_VALUES = (0.0, 1.0, 0.5, 0.25, 1 / 3, 0.9, 0.999, 1e-9, 1 - 2.0 ** -53)
M_ROWS = ((2, 4096), (3, 4096), (5, 4096), (127, 4096), (16384, 256), (16512, 128), (24576, 96))


def quantile_rows(n, m, seed):
    """Rows in [0, 1] with heavy ties: half exact zeros, a few ones, a 2^-8 grid and some -0.0;
    continuous rows; all-zero, one-non-zero, all-equal and two-valued rows."""
    rng = np.random.default_rng(seed)
    X = np.empty((n, m))
    for r in range(n):
        k = r % 8
        if k <= 2:
            v = rng.integers(0, 257, m) / 256.0
            v[rng.random(m) < 0.5] = 0.0
            v[rng.integers(0, m, max(1, m // 50))] = 1.0
        elif k == 3:
            v = rng.random(m)
            v[rng.random(m) < 0.2] = 0.0
        elif k == 4:
            v = np.zeros(m)
        elif k == 5:
            v = np.zeros(m)
            v[rng.integers(0, m)] = rng.random()
        elif k == 6:
            v = np.full(m, 0.37)
        else:
            v = np.where(rng.random(m) < 0.5, 0.25, 0.75)
        if k in (0, 1, 3, 4):
            v[np.flatnonzero(v == 0.0)[::2]] = -0.0
        X[r] = v
    return X


def numpy_normalize(X, q):
    """numpy's within_syll_normalize, row by row, with zeros made +0.0: numpy keeps a -0.0 where the
    input had one and the quantile is 0, the kernel documents that its zeros are +0.0."""
    s = X.copy()
    s -= np.quantile(s, q, axis=1, keepdims=True)
    s[s < 0.0] = 0.0
    s /= s.max(axis=1, keepdims=True) + 1e-12
    return s + 0.0


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.int64 if a.dtype == np.float64 else np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", M_ROWS)
def test_quantile_normalize_bit_exact(m, n):
    """within_syll_normalize on the device equals numpy's float64 expression bit for bit, every
    zero +0.0, and spec32 is its float32 cast, for every q in Q_VALUES."""
    X = quantile_rows(n, m, seed=m)
    assert (np.signbit(X) & (X == 0)).any()
    Xd = dev(X)
    for q in Q_VALUES:
        s64 = Xd.clone()
        s32 = Guarded((n, m), torch.float32)
        _lib.call("ava_b200_quantile_normalize", s64.data_ptr(), s32.t.data_ptr(), n, m, q, stream())
        torch.cuda.synchronize()
        assert s32.guards_ok()
        exp = numpy_normalize(X, q)
        got = s64.cpu().numpy()
        bad = np.flatnonzero((bits(got) != bits(exp)).any(axis=1))
        assert len(bad) == 0, (q, len(bad), bad[:8].tolist())
        assert np.array_equal(bits(s32.t.cpu().numpy()), bits(exp.astype(np.float32))), q


@pytest.mark.gpu
def test_within_syll_normalize_through_spec_engine():
    """SpecEngine with within_syll_normalize at 128 x 192: the normalised float64 and float32 outputs
    equal numpy's normalisation of the same engine's unnormalised spectrograms, bit for bit."""
    fs = 32000
    p = dict(spec_oracle.FINCH_P, within_syll_normalize=True, normalize_quantile=0.37)
    audio = [spec_oracle.synth_audio(60 + i, int(1.5 * fs), fs) for i in range(2)]
    eng_n = pre.SpecEngine(audio, fs, p)
    eng_r = pre.SpecEngine(audio, fs, dict(p, within_syll_normalize=False))
    rng = np.random.default_rng(8)
    n = 33
    files = rng.integers(0, 2, n)
    on = rng.uniform(0.0, 1.3, n)
    t1, t2 = np.maximum(0.0, on - 0.05), on + 0.17
    tt = np.linspace(on, on + 0.12, 192, axis=-1)
    a32, a64 = eng_n.specs(files, t1, t2, tt, want_float64=True)
    _, r64 = eng_r.specs(files, t1, t2, tt, want_float64=True)
    torch.cuda.synchronize()
    raw = r64.cpu().numpy().reshape(n, -1)
    exp = numpy_normalize(raw, 0.37).reshape(n, 128, 192)
    assert np.array_equal(bits(a64.cpu().numpy()), bits(exp))
    assert np.array_equal(bits(a32.cpu().numpy()), bits(exp.astype(np.float32)))


# --------------------------------------------------------------------------- time tables
@pytest.mark.gpu
@pytest.mark.parametrize("N", (16, 512, 4096))
def test_window_time_tables_bit_exact(N):
    """ava_b200_window_time_tables against the host bracket, bit for bit: every hop and sample rate,
    n_t 2 to 300, windows of K = 3 frames, at the file start and running past its end."""
    rng = np.random.default_rng(N)
    for hop in (N // 2, N // 4, N, N // 2 + 3):
        for fs in FSS:
            flen = max(20 * N, fs // 2)
            n = 97
            wl = rng.uniform(N / fs, 40 * hop / fs, n)
            on = rng.uniform(-0.05, flen / fs, n)
            on[0] = 0.0
            on[1] = (flen - N // 2) / fs                     # runs past the end of the file
            t1, t2 = np.maximum(0.0, on), on + wl
            t2[2] = t1[2] + N / fs                           # exactly nperseg samples
            t2[3] = t1[3] + (N // 2) / fs                    # too short: K = 3
            segs = [segment_tables(N, hop, fs, flen, a, z) for a, z in zip(t1, t2)]
            K = np.array([s[2] for s in segs])
            kmax = int(K.max())
            base = (np.arange(N / 2, N / 2 + kmax * hop, hop) / float(fs)) - (N / 2) / fs
            assert (K == 3).any()
            for n_t in (2, 3, 127, 129, 300):
                tt = np.linspace(on, on + wl, n_t, axis=-1).reshape(n, n_t)
                t_idx, t_frac = pre.bracket(t1, base, K, tt)
                ti = Guarded((n, n_t), torch.int32)
                tf = Guarded((n, n_t), torch.float64)
                g0, Kd, bd, ts, te = dev(t1), dev(K.astype(np.int32)), dev(base), dev(on), dev(on + wl)
                _lib.call("ava_b200_window_time_tables", g0.data_ptr(), Kd.data_ptr(), bd.data_ptr(), kmax,
                          ts.data_ptr(), te.data_ptr(), n, n_t, ti.t.data_ptr(), tf.t.data_ptr(), stream())
                torch.cuda.synchronize()
                assert ti.guards_ok() and tf.guards_ok()
                np.testing.assert_array_equal(ti.t.cpu().numpy(), t_idx)
                assert np.array_equal(tf.t.cpu().numpy().view(np.int64), t_frac.view(np.int64)), (hop, fs, n_t)
                assert (t_idx < 0).any() and (t_idx >= 0).any()


# ------------------------------------------------------------------------------ rejections
def _expect_rejected(name, args, outs, match):
    n0 = _lib.launch_count()
    with pytest.raises(_lib.AvaB200Error, match=match) as e:
        _lib.call(name, *args)
    torch.cuda.synchronize()
    assert str(e.value).split("failed: ", 1)[1].strip()
    assert _lib.launch_count() == n0
    for o in outs:
        assert o.untouched()


@pytest.mark.gpu
def test_get_spec_rejections():
    """Bad nperseg, noverlap, spec range, sample type, shape or outputs raise AvaB200Error with a
    message, launch nothing and leave the NaN outputs as they were; n = 0 launches nothing."""
    b = build_case(CONFIG_IDS[0])
    L = Launch.of_case(b)
    o32 = Guarded((1, L.n_f, L.n_t), torch.float32)
    o64 = Guarded((1, L.n_f, L.n_t), torch.float64)

    def args(**kw):
        a = dict(audio=L.audio.data_ptr(), is_f32=L.is_f32, seg_start=L.seg_start.data_ptr(),
                 seg_len=L.seg_len.data_ptr(), n=1, nperseg=L.N, noverlap=L.N - L.hop, remove_dc=1,
                 window=L.window.data_ptr(), scale=L.scale, t_idx=L.t_idx.data_ptr(), t_frac=L.t_frac.data_ptr(),
                 n_t=L.n_t, f_idx=L.f_idx.data_ptr(), f_frac=L.f_frac.data_ptr(), n_f=L.n_f,
                 max_frames=L.max_frames, smin=2.0, smax=6.5, out=o32.t.data_ptr(), out64=o64.t.data_ptr(),
                 stream=stream())
        a.update(kw)
        return list(a.values())

    bad = [(dict(nperseg=8), "nperseg"), (dict(nperseg=8192), "nperseg"), (dict(nperseg=1000), "nperseg"),
           (dict(noverlap=L.N), "noverlap"), (dict(noverlap=-1), "noverlap"), (dict(smax=2.0), "spec_max"),
           (dict(is_f32=3), "sample type"), (dict(is_f32=-1), "sample type"), (dict(n_f=0), "n_f"),
           (dict(n_t=0), "n_t"), (dict(out=None, out64=None), "no output"),
           (dict(nperseg=4096, noverlap=2048, max_frames=10000), "shared memory")]
    for kw, match in bad:
        _expect_rejected("ava_b200_get_spec_batch", args(**kw), (o32, o64), match)
    n0 = _lib.launch_count()
    _lib.call("ava_b200_get_spec_batch", *args(n=0))
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0 and o32.untouched() and o64.untouched()
    _lib.call("ava_b200_get_spec_batch", *args())
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0 + 1 and not bool(torch.isnan(o64.t).any())


@pytest.mark.gpu
def test_quantile_and_time_table_rejections():
    s64 = Guarded((4, 24577), torch.float64)
    s32 = Guarded((4, 24577), torch.float32)
    for m, q, match in ((1, 0.5, "m=1"), (24577, 0.5, "m=24577"), (100, -0.01, "outside"), (100, 1.01, "outside")):
        _expect_rejected("ava_b200_quantile_normalize", (s64.t.data_ptr(), s32.t.data_ptr(), 4, m, q, stream()),
                         (s64, s32), match)
    n0 = _lib.launch_count()
    _lib.call("ava_b200_quantile_normalize", s64.t.data_ptr(), s32.t.data_ptr(), 0, 100, 0.5, stream())
    assert _lib.launch_count() == n0 and s64.untouched() and s32.untouched()
    g0, K = dev(np.zeros(2)), dev(np.array([3, 3], np.int32))
    base = dev(np.arange(4) * 0.01)
    ts, te = dev(np.array([0.0, 0.01])), dev(np.array([0.02, 0.03]))
    ti = Guarded((2, 8), torch.int32)
    tf = Guarded((2, 8), torch.float64)
    for kmax, n_t in ((2, 8), (4, 1)):
        _expect_rejected("ava_b200_window_time_tables",
                         (g0.data_ptr(), K.data_ptr(), base.data_ptr(), kmax, ts.data_ptr(), te.data_ptr(), 2, n_t,
                          ti.t.data_ptr(), tf.t.data_ptr(), stream()), (ti, tf), "window_time_tables")
    _lib.call("ava_b200_window_time_tables", g0.data_ptr(), K.data_ptr(), base.data_ptr(), 4, ts.data_ptr(),
              te.data_ptr(), 0, 8, ti.t.data_ptr(), tf.t.data_ptr(), stream())
    assert _lib.launch_count() == n0 and ti.untouched() and tf.untouched()
