"""
TEST INFRASTRUCTURE ONLY -- golden-vector generator.

Runs the UNMODIFIED reference (imported from /root/reference through
oracle/_ref_import.py) on seeded synthetic inputs and writes small fixtures to
tests/golden/.  Run in the build container only:

    python -m oracle.make_golden

Versions the goldens were produced with are stored in each file's `versions` field.
Inputs/weights are regenerated from seeds by oracle.vae_oracle.make_* so they are
not stored.  Large tensors (fc1/fc8 weight grads, x_rec at B=64) are stored as a
digest: (sum, L2 norm, values at 4096 seeded indices).
"""
import copy
import importlib
import json
import os
import sys
import tempfile

import numpy as np
import scipy
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import _ref_import, spec_oracle, vae_oracle  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
FULL_LIMIT = 20000
N_DIGEST = 4096


def versions():
    return "torch=%s numpy=%s scipy=%s" % (torch.__version__, np.__version__,
                                           scipy.__version__)


def digest_indices(numel, salt=0):
    rng = np.random.default_rng(77 + salt)
    return rng.integers(0, numel, size=N_DIGEST)


def digest(a, salt=0):
    a = np.asarray(a, dtype=np.float64).ravel()
    idx = digest_indices(a.size, salt)
    return np.concatenate([[a.sum(), np.sqrt((a * a).sum())], a[idx]])


def store(out, key, arr):
    arr = np.asarray(arr)
    if arr.size <= FULL_LIMIT:
        out[key] = arr
    else:
        out[key + "__digest"] = digest(arr)


def load_into_reference(model, P):
    sd = model.state_dict()
    for k in sd:
        sd[k] = P[k].clone()
    model.load_state_dict(sd)


class _InjectNoise:
    """Feeds prepared (eps_W, eps_D) to LowRankMultivariateNormal.rsample by
    replacing torch's `_standard_normal` helper in that module (torch internal;
    the reference's own code stays unmodified)."""

    def __init__(self, tensors):
        import torch.distributions.lowrank_multivariate_normal as lr
        self.lr = lr
        self.queue = list(tensors)

    def __enter__(self):
        self.orig = self.lr._standard_normal

        def fake(shape, dtype, device):
            t = self.queue.pop(0)
            assert tuple(t.shape) == tuple(shape), (t.shape, shape)
            return t.to(dtype)
        self.lr._standard_normal = fake
        return self

    def __exit__(self, *a):
        self.lr._standard_normal = self.orig


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    den = np.abs(b).max()
    return np.abs(a - b).max() / den if den > 0 else np.abs(a).max()


def vae_case(ref_vae, name, seed, batch, train, prec=10.0):
    """Reference run twice on identical weights/inputs/noise: its stock fp32 path
    (noise drawn by the reference itself under torch.manual_seed) and the same
    unmodified code in float64 (`.double()`, noise injected) as the exact
    answer.  Stored: the float64 results, and for each tensor the relative
    error of the reference's own fp32 result against it (`err32:*`)."""
    P = vae_oracle.make_params(seed)
    x = vae_oracle.make_input(seed, batch)
    out = {"versions": np.array(versions()), "seed": seed, "batch": batch,
           "train": int(train), "model_precision": prec}
    # The noise the reference draws (eps_W first, then eps_D; SURVEY a5).
    torch.manual_seed(seed)
    eps_w = torch.randn(batch, 1)
    eps_d = torch.randn(batch, 32)
    out["eps_w"] = eps_w.numpy()
    out["eps_d"] = eps_d.numpy()

    def run(dtype, inject):
        model = ref_vae.VAE(save_dir='', model_precision=prec, device_name='cpu')
        load_into_reference(model, P)
        model.to(dtype)
        model.train(train)
        xx = x.to(dtype)
        res = {}
        m2 = copy.deepcopy(model)
        with torch.no_grad():
            mu, u, d = m2.encode(xx)
        res["mu"], res["u"], res["d"] = mu.numpy(), u.numpy(), d.numpy()
        m3 = copy.deepcopy(model)
        torch.manual_seed(seed)
        with torch.no_grad():
            if inject:
                with _InjectNoise([eps_w, eps_d]):
                    _, z, x_rec = m3.forward(xx, return_latent_rec=True)
            else:
                _, z, x_rec = m3.forward(xx, return_latent_rec=True)
        res["z"], res["x_rec"] = z, x_rec
        # forward + backward exactly as train_epoch does (vae.py:348-352).
        torch.manual_seed(seed)
        model.optimizer.zero_grad()
        if inject:
            with _InjectNoise([eps_w, eps_d]):
                loss = model.forward(xx)
        else:
            loss = model.forward(xx)
        res["loss"] = np.array(loss.item(), dtype=np.float64)
        loss.backward()
        for k, p in model.named_parameters():
            res["grad:" + k] = p.grad.numpy().copy()
        for k, b in model.named_buffers():
            res["buf:" + k] = b.numpy().copy()
        return res

    r32 = run(torch.float32, inject=False)
    r64 = run(torch.float64, inject=True)
    for k, v in r64.items():
        store(out, k, v)
        if k.startswith("buf:") and k.endswith("tracked"):
            continue
        out["err32:" + k] = np.array(rel_err(r32[k], v))
    out["loss32"] = r32["loss"]
    np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), **out)
    worst = max(float(out[k]) for k in out if k.startswith("err32:grad"))
    print(name, "loss64", float(r64["loss"]), "loss32", float(r32["loss"]),
          "worst fp32-reference grad err vs fp64: %.2e" % worst)


def adam_case(ref_vae, name, seed, batch, steps):
    """`steps` reference train steps (vae.py:348-353) in float64 (truth) and in
    the stock fp32 path; noise injected so both see identical draws."""
    P = vae_oracle.make_params(seed)
    out = {"versions": np.array(versions()), "seed": seed, "batch": batch,
           "steps": steps}

    def run(dtype):
        model = ref_vae.VAE(save_dir='', device_name='cpu')
        load_into_reference(model, P)
        model.to(dtype)
        model.train()
        losses = []
        for s in range(steps):
            x = vae_oracle.make_input(seed + s, batch).to(dtype)
            ew, ed = vae_oracle.make_noise(seed + s, batch)
            model.optimizer.zero_grad()
            with _InjectNoise([ew, ed]):
                loss = model.forward(x)
            losses.append(loss.item())
            loss.backward()
            model.optimizer.step()
        res = {"losses": np.array(losses, dtype=np.float64)}
        for k, p in model.named_parameters():
            res["param:" + k] = p.detach().numpy().copy()
        for k, b in model.named_buffers():
            res["buf:" + k] = b.numpy().copy()
        return res

    r32, r64 = run(torch.float32), run(torch.float64)
    for k, v in r64.items():
        store(out, k, v)
        if k.startswith("buf:") and k.endswith("tracked"):
            continue
        out["err32:" + k] = np.array(rel_err(r32[k], v))
    np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), **out)
    print(name, "losses", r64["losses"], r32["losses"])


def spec_cases(ref_pre):
    out = {"versions": np.array(versions())}
    # --- mouse-syllable params (time stretch, linear freqs), int16 @ 250 kHz
    p = dict(spec_oracle.MOUSE_P)
    fs = p['fs']
    audio = spec_oracle.synth_audio(11, int(0.6 * fs), fs)
    cases = [
        ("mouse_a", 0.100, 0.180), ("mouse_b", 0.2503, 0.2871),
        ("mouse_full", 0.30, 0.50),          # duration == max_dur
        ("mouse_neg", -0.02, 0.05),          # s1 < 0
        ("mouse_end", 0.55, 0.62),           # s2 > len(audio)
        ("mouse_short", 0.4000, 0.4030),     # < nperseg samples -> zeros
    ]
    for name, t1, t2 in cases:
        spec, flag = ref_pre.get_spec(t1, t2, audio, p, fs=fs)
        assert flag
        out[name] = spec
        out[name + "_t"] = np.array([t1, t2])
    # --- finch window params (mel), explicit target_times, int16 @ 32 kHz
    p = dict(spec_oracle.FINCH_P)
    fs = p['fs']
    audio2 = spec_oracle.synth_audio(12, int(4.0 * fs), fs)
    for name, onset in [("finch_a", 1.2345), ("finch_b", 0.01), ("finch_c", 3.87),
                        ("finch_d", 2.000004)]:
        offset = onset + p['window_length']
        tt = np.linspace(onset, offset, 128)
        spec, _ = ref_pre.get_spec(max(0.0, onset - 0.05), offset + 0.05, audio2,
                                   p, fs=fs, target_times=tt)
        out[name] = spec
        out[name + "_t"] = np.array([onset])
    # --- float32 audio, non-mel, no DC removal, non-50% overlap
    p3 = dict(spec_oracle.FINCH_P)
    p3.update(mel=False, noverlap=384, max_dur=0.3, time_stretch=True)
    audio3 = (spec_oracle.synth_audio(13, int(2.0 * fs), fs, dtype=np.float64)
              / 3.0).astype(np.float32)
    spec, _ = ref_pre.get_spec(0.5, 0.7, audio3, p3, fs=fs, remove_dc_offset=False)
    out["f32_a"] = spec
    np.savez_compressed(os.path.join(GOLDEN, "spec_cases.npz"), **out)
    print("spec cases:", [k for k in out if not k.endswith("_t")])


def sampler_cases(ref_win, ref_ds, ref_pre):
    from scipy.io import wavfile
    out = {"versions": np.array(versions())}
    p = dict(spec_oracle.FINCH_P)
    p['get_spec'] = ref_pre.get_spec
    fs = p['fs']
    with tempfile.TemporaryDirectory() as tmp:
        adir, rdir = os.path.join(tmp, "audio"), os.path.join(tmp, "rois")
        os.mkdir(adir)
        os.mkdir(rdir)
        names = ["b_song", "a_song", "d_song", "c_song", "e_song"]
        rng = np.random.default_rng(5)
        for i, nm in enumerate(names):
            audio = spec_oracle.synth_audio(100 + i, int(3.0 * fs), fs)
            wavfile.write(os.path.join(adir, nm + ".wav"), fs, audio)
            n_roi = 1 + (i % 3)
            starts = np.sort(rng.uniform(0.1, 2.0, size=n_roi))
            rois = np.stack([starts, starts + rng.uniform(0.2, 0.8, size=n_roi)], 1)
            np.savetxt(os.path.join(rdir, nm + ".txt"), rois)
        part = ref_win.get_window_partition([adir], [rdir], split=0.8)
        out["part_train_audio"] = np.array(
            [os.path.basename(s) for s in part['train']['audio']])
        out["part_train_rois"] = np.array(
            [os.path.basename(s) for s in part['train']['rois']])
        out["part_test_audio"] = np.array(
            [os.path.basename(s) for s in part['test']['audio']])
        part1 = ref_win.get_window_partition([adir], [rdir], split=1.0)
        out["part1_audio"] = np.array(
            [os.path.basename(s) for s in part1['train']['audio']])
        out["part1_rois"] = np.array(
            [os.path.basename(s) for s in part1['train']['rois']])
        ds = ref_win.FixedWindowDataset(part1['train']['audio'],
                                        part1['train']['rois'], p,
                                        transform=None)
        out["file_weights"] = ds.file_weights
        for seed in (0, 1, 7):
            specs, fidx, onsets, offsets = ds.__getitem__(
                np.arange(12), seed=seed, return_seg_info=True)
            out["seed%d_files" % seed] = np.array(fidx, dtype=np.int64)
            out["seed%d_onsets" % seed] = np.array(onsets, dtype=np.float64)
            out["seed%d_offsets" % seed] = np.array(offsets, dtype=np.float64)
            if seed == 0:
                out["seed0_specs"] = np.stack(specs[:3]).astype(np.float64)
        # syllable partition: only file listing + seed-42 shuffle matter.
        hdir = os.path.join(tmp, "h5")
        os.mkdir(hdir)
        for i in range(13):
            open(os.path.join(hdir, "syllables_%04d.hdf5" % i), "w").close()
        open(os.path.join(hdir, "notes.txt"), "w").close()
        sp = ref_ds.get_syllable_partition([hdir], 0.75)
        out["syll_train"] = np.array([os.path.basename(s) for s in sp['train']])
        out["syll_test"] = np.array([os.path.basename(s) for s in sp['test']])
        sp2 = ref_ds.get_syllable_partition([hdir], 1.0, shuffle=False,
                                            max_num_files=5)
        out["syll2_train"] = np.array([os.path.basename(s) for s in sp2['train']])
    np.savez_compressed(os.path.join(GOLDEN, "sampler_cases.npz"), **out)
    print("sampler cases ok")


class _FakeH5File:
    """Stand-in for h5py.File("...", "w") that records create_dataset calls (h5py is not
    installed here; the reference's process_sylls only uses this much of it)."""
    written = {}

    def __init__(self, filename, mode="r"):
        self.filename = filename
        self.data = {}

    def __enter__(self):
        return self

    def __exit__(self, *a):
        _FakeH5File.written[os.path.basename(self.filename)] = self.data

    def create_dataset(self, key, data=None):
        self.data[key] = np.asarray(data)


PROCESS_P = dict(spec_oracle.FINCH_P)
PROCESS_P.update(max_dur=0.2, time_stretch=True, sylls_per_file=4, max_num_syllables=None)


def write_process_corpus(root):
    """Two synthetic int16 wav files + segment files (shared by the generator and the test)."""
    from scipy.io import wavfile
    adir, sdir = os.path.join(root, "audio"), os.path.join(root, "segs")
    os.makedirs(adir, exist_ok=True)
    os.makedirs(sdir, exist_ok=True)
    fs = PROCESS_P['fs']
    segs = {
        "a.wav": [(0.10, 0.18), (0.30, 0.45), (0.600, 0.6100), (0.95, 1.10)],   # 3rd: < nperseg samples
        "b.wav": [(0.05, 0.20), (0.50, 0.56), (1.42, 1.52), (0.80, 0.93), (1.10, 1.21)],  # 3rd runs off the end
    }
    for k, (name, sg) in enumerate(segs.items()):
        wavfile.write(os.path.join(adir, name), fs, spec_oracle.synth_audio(21 + k, int(1.5 * fs), fs))
        np.savetxt(os.path.join(sdir, name[:-4] + ".txt"), np.array(sg), header="onset offset")
    return adir, sdir


def process_case(ref_pre):
    import tempfile
    _ref_import.install_stubs()
    import ava.preprocessing.preprocess as ref_pp
    ref_pp.h5py.File = _FakeH5File
    _FakeH5File.written = {}
    p = dict(PROCESS_P)
    p['get_spec'] = ref_pre.get_spec
    with tempfile.TemporaryDirectory() as root:
        adir, sdir = write_process_corpus(root)
        ref_pp.process_sylls(adir, sdir, os.path.join(root, "out"), p, shuffle=True, verbose=False)
    out = {"versions": np.array(versions())}
    for fn, d in sorted(_FakeH5File.written.items()):
        for key, v in d.items():
            if key == 'audio_filenames':
                v = np.array([os.path.basename(i.decode()) for i in v]).astype('S')
            out[fn + ":" + key] = v
    np.savez_compressed(os.path.join(GOLDEN, "process_sylls.npz"), **out)
    print("process_sylls files:", sorted(_FakeH5File.written))


def mmd_latent(seed=31):
    rng = np.random.default_rng(seed)
    sizes, shifts = (120, 150, 130), (0.0, 0.35, -0.5)
    latent = np.concatenate([rng.standard_normal((n, 32)) + s for n, s in zip(sizes, shifts)])
    condition = np.concatenate([np.full(n, 10 * (k + 1)) for k, n in enumerate(sizes)])
    perm = rng.permutation(len(latent))
    return latent[perm], condition[perm]


def mmd_case():
    _ref_import.install_stubs()
    import types
    for name, attrs in (("matplotlib.collections", {"PolyCollection": None}),
                        ("matplotlib.colors", {"cnames": {}, "to_rgba": None})):
        if name not in sys.modules:
            m = types.ModuleType(name)
            for k, v in attrs.items():
                setattr(m, k, v)
            sys.modules[name] = m
    import ava.plotting.mmd_plots as ref_mmd
    latent, condition = mmd_latent()
    out = {"versions": np.array(versions())}
    sigma = ref_mmd.estimate_median_sigma(latent)
    out["sigma"] = np.array(sigma)
    conds = np.unique(condition)
    groups = [np.argwhere(condition == c).flatten() for c in conds]
    m = np.zeros((3, 3))
    lin = np.zeros((3, 3))
    sub = np.zeros((3, 3))
    for i in range(2):
        for j in range(i + 1, 3):
            m[i, j] = m[j, i] = ref_mmd._estimate_mmd2(latent, groups[i], groups[j], sigma=sigma)
            lin[i, j] = lin[j, i] = ref_mmd._estimate_mmd2_linear_time(latent, groups[i], groups[j], sigma=sigma)
            sub[i, j] = sub[j, i] = ref_mmd._estimate_mmd2(latent, groups[i].copy(), groups[j].copy(),
                                                           sigma=sigma, max_n=64, seed=5)
    out["mmd2"], out["mmd2_linear"], out["mmd2_max64_seed5"] = m, lin, sub
    out["sigma_n500_seed7"] = np.array(ref_mmd.estimate_median_sigma(latent, n=500, seed=7))
    np.savez_compressed(os.path.join(GOLDEN, "mmd_cases.npz"), **out)
    print("mmd cases: sigma", sigma, "mmd2", m[0, 1], m[0, 2], m[1, 2])


# ---------------------------------------------------------------- SURVEY 8(f) N1
class _MemH5File:
    """In-memory stand-in for h5py.File (h5py is not installed here): datasets live in a
    process-global store keyed by path; an empty file of the same name is kept on disk so
    that os.listdir-based discovery (get_hdf5s_from_dir) works.  Covers what the reference's
    DataContainer / SyllableDataset use: open modes r/a/w, f[key], key in f, f.keys(),
    create_dataset."""
    store = {}

    def __init__(self, filename, mode="r"):
        self.filename = os.path.abspath(filename)
        if mode == "w" or (mode == "a" and self.filename not in _MemH5File.store):
            _MemH5File.store[self.filename] = {}
            open(self.filename, "a").close()
        assert self.filename in _MemH5File.store, "no such file: " + filename
        self.data = _MemH5File.store[self.filename]

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False

    def __getitem__(self, key):
        return self.data[key]

    def __contains__(self, key):
        return key in self.data

    def keys(self):
        return self.data.keys()

    def create_dataset(self, key, data=None):
        assert key not in self.data, "name already exists"
        self.data[key] = np.asarray(data)


CONTAINER_SEED = 11
CONTAINER_SPF = 24            # syllables per file
CONTAINER_FILES = (3, 2)      # files in spec dir 0 / 1


def container_corpus():
    """The synthetic syllable corpus of the DataContainer case: per spec dir a list of
    (basename, specs float64 [spf,128,128]); shared by the generator and the test."""
    n = CONTAINER_SPF * sum(CONTAINER_FILES)
    specs = vae_oracle.make_input(CONTAINER_SEED, n).double().numpy()
    dirs, k = [], 0
    for d, nf in enumerate(CONTAINER_FILES):
        files = []
        for j in range(nf):
            files.append(("syllables_%04d" % j, specs[k:k + CONTAINER_SPF]))
            k += CONTAINER_SPF
        dirs.append(files)
    return dirs


def container_case(ref_vae):
    """The reference's DataContainer.request('latent_means') and request('latent_mean_pca')
    (ava/data/data_container.py:435-487, 538-551) run unmodified on the synthetic corpus,
    with the in-memory h5py stand-in and the reference VAE on the CPU."""
    import tempfile
    import types
    _ref_import.install_stubs()
    for name, attrs in (("umap", {"UMAP": None}), ("numba", None), ("numba.errors", None)):
        if name not in sys.modules and attrs is not None:
            m = types.ModuleType(name)
            for k, v in attrs.items():
                setattr(m, k, v)
            sys.modules[name] = m
    import h5py
    h5py.File = _MemH5File
    import ava.data.data_container as ref_dc
    import ava.models.vae_dataset as ref_ds
    import ava.models.utils as ref_mu
    ref_dc.h5py.File = ref_ds.h5py.File = ref_mu.h5py.File = _MemH5File
    _MemH5File.store = {}
    out = {"versions": np.array(versions())}
    with tempfile.TemporaryDirectory() as root:
        spec_dirs = [os.path.join(root, "specs%d" % d) for d in range(len(CONTAINER_FILES))]
        proj_dirs = [os.path.join(root, "proj%d" % d) for d in range(len(CONTAINER_FILES))]
        for sd, files in zip(spec_dirs, container_corpus()):
            os.makedirs(sd)
            for base, specs in files:
                with _MemH5File(os.path.join(sd, base + ".hdf5"), "w") as f:
                    f.create_dataset("specs", data=specs)
        model = ref_vae.VAE(save_dir=root, device_name='cpu')
        load_into_reference(model, vae_oracle.make_params(CONTAINER_SEED))
        model.save_state("checkpoint_000.tar")
        # torch >= 2.6 defaults torch.load to weights_only=True; the reference predates it
        orig_load = torch.load
        torch.load = lambda *a, **k: orig_load(*a, **{**k, "weights_only": False})
        orig_loaders = ref_dc.get_syllable_data_loaders
        # forked DataLoader workers are not needed for a 120-syllable corpus
        ref_dc.get_syllable_data_loaders = lambda part, **k: orig_loaders(part, num_workers=0, **k)
        try:
            dc = ref_dc.DataContainer(spec_dirs=spec_dirs, projection_dirs=proj_dirs,
                                      model_filename=os.path.join(root, "checkpoint_000.tar"),
                                      verbose=False)
            pca = dc.request('latent_mean_pca')
            latent = dc.request('latent_means')   # now read back from the projection files
        finally:
            torch.load = orig_load
            ref_dc.get_syllable_data_loaders = orig_loaders
        out["latent_means"] = latent
        out["latent_mean_pca"] = pca
        for d, pd in enumerate(proj_dirs):
            for fn in sorted(os.listdir(pd)):
                data = _MemH5File.store[os.path.abspath(os.path.join(pd, fn))]
                out["proj%d/%s:keys" % (d, fn)] = np.array(sorted(data.keys())).astype('S')
                out["proj%d/%s:latent_means" % (d, fn)] = data['latent_means']
    np.savez_compressed(os.path.join(GOLDEN, "container_case.npz"), **out)
    print("container case: latent", latent.shape, "pca", pca.shape, "first", pca[0])


def pca_case():
    """scikit-learn's PCA exactly as the reference constructs it (data_container.py:543),
    on synthetic latent clouds: one above 500 rows (covariance_eigh route) and one below
    (full-SVD route)."""
    import sklearn
    from sklearn.decomposition import PCA
    from oracle import pca_oracle
    out = {"versions": np.array(versions() + " sklearn " + sklearn.__version__)}
    for name, seed, n, d in (("big", 5, 3000, 32), ("small", 6, 200, 32), ("z8", 7, 1000, 8),
                             ("z64", 8, 1500, 64)):
        x = pca_oracle.synth_latents(seed, n, d)
        transform = PCA(n_components=2, copy=False, random_state=42)
        emb = transform.fit_transform(x.copy())
        out[name + ":embedding"] = emb
        out[name + ":mean"] = transform.mean_
        out[name + ":components"] = transform.components_
        out[name + ":explained_variance"] = transform.explained_variance_
        out[name + ":explained_variance_ratio"] = transform.explained_variance_ratio_
        out[name + ":shape"] = np.array([seed, n, d])
        o_emb, _ = pca_oracle.pca_fit_transform(x, 2)
        print("pca case", name, "oracle vs sklearn:", np.abs(o_emb - emb).max())
    np.savez_compressed(os.path.join(GOLDEN, "pca_cases.npz"), **out)



# ---------------------------------------------------------------- SURVEY 8(f) N3
WARP_DURS = (0.80, 0.93, 0.87, 1.02)        # seconds of the four synthetic "motifs"


def write_warp_corpus(root):
    """Four synthetic int16 wav files of different lengths + a saved 3-knot warp (the format
    WarpedWindowDataset itself saves, window_vae_dataset.py:497-506); shared by the generator
    and the test."""
    from scipy.io import wavfile
    p = dict(spec_oracle.FINCH_P)
    fs = p['fs']
    adir = os.path.join(root, "motifs")
    os.makedirs(adir, exist_ok=True)
    names = []
    for i, d in enumerate(WARP_DURS):
        fn = os.path.join(adir, "motif_%d.wav" % i)
        wavfile.write(fn, fs, spec_oracle.synth_audio(60 + i, int(d * fs), fs))
        names.append(fn)
    rng = np.random.default_rng(17)
    x_knots = np.sort(rng.uniform(0.05, 0.95, size=(len(names), 5)), axis=1)
    y_knots = np.sort(rng.uniform(0.05, 0.95, size=(len(names), 5)), axis=1)
    x_knots[:, 0] = y_knots[:, 0] = 0.0
    x_knots[:, -1] = y_knots[:, -1] = 1.0
    warp_fn = os.path.join(root, "knots.npy")
    np.save(warp_fn, {'x_knots': x_knots, 'y_knots': y_knots, 'template_dur': 0.79,
                      'audio_filenames': sorted(names), 'warp_params': {}})
    return names, warp_fn, p


def warped_case(ref_win, ref_pre):
    """The reference's WarpedWindowDataset run unmodified (window_vae_dataset.py:359-640) with
    the null warp and with saved knots: template duration, and per seed the file each item was
    drawn from and its un-warped target times (captured at the p['get_spec'] plugin boundary),
    plus a few spectrograms from the reference's own get_spec."""
    import tempfile
    out = {"versions": np.array(versions())}
    with tempfile.TemporaryDirectory() as root:
        names, warp_fn, p = write_warp_corpus(root)
        captured = []

        def spy_get_spec(t1, t2, audio, p_, fs=32000, max_dur=None, target_times=None, **kw):
            captured.append((t1, t2, len(audio), np.array(target_times)))
            return ref_pre.get_spec(t1, t2, audio, p_, fs=fs, max_dur=max_dur, target_times=target_times)
        p['get_spec'] = spy_get_spec
        for tag, kw in (("null", dict(warp_type='null', save_warp=False)),
                        ("knots", dict(load_warp=True, save_warp=False, warp_fn=warp_fn))):
            ds = ref_win.WarpedWindowDataset(list(names), p, transform=None, **kw)
            lens = [len(a) for a in ds.audio]
            out[tag + ":template_dur"] = np.array(ds.template_dur)
            out[tag + ":window_frac"] = np.array(ds.window_frac)
            for seed, n in ((0, 6), (5, 40)):
                del captured[:]
                specs = ds.__getitem__(np.arange(n), seed=seed)
                assert len(captured) == n
                out["%s:seed%d_files" % (tag, seed)] = np.array([lens.index(c[2]) for c in captured])
                out["%s:seed%d_times" % (tag, seed)] = np.stack([c[3] for c in captured])
                assert all(c[0] == 0.0 and c[1] == ds.template_dur for c in captured)
                if seed == 0:
                    out[tag + ":seed0_specs"] = np.stack(specs[:2])
            single = ds.__getitem__(0, seed=9)
            out[tag + ":single_seed9"] = np.asarray(single)
    np.savez_compressed(os.path.join(GOLDEN, "warped_cases.npz"), **out)
    print("warped cases: template_dur", float(out["null:template_dur"]), float(out["knots:template_dur"]))


def round2_cases(ref_win, ref_pre):
    """Round-2 additions (VERDICT items 1e, 9, 12, 13): float64 audio (the reference's complex128
    STFT path), within_syll_normalize, and the silence-rejection loop with REAL rejections."""
    from scipy.io import wavfile
    out = {"versions": np.array(versions())}
    # --- float64 audio, finch and mouse parameters
    p = dict(spec_oracle.FINCH_P)
    fs = p['fs']
    a64 = spec_oracle.synth_audio(21, int(2.0 * fs), fs, dtype=np.float64) / 7.0 + 0.123456789
    assert a64.dtype == np.float64
    for name, onset in [("f64_a", 0.7131), ("f64_b", 0.02)]:
        tt = np.linspace(onset, onset + p['window_length'], 128)
        spec, _ = ref_pre.get_spec(max(0.0, onset - 0.05), onset + p['window_length'] + 0.05, a64, p,
                                   fs=fs, target_times=tt)
        out[name] = spec
        out[name + "_t"] = np.array([onset])
    # --- within_syll_normalize (preprocessing/utils.py:106-109)
    for q in (0.5, 0.87):
        pn = dict(spec_oracle.MOUSE_P)
        pn.update(within_syll_normalize=True, normalize_quantile=q)
        fsm = pn['fs']
        am = spec_oracle.synth_audio(11, int(0.6 * fsm), fsm)
        spec, _ = ref_pre.get_spec(0.100, 0.180, am, pn, fs=fsm)
        out["norm_q%02d" % int(100 * q)] = spec
    pn = dict(spec_oracle.FINCH_P)
    pn.update(within_syll_normalize=True, normalize_quantile=0.5)
    a2 = spec_oracle.synth_audio(12, int(4.0 * fs), fs)
    tt = np.linspace(1.2345, 1.2345 + pn['window_length'], 128)
    spec, _ = ref_pre.get_spec(1.2345 - 0.05, 1.2345 + pn['window_length'] + 0.05, a2, pn, fs=fs,
                               target_times=tt)
    out["norm_finch"] = spec
    # --- FixedWindowDataset with real rejections
    calls = []
    real = ref_pre.get_spec

    def spy(*a, **k):
        calls.append(1)
        return real(*a, **k)
    p = dict(spec_oracle.FINCH_P)
    p['get_spec'] = spy
    with tempfile.TemporaryDirectory() as tmp:
        adir, rdir = os.path.join(tmp, "audio"), os.path.join(tmp, "rois")
        os.mkdir(adir)
        os.mkdir(rdir)
        for i, nm in enumerate(["x_song", "y_song", "z_song"]):
            wavfile.write(os.path.join(adir, nm + ".wav"), fs, spec_oracle.silent_half_audio(200 + i, fs))
            np.savetxt(os.path.join(rdir, nm + ".txt"), np.array([[0.2, 2.8]]))
        part = ref_win.get_window_partition([adir], [rdir], split=1.0)
        ds = ref_win.FixedWindowDataset(part['train']['audio'], part['train']['rois'], p,
                                        transform=None, min_spec_val=0.3)
        for seed in (0, 3):
            calls.clear()
            specs, fidx, onsets, offsets = ds.__getitem__(np.arange(16), seed=seed, return_seg_info=True)
            out["rej_seed%d_files" % seed] = np.array(fidx, dtype=np.int64)
            out["rej_seed%d_onsets" % seed] = np.array(onsets, dtype=np.float64)
            out["rej_seed%d_candidates" % seed] = np.array(len(calls))
            assert len(calls) > 16, "no rejection happened"
            assert all(np.max(sp) >= 0.3 for sp in specs)
            if seed == 0:
                out["rej_seed0_specs"] = np.stack(specs[:2]).astype(np.float64)
        out["rej_audio_order"] = np.array([os.path.basename(f) for f in part['train']['audio']])
    np.savez_compressed(os.path.join(GOLDEN, "round2_cases.npz"), **out)
    print("round-2 cases: candidates", int(out["rej_seed0_candidates"]), int(out["rej_seed3_candidates"]))


CKPT_SEED = 11


def checkpoint_recipe(model):
    """The state the checkpoint interchange tests save, on the reference's VAE or this package's CPU
    model alike: seeded parameters, BatchNorm buffers and gradients, one step of the model's own
    torch.optim.Adam (so the optimizer state is populated), epoch 4 and one train / test loss."""
    g = torch.Generator().manual_seed(CKPT_SEED)
    with torch.no_grad():
        for _, p in model.named_parameters():
            p.copy_(torch.randn(p.shape, generator=g) * 0.05)
        for k, b in model.named_buffers():
            if k.endswith("num_batches_tracked"):
                b.fill_(1)
            else:
                b.copy_(torch.rand(b.shape, generator=g) + (0.5 if k.endswith("running_var") else 0.0))
    for _, p in model.named_parameters():
        p.grad = torch.randn(p.shape, generator=g) * 0.01
    model.optimizer.step()
    model.epoch = 4
    model.loss['train'][3] = 12.5
    model.loss['test'][3] = 13.5


def _ckpt_positions(numel, salt):
    return np.random.default_rng(1000 + salt).choice(numel, size=min(numel, 16), replace=False)


def checkpoint_digest(ck):
    """(structure, samples) of a checkpoint in the reference's format (ava/models/vae.py:433-446):
    the structure as JSON -- top-level keys in order, each layer's keys / shapes / dtypes, the
    optimizer's param_groups and per-parameter state layout, loss, epoch, z_dim, lr -- and the
    values of every tensor at up to 16 seeded positions, in the order checkpoint_from_golden
    rebuilds them."""
    samples = {}

    def take(key, t):
        a = t.detach().double().reshape(-1).numpy()
        samples["sample:" + key] = a[_ckpt_positions(a.size, len(samples))]
    layers = {}
    for name, v in ck.items():
        if name in ("optimizer_state", "loss") or not isinstance(v, dict):
            continue
        layers[name] = [[k, list(t.shape), str(t.dtype)] for k, t in v.items()]
        for k, t in v.items():
            take(name + "." + k, t)
    opt = ck["optimizer_state"]
    state = []
    for idx, st in opt["state"].items():
        state.append([idx, [[k, list(t.shape), str(t.dtype)] for k, t in st.items()]])
        for k, t in st.items():
            take("opt.%d.%s" % (idx, k), t)
    structure = {"top_keys": list(ck.keys()), "layers": layers,
                 "param_groups": json.loads(json.dumps(opt["param_groups"])), "state": state,
                 "loss": {s: [[e, float(x)] for e, x in d.items()] for s, d in ck["loss"].items()},
                 "epoch": ck["epoch"], "z_dim": ck["z_dim"], "lr": ck["lr"],
                 "save_dir": type(ck["save_dir"]).__name__}
    return json.dumps(structure, sort_keys=True), samples


def checkpoint_from_golden(g, save_dir):
    """A checkpoint in the reference's format rebuilt from checkpoint_case.npz: the stored
    structure, every tensor filled with seeded values and the stored samples put back at their
    positions."""
    s = json.loads(str(g["structure"]))
    gen = torch.Generator().manual_seed(5)
    n = [0]

    def make(key, shape, dtype):
        dt = getattr(torch, dtype.split(".")[1])
        t = torch.randn(shape, generator=gen, dtype=torch.float64) if dt.is_floating_point else \
            torch.randint(0, 9, shape, generator=gen)
        t = t.to(dt)
        flat = t.view(-1)
        flat[torch.from_numpy(_ckpt_positions(flat.numel(), n[0]))] = torch.from_numpy(g["sample:" + key]).to(dt)
        n[0] += 1
        return t
    ck = {}
    for name in s["top_keys"]:
        if name in s["layers"]:
            ck[name] = {k: make(name + "." + k, shape, dt) for k, shape, dt in s["layers"][name]}
    state = {idx: {k: make("opt.%d.%s" % (idx, k), shape, dt) for k, shape, dt in entries}
             for idx, entries in s["state"]}
    groups = [dict(pg, betas=tuple(pg["betas"])) for pg in s["param_groups"]]
    rest = {"optimizer_state": {"state": state, "param_groups": groups},
            "loss": {k: {e: x for e, x in v} for k, v in s["loss"].items()},
            "z_dim": s["z_dim"], "epoch": s["epoch"], "lr": s["lr"], "save_dir": save_dir}
    return {name: ck[name] if name in ck else rest[name] for name in s["top_keys"]}


def checkpoint_case(vae_cls, source):
    """tests/golden/checkpoint_case.npz: structure and sampled values of the checkpoint `vae_cls`
    writes after checkpoint_recipe."""
    with tempfile.TemporaryDirectory() as d:
        model = vae_cls(save_dir=d, device_name='cpu')
        checkpoint_recipe(model)
        model.save_state("checkpoint_004.tar")
        ck = torch.load(os.path.join(d, "checkpoint_004.tar"), map_location="cpu")
    structure, samples = checkpoint_digest(ck)
    out = dict(samples, structure=np.array(structure), source=np.array(source), versions=np.array(versions()))
    np.savez_compressed(os.path.join(GOLDEN, "checkpoint_case.npz"), **out)
    print("checkpoint case (%s): %d top-level keys, %d sampled tensors" % (source, len(ck), len(samples)))


def main():
    os.makedirs(GOLDEN, exist_ok=True)
    torch.set_num_threads(8)
    which = sys.argv[1:] or ["vae", "adam", "spec", "sampler", "process", "mmd", "container", "pca", "warped",
                             "round2", "checkpoint"]
    if which == ["checkpoint"] and not _ref_import.reference_available():
        # without the reference: this package's save_state, a line-for-line restatement of the
        # reference's (vae.py:433-446); the interchange test checks the file against the reference
        # wherever the reference is present
        vae = importlib.import_module("autoencoded-vocal-analysis_b200.models.vae")
        checkpoint_case(vae.VAE, "this package's save_state (restates ava/models/vae.py:433-446)")
        return
    ref_vae, ref_pre, ref_win, ref_ds = _ref_import.import_reference()
    if "vae" in which:
        vae_case(ref_vae, "vae_train_b7", seed=0, batch=7, train=True)
        vae_case(ref_vae, "vae_eval_b7", seed=1, batch=7, train=False)
        vae_case(ref_vae, "vae_train_b64", seed=2, batch=64, train=True)
        vae_case(ref_vae, "vae_train_b1", seed=3, batch=1, train=True, prec=4.0)
    if "adam" in which:
        adam_case(ref_vae, "adam_b5_s3", seed=4, batch=5, steps=3)
    if "spec" in which:
        spec_cases(ref_pre)
    if "sampler" in which:
        sampler_cases(ref_win, ref_ds, ref_pre)
    if "process" in which:
        process_case(ref_pre)
    if "mmd" in which:
        mmd_case()
    if "container" in which:
        container_case(ref_vae)
    if "pca" in which:
        pca_case()
    if "warped" in which:
        warped_case(ref_win, ref_pre)
    if "round2" in which:
        round2_cases(ref_win, ref_pre)
    if "checkpoint" in which:
        checkpoint_case(ref_vae.VAE, "reference ava/models/vae.py save_state")


if __name__ == "__main__":
    main()
