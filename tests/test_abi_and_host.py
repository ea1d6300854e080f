"""CPU tests: the C-ABI library loads and exports every symbol include/ava_b200.h declares
(no compute calls), and the host-side mirror of the reference interface behaves like the
reference's (parameter registration, checkpoint layout, loud failure without CUDA)."""
import importlib
import json
import os
import re

import numpy as np
import pytest
import torch

from oracle import spec_oracle, vae_oracle
from tests.helpers import ROOT, load_golden

PKG = "autoencoded-vocal-analysis_b200"


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "ava_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(ava_b200_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 20
    lib = importlib.import_module(PKG + "._lib")
    handle = lib.lib()
    for name in declared:
        assert hasattr(handle, name), "missing export " + name
    assert sorted(lib.SIGNATURES) == declared       # the ctypes table covers the header
    assert handle.ava_b200_abi_version() == int(re.search(r"#define AVA_B200_ABI_VERSION (\d+)", hdr).group(1))
    assert lib.launch_count() >= 0 and lib.last_error() == ""


def test_alias_module_and_reference_surface():
    import ava_b200
    from ava_b200.models import vae, vae_dataset, window_vae_dataset
    from ava_b200.preprocessing import utils as pre
    assert vae.X_SHAPE == (128, 128) and vae.X_DIM == 16384
    for name in ("encode", "decode", "forward", "train_epoch", "test_epoch", "train_loop",
                 "save_state", "load_state", "visualize", "get_latent", "compute_loss"):
        assert callable(getattr(vae.VAE, name))
    for name in ("get_syllable_partition", "get_syllable_data_loaders", "SyllableDataset"):
        assert hasattr(vae_dataset, name)
    for name in ("get_window_partition", "get_fixed_window_data_loaders", "FixedWindowDataset",
                 "get_warped_window_data_loaders", "WarpedWindowDataset"):
        assert hasattr(window_vae_dataset, name)
    assert callable(pre.get_spec) and pre.EPSILON == 1e-12
    assert ava_b200.__version__


def test_vae_container_matches_reference_layout(tmp_path):
    vae = importlib.import_module(PKG + ".models.vae")
    model = vae.VAE(save_dir=str(tmp_path), device_name='cpu')
    names = [k for k, _ in model.named_parameters()]
    want = vae_oracle.param_order()
    assert names == [k for k, _ in want]                       # registration order (Adam index)
    assert [tuple(p.shape) for p in model.parameters()] == [s for _, s in want]
    assert sum(p.numel() for p in model.parameters()) == 17426323
    assert len(model.state_dict()) == 122
    assert set(model._get_layers()) == {'fc1', 'fc2', 'fc31', 'fc32', 'fc33', 'fc41', 'fc42',
                                        'fc43', 'fc5', 'fc6', 'fc7', 'fc8'} | \
        {'bn%d' % i for i in range(1, 15)} | {'conv%d' % i for i in range(1, 8)} | \
        {'convt%d' % i for i in range(1, 8)}
    # flat storage: parameters are views, 16-byte aligned, heads contiguous
    base = model._flat_p.data_ptr()
    for k, p in model.named_parameters():
        assert p.data_ptr() == base + 4 * model._off[k]
        if not k.startswith(("fc3", "fc4")):
            assert model._off[k] % 4 == 0
    assert model._off["fc32.weight"] == model._off["fc31.weight"] + 64 * 256
    assert model._off["fc43.bias"] == model._off["fc41.bias"] + 64
    # load seeded weights, checkpoint round trip in the reference's layout
    P = vae_oracle.make_params(3)
    model.load_flat_state(P)
    for k, v in model.state_dict().items():
        assert torch.equal(v.cpu(), P[k]), k
    model.epoch = 7
    model.loss['train'][6] = 1.5
    model.save_state("ck.tar")
    ck = torch.load(os.path.join(str(tmp_path), "ck.tar"), map_location="cpu")
    assert len(ck) == 46 and ck['z_dim'] == 32 and ck['epoch'] == 7 and ck['lr'] == 1e-3
    assert list(ck['bn3'].keys()) == ['weight', 'bias', 'running_mean', 'running_var',
                                      'num_batches_tracked']
    assert ck['optimizer_state']['state'] == {}                # no step taken yet (as torch)
    model2 = vae.VAE(save_dir=str(tmp_path), device_name='cpu')
    model2.load_state(os.path.join(str(tmp_path), "ck.tar"))
    assert model2.epoch == 7 and model2.loss['train'][6] == 1.5
    for (k, a), (_, b) in zip(model.state_dict().items(), model2.state_dict().items()):
        assert torch.equal(a, b), k
    # a checkpoint written by torch's own Adam state (what the reference saves) is adopted
    ref_like = vae.VAE(save_dir=str(tmp_path), device_name='cpu')
    ref_like.load_flat_state(P)
    for p in ref_like.parameters():
        p.grad = torch.full_like(p, 0.01)
    ref_like.optimizer.step()                                   # torch Adam creates its state
    ref_like.save_state("ck2.tar")
    model3 = vae.VAE(save_dir=str(tmp_path), device_name='cpu')
    model3.load_state(os.path.join(str(tmp_path), "ck2.tar"))
    assert model3._step_host == 1
    k0 = "fc1.weight"
    st = ref_like.optimizer.state[dict(ref_like.named_parameters())[k0]]
    assert torch.equal(model3._views_m[k0], st['exp_avg'])
    assert torch.equal(model3._views_v[k0], st['exp_avg_sq'])
    # no CPU fallback
    with pytest.raises(RuntimeError, match="CUDA"):
        model.forward(torch.zeros(2, 128, 128))
    with pytest.raises(RuntimeError, match="CUDA"):
        model.get_latent([torch.zeros(2, 128, 128)])
    with pytest.raises(ValueError):
        model._as_input(torch.zeros(2, 64, 64))


def test_checkpoints_interchange_with_the_real_reference(tmp_path, monkeypatch):
    """A checkpoint written by the UNMODIFIED reference VAE (ava/models/vae.py:432-472, imported from
    /root/reference; one torch-Adam step taken so the optimizer state is populated) loads into this
    package's VAE, and a checkpoint written here loads into the reference -- parameters, BatchNorm
    buffers, Adam moments / step, epoch and loss history identical.  Runs where the reference is
    mounted (the CPU container); skipped on the GPU box."""
    from oracle import _ref_import
    if not _ref_import.reference_available():
        pytest.skip("/root/reference not present")
    # (the stand-in h5py / affinewarp / matplotlib modules the reference import needs must not
    # leak into the tests that follow)
    import sys
    for name in ("h5py", "affinewarp", "affinewarp.crossval", "matplotlib", "matplotlib.pyplot"):
        if name not in sys.modules:
            monkeypatch.setitem(sys.modules, name, None)
            monkeypatch.delitem(sys.modules, name)
    ref_vae = _ref_import.import_reference()[0]
    vae = importlib.import_module(PKG + ".models.vae")
    rdir, odir = str(tmp_path / "ref"), str(tmp_path / "ours")
    torch.manual_seed(11)
    ref = ref_vae.VAE(save_dir=rdir, device_name='cpu')
    x = torch.rand(3, 128, 128)
    ref.train()
    ref.optimizer.zero_grad()
    ref.forward(x).backward()
    ref.optimizer.step()
    ref.epoch = 4
    ref.loss['train'][3] = 12.5
    ref.loss['test'][3] = 13.5
    ref.save_state(os.path.join(rdir, "checkpoint_004.tar"))
    # reference -> ours
    ours = vae.VAE(save_dir=odir, device_name='cpu')
    ours.load_state(os.path.join(rdir, "checkpoint_004.tar"))
    assert ours.epoch == 4 and ours.loss['train'][3] == 12.5 and ours.loss['test'][3] == 13.5
    rsd = ref.state_dict()
    osd = ours.state_dict()
    assert list(rsd.keys()) == list(osd.keys())
    for k in rsd:
        assert torch.equal(rsd[k], osd[k]), k
    assert ours._step_host == 1
    rparams = dict(ref.named_parameters())
    for k in ("conv1.weight", "fc1.weight", "fc43.bias", "bn14.weight", "convt7.bias"):
        st = ref.optimizer.state[rparams[k]]
        assert torch.equal(ours._views_m[k], st['exp_avg']), k
        assert torch.equal(ours._views_v[k], st['exp_avg_sq']), k
    # ours -> reference (written from the flat native state: moments, step and all)
    ours.save_state(os.path.join(odir, "checkpoint_004.tar"))
    ref2 = ref_vae.VAE(save_dir=rdir, device_name='cpu')
    ref2.load_state(os.path.join(odir, "checkpoint_004.tar"))
    assert ref2.epoch == 4 and ref2.loss['train'][3] == 12.5
    for k, v in ref2.state_dict().items():
        assert torch.equal(v, rsd[k]), k
    r2params = dict(ref2.named_parameters())
    for k in ("conv1.weight", "fc1.weight", "fc43.bias", "bn14.weight"):
        a, b = ref2.optimizer.state[r2params[k]], ref.optimizer.state[rparams[k]]
        assert torch.equal(a['exp_avg'], b['exp_avg']) and torch.equal(a['exp_avg_sq'], b['exp_avg_sq']), k
        assert float(a['step']) == float(b['step']) == 1.0
    # and the reference keeps training from it (its own Adam accepts the restored state)
    ref2.train()
    ref2.optimizer.zero_grad()
    ref2.forward(x).backward()
    ref2.optimizer.step()
    assert float(ref2.optimizer.state[r2params["fc1.weight"]]['step']) == 2.0
    # the stored checkpoint golden is what the reference itself writes
    from oracle import make_golden
    ref3 = ref_vae.VAE(save_dir=rdir, device_name='cpu')
    make_golden.checkpoint_recipe(ref3)
    ref3.save_state("golden.tar")
    structure, samples = make_golden.checkpoint_digest(torch.load(os.path.join(rdir, "golden.tar"), map_location="cpu"))
    g = load_golden("checkpoint_case")
    assert json.loads(structure) == json.loads(str(g["structure"]))
    assert sorted(samples) == sorted(k for k in g.files if k.startswith("sample:"))
    for k, v in samples.items():
        assert np.array_equal(v, g[k]), k


def test_checkpoints_interchange_with_reference_golden(tmp_path):
    """The checkpoint format of the reference (ava/models/vae.py:433-472) from the stored golden
    (tests/golden/checkpoint_case.npz: structure and sampled values of the checkpoint written after
    oracle.make_golden.checkpoint_recipe): what this package writes has that structure and those
    values, and a checkpoint rebuilt from the golden loads here -- parameters, BatchNorm buffers,
    Adam moments and step, epoch and loss history -- and is written back unchanged."""
    from oracle import make_golden
    vae = importlib.import_module(PKG + ".models.vae")
    g = load_golden("checkpoint_case")
    want = json.loads(str(g["structure"]))
    sample_keys = sorted(k for k in g.files if k.startswith("sample:"))

    def check(path):
        structure, samples = make_golden.checkpoint_digest(torch.load(path, map_location="cpu"))
        assert json.loads(structure) == want
        assert sorted(samples) == sample_keys
        for k, v in samples.items():
            assert np.array_equal(v, g[k]), k
    # ours -> golden
    ours = vae.VAE(save_dir=str(tmp_path), device_name='cpu')
    make_golden.checkpoint_recipe(ours)
    ours.save_state("ours.tar")
    check(str(tmp_path / "ours.tar"))
    # golden -> ours
    ck = make_golden.checkpoint_from_golden(g, str(tmp_path))
    torch.save(ck, str(tmp_path / "golden.tar"))
    model = vae.VAE(save_dir=str(tmp_path), device_name='cpu')
    model.load_state(str(tmp_path / "golden.tar"))
    assert model.epoch == ck["epoch"] == 4 and model.loss == ck["loss"]
    sd = model.state_dict()
    for name, layer in ck.items():
        if name in want["layers"]:
            for k, t in layer.items():
                assert torch.equal(sd[name + "." + k], t), name + "." + k
    names = [k for k, _ in model.named_parameters()]
    state = ck["optimizer_state"]["state"]
    assert sorted(state) == list(range(len(names)))
    for idx, st in state.items():
        assert torch.equal(model._views_m[names[idx]], st["exp_avg"]), names[idx]
        assert torch.equal(model._views_v[names[idx]], st["exp_avg_sq"]), names[idx]
    assert model._step_host == int(state[0]["step"]) == 1
    # ... and written back in the same format with the same values
    model.save_state("again.tar")
    check(str(tmp_path / "again.tar"))


def test_time_bracketing_matches_oracle_coordinates():
    pre = importlib.import_module(PKG + ".preprocessing.utils")
    rng = np.random.default_rng(0)
    fs, nperseg, hop = 32000, 512, 256
    n = 50
    t1 = rng.uniform(0, 2.0, size=n)
    seg = rng.integers(600, 9000, size=n)
    K = pre.num_frames(seg, nperseg, hop)
    kmax = int(K.max())
    base = np.arange(nperseg / 2, nperseg / 2 + kmax * hop, hop) / float(fs) - (nperseg / 2) / fs
    tt = t1[:, None] + rng.uniform(-0.05, 0.35, size=(n, 128))
    tt[0, 0] = t1[0]                                  # exactly on the first frame time
    idx, w = pre.bracket(t1, base, K, tt)
    for r in range(n):
        _, t, _ = spec_oracle.stft(np.zeros(seg[r]), fs, nperseg, nperseg - hop)
        assert len(t) == K[r]
        g = t + t1[r]
        i = np.clip(np.searchsorted(g, tt[r], side='right') - 1, 0, len(g) - 2)
        bad = (tt[r] < g[0]) | (tt[r] > g[-1])
        assert np.array_equal(idx[r] < 0, bad)
        ok = ~bad
        assert np.array_equal(idx[r][ok], i[ok])
        assert np.array_equal(w[r][ok], ((tt[r] - g[i]) / (g[i + 1] - g[i]))[ok])


def test_window_sampler_bit_exact_on_cpu():
    win = importlib.import_module(PKG + ".models.window_vae_dataset")
    p = dict(spec_oracle.FINCH_P)
    rng = np.random.default_rng(1)
    rois = [np.sort(rng.uniform(0, 50, size=(k, 2)), axis=1) + np.array([0.0, 1.0])
            for k in (1, 3, 2, 5)]
    ds = win.FixedWindowDataset(["d.wav", "b.wav", "a.wav", "c.wav"], None, p,
                                audio=[np.zeros(10, np.int16)] * 4, fs=32000, rois=rois)
    for seed in (0, 5):
        want_f, want_on = spec_oracle.sample_windows(40, seed, ds.rois, ds.file_weights,
                                                     ds.roi_weights, p['window_length'])
        np.random.seed(seed)
        got_f, got_on = ds._draw(40)
        assert np.array_equal(got_f, want_f) and np.array_equal(got_on, want_on)
    g = load_golden("sampler_cases")
    assert g["seed0_files"].shape == (12,)


def test_next_rows_host_logic_and_no_cpu_fallback(tmp_path):
    """process_sylls / mmd_plots (SURVEY 8(f) N2, N4): file pairing and parsing follow the
    reference; compute raises without a CUDA device instead of falling back."""
    import importlib
    import numpy as np
    import pytest
    import torch
    pp = importlib.import_module(PKG + ".preprocessing.preprocess")
    mmd = importlib.import_module(PKG + ".plotting.mmd_plots")
    adir, sdir = tmp_path / "audio", tmp_path / "segs"
    adir.mkdir()
    sdir.mkdir()
    for name in ("b.wav", "a.wav", "c.wav", "notes.md"):
        (adir / name).write_bytes(b"")
    np.savetxt(sdir / "a.txt", np.array([[0.1, 0.2], [0.3, 0.45]]), header="onset offset")
    np.savetxt(sdir / "c.txt", np.zeros((0, 2)), header="none")
    a, s = pp.get_audio_seg_filenames(str(adir), str(sdir), {})
    assert [os.path.basename(i) for i in a] == ["a.wav", "c.wav"]       # b.wav has no segment file
    assert [os.path.basename(i) for i in s] == ["a.txt", "c.txt"]
    assert [os.path.basename(i) for i in pp.get_audio_filenames(str(adir))] == ["a.wav", "b.wav", "c.wav"]
    on, off = pp.read_onsets_offsets_from_file(str(sdir / "a.txt"), {})
    assert list(on) == [0.1, 0.3] and list(off) == [0.2, 0.45]
    on, off = pp.read_onsets_offsets_from_file(str(sdir / "c.txt"), {})
    assert len(on) == 0 and len(off) == 0
    assert pp.is_audio_file("x.wav") and not pp.is_audio_file("x.WAV") and not pp.is_audio_file("wav")
    # MMD^2 from Gram block sums == the reference's three-term estimator
    rng = np.random.default_rng(0)
    x, y = rng.standard_normal((7, 4)), rng.standard_normal((9, 4)) + 0.3
    A = -0.5 / 1.7 ** 2
    k = lambda u, v: np.exp(A * ((u[:, None] - v[None]) ** 2).sum(-1))     # noqa: E731
    S = np.array([[k(x, x).sum(), k(x, y).sum()], [k(y, x).sum(), k(y, y).sum()]])
    from oracle import mmd_oracle
    lat = np.concatenate([x, y])
    want = mmd_oracle.estimate_mmd2(lat, np.arange(7), np.arange(7, 16), 1.7)
    assert abs(mmd._mmd2_from_sums(S, [7, 9], 0, 1) - want) <= 1e-12
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            mmd.estimate_median_sigma(lat)
        with pytest.raises(RuntimeError):
            pp._syll_specs_batched(np.array([0.1]), np.array([0.2]), np.zeros(32000, np.int16), 32000,
                                   {'max_dur': 0.2, 'time_stretch': False, 'num_time_bins': 128,
                                    'nperseg': 512, 'noverlap': 256, 'within_syll_normalize': False}, None)


def test_data_container_host_logic_and_no_cpu_fallback(tmp_path):
    """SURVEY 8(f) N1: the DataContainer request/read/write protocol follows the reference
    (ava/data/data_container.py:251-373, 652-716); computing latent means or the PCA without
    a CUDA device raises instead of falling back."""
    import importlib
    import numpy as np
    import pytest
    import torch
    dcm = importlib.import_module(PKG + ".data.data_container")
    mu = importlib.import_module(PKG + ".models.utils")
    assert dcm.PROJECTION_FIELDS == ['latent_means', 'latent_mean_pca', 'latent_mean_umap']
    assert dcm.SPEC_FIELDS == ['specs', 'onsets', 'offsets', 'audio_filenames']
    assert len(dcm.ALL_FIELDS) == 1 + 1 + 2 + 3 + 4 + 14 + 16 + 15
    try:
        import h5py  # noqa: F401
        ext = ".hdf5"
    except ImportError:
        ext = ".npz"
    sdirs = [str(tmp_path / "s0"), str(tmp_path / "s1")]
    pdirs = [str(tmp_path / "p0"), str(tmp_path / "p1")]
    rng = np.random.default_rng(0)
    k = 0
    for sd, nf in zip(sdirs, (2, 1)):
        os.makedirs(sd)
        for j in range(nf):
            fn = os.path.join(sd, "syllables_%04d%s" % (j, ext))
            mu.append_field(fn, 'specs', rng.random((3, 128, 128)))
            mu.append_field(fn, 'onsets', np.arange(3) + 10.0 * k)
            mu.append_field(fn, 'offsets', np.arange(3) + 10.0 * k + 0.5)
            mu.append_field(fn, 'audio_filenames', np.array(["f%d.wav" % k] * 3).astype('S'))
            k += 1
    with pytest.raises(Exception):
        mu.append_field(fn, 'specs', np.zeros(3))            # like h5py: no overwrite
    assert mu.stored_fields(fn) == {'specs': 3, 'onsets': 3, 'offsets': 3, 'audio_filenames': 3}
    dc = dcm.DataContainer(spec_dirs=sdirs, projection_dirs=pdirs, model_filename="none.tar",
                           verbose=False, plots_dir=str(tmp_path / "plots"))
    assert os.path.isdir(tmp_path / "plots")
    assert set(dc.fields) == set(dcm.SPEC_FIELDS) and dc.sylls_per_file is None
    assert list(dc.request('onsets')) == [0., 1., 2., 10., 11., 12., 20., 21., 22.]
    assert list(dc.request('audio_filenames')) == ["f0.wav"] * 3 + ["f1.wav"] * 3 + ["f2.wav"] * 3
    assert dc.request('specs').shape == (9, 128, 128)
    with pytest.raises(NotImplementedError):
        dc.request('not_a_field')
    with pytest.raises(NotImplementedError):
        dc.request('latent_mean_umap')
    with pytest.raises(AssertionError):
        dcm.DataContainer(spec_dirs=sdirs, verbose=False).request('latent_means')
    # projections written file by file in directory order, picked up by a new container
    dc.sylls_per_file = 3
    for pd in pdirs:
        os.makedirs(pd)
    emb = np.arange(18.0).reshape(9, 2)
    dc._write_projection('latent_mean_pca', emb)
    assert sorted(os.listdir(pdirs[0])) == ["syllables_0000" + ext, "syllables_0001" + ext]
    dc2 = dcm.DataContainer(spec_dirs=sdirs, projection_dirs=pdirs, verbose=False)
    assert 'latent_mean_pca' in dc2.fields and dc2.sylls_per_file == 3
    np.testing.assert_array_equal(dc2.request('latent_mean_pca'), emb)
    dc2.clear_projections()
    assert os.listdir(pdirs[0]) == [] and 'latent_mean_pca' not in dc2.fields
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            dcm.LatentPCA(2).fit_transform(rng.standard_normal((50, 32)))


def test_streaming_syllable_loader_matches_resident(tmp_path):
    """The file-at-a-time loader used by DataContainer yields exactly the batches of the
    resident loader (batches may straddle files; ragged last batch kept)."""
    import importlib
    import numpy as np
    import torch
    ds = importlib.import_module(PKG + ".models.vae_dataset")
    rng = np.random.default_rng(1)
    fns = []
    for j in range(5):
        fn = str(tmp_path / ("s%d.npy" % j))
        np.save(fn, rng.random((7, 128, 128)))
        fns.append(fn)
    dataset = ds.SyllableDataset(fns, 7)
    for bs in (1, 4, 7, 10, 64):
        a = list(ds.DeviceSyllableLoader(dataset, batch_size=bs, device="cpu"))
        loader = ds.DeviceSyllableLoader(dataset, batch_size=bs, device="cpu", streaming=True)
        b = list(loader)
        assert len(a) == len(b) == len(loader)
        assert all(torch.equal(x, y) for x, y in zip(a, b))
        assert sum(len(x) for x in b) == len(dataset) == 35


def test_hdf5_code_path_with_stand_in_h5py(tmp_path, monkeypatch):
    """h5py is not installed in this environment, so the HDF5 branches of the file helpers
    would otherwise never run: exercise them through an in-memory stand-in for ``h5py.File``
    (the same one the golden generator uses to run the reference's DataContainer)."""
    import importlib
    import sys
    import types
    import numpy as np
    from oracle.make_golden import _MemH5File
    try:
        import h5py  # noqa: F401
        pytest.skip("real h5py present: the HDF5 branches are exercised by the other tests")
    except ImportError:
        pass
    fake = types.ModuleType("h5py")
    fake.File = _MemH5File
    monkeypatch.setitem(sys.modules, "h5py", fake)
    _MemH5File.store = {}
    mu = importlib.import_module(PKG + ".models.utils")
    dcm = importlib.import_module(PKG + ".data.data_container")
    sd, pd = str(tmp_path / "specs"), str(tmp_path / "proj")
    os.makedirs(sd)
    os.makedirs(pd)
    rng = np.random.default_rng(0)
    for j in range(2):
        fn = os.path.join(sd, "syllables_%04d.hdf5" % j)
        mu.append_field(fn, 'specs', rng.random((3, 128, 128)))
        mu.append_field(fn, 'onsets', np.arange(3.0) + 10 * j)
        mu.append_field(fn, 'offsets', np.arange(3.0) + 10 * j + 0.5)
        mu.append_field(fn, 'audio_filenames', np.array(["f%d.wav" % j] * 3).astype('S'))
    (tmp_path / "specs" / "notes.npz").write_bytes(b"")          # ignored when h5py is importable
    assert [os.path.basename(f) for f in mu.get_hdf5s_from_dir(sd)] == ["syllables_0000.hdf5",
                                                                        "syllables_0001.hdf5"]
    assert mu.stored_fields(os.path.join(sd, "syllables_0001.hdf5")) == \
        {'specs': 3, 'onsets': 3, 'offsets': 3, 'audio_filenames': 3}
    assert mu.read_specs(os.path.join(sd, "syllables_0000.hdf5")).shape == (3, 128, 128)
    with pytest.raises(AssertionError):
        mu.append_field(os.path.join(sd, "syllables_0000.hdf5"), 'specs', np.zeros(3))
    with pytest.raises(AssertionError):
        mu.read_field(os.path.join(sd, "syllables_0000.hdf5"), 'latent_means')
    dc = dcm.DataContainer(spec_dirs=[sd], projection_dirs=[pd], verbose=False)
    assert list(dc.request('onsets')) == [0., 1., 2., 10., 11., 12.]
    assert list(dc.request('audio_filenames')) == ["f0.wav"] * 3 + ["f1.wav"] * 3
    dc.sylls_per_file = 3
    dc._write_projection('latent_means', np.arange(6 * 32.0).reshape(6, 32))
    dc2 = dcm.DataContainer(spec_dirs=[sd], projection_dirs=[pd], verbose=False)
    assert 'latent_means' in dc2.fields and dc2.sylls_per_file == 3
    np.testing.assert_array_equal(dc2.request('latent_means'), np.arange(6 * 32.0).reshape(6, 32))
    # the syllable partition / dataset read the same files
    ds = importlib.import_module(PKG + ".models.vae_dataset")
    part = ds.get_syllable_partition([sd], 1, shuffle=False)
    assert len(part['train']) == 2 and mu._get_sylls_per_file(part) == 3
    item = ds.SyllableDataset(part['train'], 3, transform=mu.numpy_to_tensor)[4]
    assert tuple(item.shape) == (128, 128) and str(item.dtype) == "torch.float32"


def test_warped_window_sampling_vectorised_equals_reference_loop(tmp_path):
    """WarpedWindowDataset._draw (vectorised linspace / inverse warp) against the reference's
    per-item loop (ava/models/window_vae_dataset.py:613-624) restated literally: same draws
    from the legacy global stream, bit-identical target times -- null warp and saved knots."""
    import importlib
    import numpy as np
    win = importlib.import_module(PKG + ".models.window_vae_dataset")
    fs = 32000
    p = {'fs': fs, 'nperseg': 512, 'noverlap': 256, 'num_time_bins': 128, 'num_freq_bins': 128,
         'window_length': 0.12, 'min_freq': 400, 'max_freq': 10e3, 'spec_min_val': 2.0,
         'spec_max_val': 6.5, 'mel': True, 'time_stretch': False, 'within_syll_normalize': False,
         'max_dur': 1e9}
    rng = np.random.default_rng(0)
    audio = [np.zeros(int(fs * d), np.int16) for d in (0.9, 1.0, 1.1, 0.95)]
    names = ["m%d.wav" % i for i in range(4)]
    knots_fn = str(tmp_path / "knots.npy")
    x_knots = np.sort(rng.uniform(0, 1, size=(4, 5)), axis=1)
    y_knots = np.sort(rng.uniform(0, 1, size=(4, 5)), axis=1)
    x_knots[:, 0] = y_knots[:, 0] = 0.0
    x_knots[:, -1] = y_knots[:, -1] = 1.0
    np.save(knots_fn, {'x_knots': x_knots, 'y_knots': y_knots, 'template_dur': 0.93,
                       'audio_filenames': np.array(sorted(names))})
    datasets = [win.WarpedWindowDataset(names, p, warp_type='null', audio=audio, fs=fs),
                win.WarpedWindowDataset(names, p, load_warp=True, warp_fn=knots_fn, audio=audio, fs=fs)]

    def reference_loop(ds, n, seed):
        np.random.seed(seed)
        files, tts = [], []
        for _ in range(n):
            file_index = np.random.randint(len(ds.audio))
            start_t = ds.start_q + np.random.rand() * (ds.stop_q - ds.start_q - ds.window_frac)
            stop_t = start_t + ds.window_frac
            t_vals = np.linspace(start_t, stop_t, ds.p['num_time_bins'])
            files.append(file_index)
            tts.append(ds._get_unwarped_times(t_vals, file_index) * ds.template_dur)
        np.random.seed(None)
        return np.array(files), np.array(tts)

    for ds in datasets:
        for n, seed in ((1, 0), (7, 1), (300, 2)):
            f_ref, t_ref = reference_loop(ds, n, seed)
            f_new, t_new = ds._draw(n, seed)
            assert np.array_equal(f_new, f_ref)
            assert np.array_equal(t_new, t_ref)            # bit-identical


def test_shard_files_partitions_and_aligns():
    """vae_dataset.shard_files: the ranks' blocks tile [0, n_files) in order; interior boundaries
    fall on batch boundaries whenever a file boundary that is also a batch boundary exists."""
    import importlib
    import numpy as np
    ds = importlib.import_module(PKG + ".models.vae_dataset")
    rng = np.random.default_rng(0)
    for _ in range(300):
        n = int(rng.integers(0, 200))
        world = int(rng.integers(1, 9))
        spf = int(rng.choice([1, 3, 4, 24, 100, 512]))
        batch = int(rng.choice([1, 4, 64, 1024]))
        blocks = [ds.shard_files(n, r, world, spf, batch) for r in range(world)]
        assert blocks[0][0] == 0 and blocks[-1][1] == n
        assert all(lo <= hi for lo, hi in blocks)
        assert all(blocks[r][1] == blocks[r + 1][0] for r in range(world - 1))
        q = batch // np.gcd(batch, spf)
        for lo, hi in blocks[1:]:
            if lo not in (0, n):
                assert (lo * spf) % batch == 0 or q > n, (n, world, spf, batch, blocks)
    # batch size 1 (eval-mode BatchNorm: no alignment needed) splits evenly
    assert [ds.shard_files(100, r, 8) for r in range(8)] == [(12 * r + (r * 4) // 8, 12 * (r + 1) + ((r + 1) * 4) // 8)
                                                              for r in range(8)]
