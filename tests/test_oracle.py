"""CPU tests: the oracle restatement against the golden vectors produced by the UNMODIFIED
reference (tests/golden/make_golden.py), plus the length arithmetic pinned by the reference's
own FLAC fixtures (SURVEY 8c)."""
import importlib.util
import os

import numpy as np
import torch
import pytest
from conftest import GOLDEN, golden, rel_rms
from oracle import vf_oracle as O


def test_frontend_matches_reference(states):
    g = golden("frontend")
    sp, mel = O.frontend(torch.from_numpy(g["wav"]), states[0])
    assert rel_rms(mel.numpy(), g["mel"]) < 1e-6
    assert rel_rms(sp.numpy()[:, :, :4], g["sp_slice"]) < 1e-6


@pytest.mark.parametrize("T", [1, 63, 65])
def test_analysis_matches_reference(states, T):
    g = golden(f"analysis_T{T}")
    out = O.analysis(torch.from_numpy(g["mel"]), states[0])
    assert rel_rms(out.numpy(), g["out"]) < 2e-5


def test_analysis_mode2_matches_reference(states):
    g = golden("analysis_mode2")
    T = g["mel"].shape[2]
    masks = [torch.from_numpy(np.unpackbits(g[k])[: T * 512].reshape(1, 1, T, 512).astype(bool)) for k in ("mask0", "mask1")]
    out = O.analysis(torch.from_numpy(g["mel"]), states[0], train=True, drop_masks=masks)
    assert rel_rms(out.numpy(), g["out"]) < 1e-4


@pytest.mark.parametrize("T", [3, 20])
def test_vocoder_matches_reference(states, T):
    g = golden(f"vocoder_T{T}")
    out = O.vocoder_forward(torch.from_numpy(g["mel"]), states[1])
    assert out.shape[-1] == (T + T % 2 + 4) * 441
    assert rel_rms(out.numpy(), g["out"]) < 2e-5


def test_restore_mode0_matches_reference(states):
    g = golden("restore_mode0")
    out = O.restore_inmem(g["wav"], states[0], states[1], mode=0)
    assert out.shape == g["out"].shape == (1, g["wav"].shape[0])
    assert rel_rms(out, g["out"]) < 1e-4


def test_fixture_lengths():
    """Sample counts of the reference's own fixtures (FLAC STREAMINFO, BASELINE.md):
    mode 0: 132300 -> 132300; mode 1 -> 132096; oracle: 96076 -> 97902."""
    L = 132300
    T = 1 + L // 441
    S = (T + T % 2 + 4) * 441
    assert O.trim_center(torch.zeros(1, 1, S), L).shape[-1] == 132300
    y = O.remove_higher_frequency(np.random.RandomState(0).randn(L).astype(np.float32) * 0.1)
    assert y.shape[0] == 132096
    cond = O.oracle_cond(np.random.RandomState(1).randn(96076).astype(np.float32) * 0.1)
    assert cond.shape[-1] * 441 == 97902


def test_remove_higher_frequency_against_scipy():
    """Independent check of the librosa-0.10.1 stft/istft restatement (mode 1 pre-filter,
    voicefixer/base.py:87-104) with scipy.signal.stft/istft (librosa itself is not installed)."""
    from scipy import signal
    rs = np.random.RandomState(3)
    L = 30000
    t = np.arange(L) / 44100.0
    wav = (0.5 * np.sin(2 * np.pi * 300 * t) + 0.2 * np.sin(2 * np.pi * 3000 * t) + 0.02 * rs.randn(L)).astype(np.float32)
    y = O.remove_higher_frequency(wav, ratio=0.95)
    assert y.shape[0] == 512 * (L // 512)
    win = signal.get_window("hann", 2048, fftbins=True)
    _, _, Z = signal.stft(wav.astype(np.float64), window=win, nperseg=2048, noverlap=2048 - 512, boundary="zeros",
                          padded=False)
    Z = Z * win.sum()                                   # librosa scaling
    spec = np.abs(Z)
    feature = np.log10(spec + 1e-8)
    feature[feature < 0] = 0
    e = feature.sum(1)
    thr = e.sum() * 0.95
    cur, i = e[0], 0
    while i < e.shape[0] and cur < thr:
        cur += e[i + 1]
        i += 1
    assert 0 < i < 1025
    Z[i:] = 0
    _, ref = signal.istft(Z / win.sum(), window=win, nperseg=2048, noverlap=2048 - 512, boundary=True)
    n = min(len(ref), len(y))
    assert abs(len(ref) - len(y)) <= 512
    assert np.max(np.abs(ref[:n] - y[:n])) < 2e-4


def test_slaney_basis_matches_torchaudio_formula():
    """oracle()'s mel basis = melscale_fbanks(norm='slaney', mel_scale='htk') transposed
    (voicefixer/tools/mel_scale.py:226-229 is the same formula in fp32)."""
    from voicefixer_b200 import synthetic
    fb = synthetic.htk_mel_fb().double()
    m_pts = torch.linspace(0.0, 2595.0 * np.log10(1.0 + 22050.0 / 700.0), 130, dtype=torch.float64)
    f_pts = 700.0 * (10 ** (m_pts / 2595.0) - 1.0)
    enorm = 2.0 / (f_pts[2:130] - f_pts[:128])
    ref = (fb * enorm[None, :]).t().numpy()
    assert np.max(np.abs(O.slaney_htk_mel_basis() - ref)) < 2e-6


def _live_pin():
    """tests/golden/live_pin.py: regenerates the inputs of live_pin.npz and runs the oracle on them."""
    spec = importlib.util.spec_from_file_location("live_pin", os.path.join(GOLDEN, "live_pin.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_slaney_basis_matches_the_reference_melscale_fbanks():
    """The one independent cross-check of Vocoder.oracle()'s mel basis that exists offline (librosa is absent): the
    reference's OWN implementation of the same filterbank, melscale_fbanks(..., norm="slaney", mel_scale="htk")
    (voicefixer/tools/mel_scale.py:173-238, Slaney branch :226-229), run unmodified by tests/golden/live_pin.py and
    stored in live_pin.npz -- against both the oracle's and the product's (wavio) restatement of librosa.filters.mel."""
    ref = _live_pin().stored_filterbank(golden("live_pin")).T      # (128, 1025) like librosa.filters.mel
    from voicefixer_b200 import wavio
    assert ref.shape == (128, 1025)
    scale = float(np.max(np.abs(ref)))
    assert np.max(np.abs(O.slaney_htk_mel_basis() - ref)) < 2e-6 * max(1.0, scale / 1e-2)
    assert np.max(np.abs(wavio.slaney_htk_mel_basis() - ref)) < 2e-6 * max(1.0, scale / 1e-2)
    assert np.max(np.abs(wavio.slaney_htk_mel_basis() - ref)) / scale < 1e-4      # fp32 (reference) vs float64 build


@pytest.mark.timeout(900)
def test_oracle_live_against_unmodified_reference_on_fresh_inputs(states):
    """The oracle against what the unmodified reference (its own VoiceFixer() / Vocoder() loading seeded synthetic
    checkpoints) computed on inputs that are not in the other fixtures -- analysis at the 64-frame grid edges, vocoder
    at odd / even T, restore_inmem modes 0 and 2 (with the dropout masks the reference drew), and the your_vocoder_func
    hook.  tests/golden/live_pin.py ran the reference and stored a fixed sample of every output in live_pin.npz."""
    lp, g = _live_pin(), golden("live_pin")
    x = lp.inputs(int(g["seed"]))
    for k, v in x.items():                                              # the inputs the reference saw
        assert np.isclose(np.sum(np.asarray(v, np.float64)), g["insum_" + k], rtol=1e-12, atol=0), k
    out = lp.oracle_outputs(x, states[0], states[1], lp.stored_masks(g))
    assert set(out) == {"analysis_T2", "analysis_T64", "analysis_T128", "analysis_T257", "vocoder_T5", "vocoder_T12",
                        "restore_mode0_1.3s", "restore_mode2_1.6s", "hook_mel", "hook_out"}
    for k, v in out.items():
        assert v.shape == tuple(g["shape_" + k]), k
        err = rel_rms(lp.sample(v), g["ref_" + k])
        assert err < (2e-5 if k != "hook_mel" else 5e-5), (k, err)     # fp32 restatement: same ops, same order
