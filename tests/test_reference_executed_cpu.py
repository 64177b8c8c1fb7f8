"""The reference's OWN featurizer / augmentation code, executed and stored, against the oracle (CPU tests).

`open_seq2seq/data/speech2text/speech_utils.py` is plain NumPy around three third-party packages that are absent
from this image (resampy, librosa, h5py).  It is loaded BY PATH from a checkout of it (never copied) with those
imports replaced by stand-ins whose numerical primitives are the oracle's restatements of the published algorithms
(`resampy.resample` -> oracle.augment.resample, `librosa.core.stft` -> oracle.featurizer.stft_power,
`librosa.filters.mel` -> oracle.featurizer.mel_filterbank; python_speech_features' `sigproc.framesig`,
`sigproc.logpowspec`, `logfbank`, `mfcc` -> oracle.featurizer.psf_*).  Everything else that runs is the reference itself:
normalisation and gain, the order and kind of every random draw (stretch factor, noise level, noise, dither,
spec-augment bands), pre-emphasis, the log / floor constants, the normalisation axes, the mask application.  The
oracle's own composition of those steps -- the thing every GPU parity test compares with -- has to reproduce its
output from the same random stream.  For the psf backend the reference's re-quantisation to int16, its padding rule, the
arguments it passes (Hann frames for `spectrogram` only, nfilt = 2 F and ceplifter = 2 F for `mfcc`, highfreq) and its
global normalisation are what is checked.

The reference's outputs are stored under tests/golden/reference/reference_speech_utils.json (tests/refpins.py;
OS2S_REFERENCE_ROOT re-runs the reference and rewrites them); tools/make_golden_reference_draws.py stores its draws
as a fixture of their own (tests/golden/reference_augmentation_draws.json).
"""
import importlib.util
import json
import os
import sys
import types

import numpy as np
import pytest

from oracle import augment as AU
from oracle import featurizer as FZ
from tests import refpins as RP

PINS = RP.Pins("reference_speech_utils")
_REF = {}


def load_reference_speech_utils(root):
    """open_seq2seq/data/speech2text/speech_utils.py of the reference checkout at `root`, over the stand-ins."""
    rs = types.ModuleType("resampy")

    def resample(x, sr_orig, sr_new, filter="kaiser_best"):
        assert filter == "kaiser_best"
        return AU.resample(x, sr_orig, sr_new)
    rs.resample = resample
    librosa = types.ModuleType("librosa")
    librosa.core = types.ModuleType("librosa.core")
    librosa.filters = types.ModuleType("librosa.filters")

    def stft(signal, n_fft, hop_length, win_length, center=True, window=np.hanning):
        assert center and window is np.hanning
        return np.sqrt(FZ.stft_power(signal, n_fft=n_fft, hop=hop_length, win_length=win_length))
    librosa.core.stft = stft
    librosa.filters.mel = lambda sr, n_fft, n_mels, fmin, fmax: FZ.mel_filterbank(sr, n_fft, n_mels=n_mels, fmin=fmin,
                                                                                  fmax=fmax)
    # python_speech_features (v0.6) entry points the reference calls, from the oracle's restated primitives
    psf = types.ModuleType("python_speech_features")
    psf.sigproc = types.ModuleType("python_speech_features.sigproc")
    psf.sigproc.framesig = lambda sig, frame_len, frame_step, winfunc: FZ._psf_frames(
        np.asarray(sig, dtype=np.float64), frame_len, frame_step, winfunc)
    psf.sigproc.logpowspec = lambda frames, NFFT: FZ.psf_logpowspec(frames, NFFT)

    def logfbank(signal, samplerate, winlen, winstep, nfilt, nfft, lowfreq, highfreq, preemph):
        return FZ.psf_log_fbank(np.asarray(signal, dtype=np.float64), samplerate, int(round(winlen * samplerate)),
                                int(round(winstep * samplerate)), nfilt, nfft, lowfreq, highfreq, preemph)

    def mfcc(signal, samplerate, winlen, winstep, numcep, nfilt, nfft, lowfreq, highfreq, preemph, ceplifter,
             appendEnergy):
        assert not appendEnergy
        return FZ.psf_mfcc(np.asarray(signal, dtype=np.float64), samplerate, int(round(winlen * samplerate)),
                           int(round(winstep * samplerate)), numcep, nfilt, nfft, lowfreq, highfreq or samplerate / 2.0,
                           preemph, ceplifter)
    psf.logfbank, psf.mfcc = logfbank, mfcc
    stand_ins = {"resampy": rs, "librosa": librosa, "librosa.core": librosa.core, "librosa.filters": librosa.filters,
                 "python_speech_features": psf, "python_speech_features.sigproc": psf.sigproc,
                 "h5py": types.ModuleType("h5py")}
    saved = {k: sys.modules.get(k) for k in stand_ins}
    sys.modules.update(stand_ins)
    try:
        spec = importlib.util.spec_from_file_location(
            "_reference_speech_utils", os.path.join(root, "open_seq2seq", "data", "speech2text", "speech_utils.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return mod


def ref(root):
    if root not in _REF:
        _REF[root] = load_reference_speech_utils(root)
    return _REF[root]


@pytest.fixture(scope="module")
def toy_signal(golden_dir):
    import scipy.io.wavfile as wavfile
    _, sig = wavfile.read(os.path.join(golden_dir, "toy_speech_data", "wav_files", "46gc040q.wav"))
    return sig.astype(np.int16)[:24000]


AUGS = [
    {"speed_perturbation_ratio": [0.9, 1.0, 1.1]},                                   # the Jasper recipe
    {"speed_perturbation_ratio": 0.1},                                               # uniform in [0.9, 1.1]
    {"speed_perturbation_ratio": [0.9, 1.1], "noise_level_min": -90, "noise_level_max": -46},
    {"noise_level_min": -60, "noise_level_max": -50},
]


def test_normalize_and_preemphasis_are_the_references(toy_signal):
    x = toy_signal.astype(np.float32)
    assert RP.equal(FZ.normalize_signal(x), PINS("normalize_signal", lambda root: ref(root).normalize_signal(x)))
    assert RP.equal(FZ.normalize_signal(x, 0.5),
                    PINS("normalize_signal/gain=0.5", lambda root: ref(root).normalize_signal(x, 0.5)))
    assert RP.equal(FZ.preemphasis(x, coeff=0.97),
                    PINS("preemphasis", lambda root: ref(root).preemphasis(x, coeff=0.97)))


@pytest.mark.parametrize("aug", AUGS)
def test_augment_audio_signal_draws_and_output_match_the_executed_reference(toy_signal, aug):
    x = FZ.normalize_signal(toy_signal.astype(np.float32))
    for seed in range(6):
        def reference(root):
            np.random.seed(seed)
            return ref(root).augment_audio_signal(x.copy(), 16000, aug)
        want = PINS("augment_audio_signal/%s/%d" % (sorted(aug.items()), seed), reference)
        got = AU.augment_audio_signal(x.copy(), 16000, aug, rng=np.random.RandomState(seed))
        assert got.shape == want.shape
        assert RP.close(got, want, rtol=0, atol=1e-6), (seed, RP.max_dev(got, want))
        # the host-side draws the GPU data layer consumes: same stream, same order
        sr_new, amp = AU.draw_augmentation(len(x), 16000, aug, np.random.RandomState(seed))
        if "speed_perturbation_ratio" in aug:
            assert AU.resample_out_len(len(x), 16000, sr_new) == len(want)
        else:
            assert sr_new <= 0 and len(want) == len(x)


@pytest.mark.parametrize("aug", [None, {"speed_perturbation_ratio": [0.9, 1.0, 1.1]},
                                 {"speed_perturbation_ratio": [0.9, 1.0, 1.1], "n_freq_mask": 2, "n_time_mask": 2,
                                  "width_freq_mask": 6, "width_time_mask": 10}])
@pytest.mark.parametrize("norm_per_feature", [True, False])
def test_logfbank_pipeline_matches_the_executed_reference(toy_signal, aug, norm_per_feature):
    """get_speech_features_librosa (speech_utils.py:322-441) as the Jasper configs call it (logfbank, 20 ms / 10 ms,
    dither 1e-5, per-feature normalisation) vs the oracle's composition: normalise -> augment -> dither ->
    logfbank -> spec-augment masks, fed from the same np.random stream."""
    for seed in (0, 3):
        def reference(root):
            np.random.seed(seed)
            f, dur = ref(root).get_speech_features_librosa(
                toy_signal, 16000, 64, features_type="logfbank", window_size=20e-3, window_stride=10e-3,
                augmentation=aug, dither=1e-5, norm_per_feature=norm_per_feature)
            return {"features": f, "zeros": f == 0, "duration": dur}
        want = PINS("logfbank/%s/norm_per_feature=%s/%d" % (sorted(aug.items()) if aug else None, norm_per_feature,
                                                             seed), reference)
        dur = want["duration"]
        rng = np.random.RandomState(seed)
        x = FZ.normalize_signal(toy_signal.astype(np.float32))
        if aug:
            x = AU.augment_audio_signal(x, 16000, aug, rng=rng)
        # (logfbank_features normalises its input again: gain 1 keeps the augmented signal as it is)
        x = x + 1e-5 * rng.randn(*x.shape)
        s = FZ.preemphasis(x, coeff=0.97)
        S = FZ.stft_power(s, n_fft=512, hop=160, win_length=320)
        f = np.log(np.dot(FZ.mel_filterbank(16000, 512, n_mels=64, fmin=0, fmax=8000), S) + 1e-20).T
        axis = 0 if norm_per_feature else None
        f = (f - np.mean(f, axis=axis)) / np.std(f, axis=axis)
        if aug:
            f = AU.apply_spec_masks(f, AU.draw_spec_masks(f.shape[0], 64, aug, rng))
        assert want["features"].shape == f.shape and abs(dur - len(x) / 16000.0) < 1e-12
        assert RP.close(f, want["features"], rtol=0, atol=2e-4), (seed, RP.max_dev(f, want["features"]))
        if aug and aug.get("n_time_mask"):
            assert RP.equal(f == 0, want["zeros"])         # the same bands are masked


def test_oracle_logfbank_features_is_that_composition(toy_signal):
    """oracle.featurizer.logfbank_features (what the GPU featurizer tests compare with) == the composition above."""
    rng = np.random.RandomState(5)
    got, _ = FZ.logfbank_features(toy_signal, dither=1e-5, rng=rng)
    rng = np.random.RandomState(5)
    x = FZ.normalize_signal(toy_signal.astype(np.float32))
    x = x + 1e-5 * rng.randn(*x.shape)
    S = FZ.stft_power(FZ.preemphasis(x), n_fft=512, hop=160, win_length=320)
    f = np.log(np.dot(FZ.mel_filterbank(16000, 512, n_mels=64, fmin=0, fmax=8000), S) + 1e-20).T
    f = (f - f.mean(axis=0)) / f.std(axis=0)
    assert np.allclose(got, f, atol=1e-9)


def test_committed_draw_fixture_matches_the_executed_reference(golden_dir):
    """tests/golden/reference_augmentation_draws.json was written by tools/make_golden_reference_draws.py from the
    reference's own augment_audio_signal; it must still describe what the reference does.  Only with
    OS2S_REFERENCE_ROOT set does this run the reference; replaying the stored answers, it checks that the two stored
    records of those draws (that fixture and tests/golden/reference/) agree, and exercises no code of this project."""
    path = os.path.join(golden_dir, "reference_augmentation_draws.json")
    fx = json.load(open(path))
    x = np.zeros(fx["n_samples"], dtype=np.float32)

    def lengths(root):
        out = []
        for case in fx["cases"]:
            np.random.seed(case["seed"])
            out.append(len(ref(root).augment_audio_signal(x.copy(), fx["sample_freq"], case["augmentation"])))
        return out
    assert PINS("augmentation_draw_lengths", lengths) == [case["n_out"] for case in fx["cases"]]


@pytest.mark.parametrize("features_type,F,fn", [("logfbank", 64, "psf_logfbank_features"),
                                               ("spectrogram", 96, "psf_spectrogram_features"),
                                               ("mfcc", 13, "psf_mfcc_features")])
@pytest.mark.parametrize("pad_to", [8, 0])
def test_psf_pipeline_matches_the_executed_reference(toy_signal, features_type, F, fn, pad_to):
    """get_speech_features_psf (speech_utils.py:444-535), the backend of the Wave2Letter(+) configs and of the
    reference's toy tests, for its three input types."""
    for n in (24000, 23873, 16001):
        sig = toy_signal[:n]
        w = PINS("psf/%s/pad_to=%d/%d" % (features_type, pad_to, n), lambda root: dict(zip(("features", "duration"), ref(
            root).get_speech_features_psf(sig, 16000, F, pad_to=pad_to, features_type=features_type, window_size=20e-3,
                                          window_stride=10e-3, augmentation=None))))
        want, dur = w["features"], w["duration"]
        got, gdur = getattr(FZ, fn)(sig, num_features=F, pad_to=pad_to)
        assert want.shape == got.shape and dur == gdur
        assert RP.close(got, want, rtol=0, atol=1e-9), (n, RP.max_dev(got, want))
        if pad_to:
            assert want.shape[0] % pad_to == 0


@pytest.mark.parametrize("config,mode", [("jasper10x5_LibriSpeech_nvgrad.py", "eval"),
                                         ("jasper10x5_LibriSpeech_nvgrad_masks.py", "train"),
                                         ("w2lplus_large_8gpus_mp.py", "train")])
def test_per_utterance_data_path_equals_the_executed_reference(golden_dir, tmp_path, config, mode):
    """Speech2TextDataLayer._parse_audio_transcript_element (speech2text.py:401-432, the py_func behind the tf.data
    pipeline) compiled from the reference's source and run with the data-layer params of a REAL example config on the
    toy wavs: the wav is read and checked, dispatched by `backend` / `input_type` with the config's window, dither,
    num_fft, norm_per_feature, pad_to and augmentation, the transcript is encoded with the vocabulary.  The drop-in
    data layer's host side (file list, wav reader, transcript ids) and the oracle's features for those parameters
    have to agree, from the same np.random stream."""
    import ast
    import copy
    import pandas as pd
    import six
    import openseq2seq_b200.compat as compat
    compat.install()
    from open_seq2seq.data import Speech2TextDataLayer
    from open_seq2seq.utils.utils import get_base_config, nested_update

    def parse_element(root):
        path = os.path.join(root, "open_seq2seq", "data", "speech2text", "speech2text.py")
        cls = next(n for n in ast.parse(open(path).read()).body if isinstance(n, ast.ClassDef)
                   and n.name == "Speech2TextDataLayer")
        fn = next(n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name == "_parse_audio_transcript_element")
        ns = {"np": np, "six": six, "get_speech_features_from_file": ref(root).get_speech_features_from_file}
        exec(compile(ast.Module(body=[fn], type_ignores=[]), path, "exec"), ns)
        return ns["_parse_audio_transcript_element"]

    toy = os.path.join(golden_dir, "toy_speech_data")
    _, cfg, _, module = get_base_config(["--config_file=" + RP.example_config(config, tmp_path), "--mode=" + mode])
    p = copy.deepcopy(cfg.get("data_layer_params", {}))
    nested_update(p, copy.deepcopy(module[mode + "_params"]["data_layer_params"]))
    p.update(dataset_files=[os.path.join(toy, "toy_data.csv")], vocab_file=os.path.join(toy, "vocab.txt"), mode=mode,
             batch_size=2)
    dl = Speech2TextDataLayer(copy.deepcopy(p), None, 1, 0)          # the drop-in: file list, vocabulary, defaults
    rp = dict(dl.params)                                             # what the reference's constructor would hold
    rp.update(bpe=False, dtype=types.SimpleNamespace(as_numpy_dtype=lambda: np.float32), mel_basis=None)
    me = types.SimpleNamespace(params=rp, autoregressive=False, end_index=None)
    rows = pd.read_csv(os.path.join(toy, "toy_data.csv"), encoding="utf-8")
    librosa_backend = rp.get("backend", "psf") == "librosa"
    aug = rp.get("augmentation") if mode == "train" else None
    assert bool(aug) == (config != "w2lplus_large_8gpus_mp.py" and mode == "train")
    for k in (0, 3, 7):
        wav = os.path.join(toy, rows["wav_filename"][k]) if not os.path.isabs(rows["wav_filename"][k]) \
            else rows["wav_filename"][k]
        if not os.path.exists(wav):
            wav = os.path.join(toy, "wav_files", os.path.basename(rows["wav_filename"][k]))
        tr = rows["transcript"][k]

        def reference(root):
            np.random.seed(11 + k)
            out = parse_element(root)(me, (wav.encode("utf-8"), tr.encode("utf-8")))
            return dict(zip(("src", "src_len", "tgt", "tgt_len", "dur"), out))
        want = PINS("parse_audio_transcript_element/%s/%s/%d" % (config, mode, k), reference)
        src, src_len, tgt_len, dur = want["src"], want["src_len"].values, want["tgt_len"].values, want["dur"].values
        # host side of the drop-in
        sig, ids = dl._load((wav, tr))
        assert RP.equal(ids, want["tgt"]) and int(tgt_len[0]) == len(ids)
        # the oracle with this config's parameters, same random stream
        rng = np.random.RandomState(11 + k)
        if librosa_backend:
            x = FZ.normalize_signal(sig.astype(np.float32))
            if aug:
                x = AU.augment_audio_signal(x, 16000, aug, rng=rng)
            if rp.get("dither", 0.0) > 0:
                x = x + rp["dither"] * rng.randn(*x.shape)
            S = FZ.stft_power(FZ.preemphasis(x), n_fft=FZ.num_fft_for(rp["window_size"], 16000),
                              hop=int(16000 * rp["window_stride"]), win_length=int(16000 * rp["window_size"]))
            f = np.log(np.dot(FZ.mel_filterbank(16000, 512, n_mels=rp["num_audio_features"], fmin=0, fmax=8000), S)
                       + 1e-20).T
            axis = 0 if rp.get("norm_per_feature", False) else None
            f = (f - np.mean(f, axis=axis)) / np.std(f, axis=axis)
            if aug:
                f = AU.apply_spec_masks(f, AU.draw_spec_masks(f.shape[0], rp["num_audio_features"], aug, rng))
            want_dur = len(x) / 16000.0
        else:
            assert rp["input_type"] == "logfbank"
            f, want_dur = FZ.psf_logfbank_features(sig, num_features=rp["num_audio_features"],
                                                   pad_to=rp.get("pad_to", 8))
        assert src.shape == f.shape and int(src_len[0]) == f.shape[0]
        assert RP.close(f, src, rtol=0, atol=3e-4), (config, k, RP.max_dev(f, src))
        assert abs(float(dur[0]) - want_dur) < 1e-6
