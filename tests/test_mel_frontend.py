"""Mel front-end (SURVEY.md 8f.3): oracle vs an independent implementation of the same published algorithm, host filter table vs
oracle, and the CUDA source (emulated on CPU / on the GPU) vs oracle."""
import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu


def _signals():
    rng = np.random.default_rng(3)
    t = np.arange(30000) / 22050.0
    chirp = 0.5 * np.sin(2 * np.pi * (100 + 3000 * t) * t)
    voiced = sum(0.3 / k * np.sin(2 * np.pi * 140 * k * t) for k in range(1, 12)) * np.hanning(t.size)
    noise = 0.05 * rng.standard_normal(t.size)
    click = np.zeros(9000); click[4000] = 0.9
    return [s.astype(np.float32) for s in (chirp + noise, voiced, noise * 0.01, click, (chirp + voiced)[:7777])]


def test_oracle_matches_an_independent_implementation():
    """librosa is absent: pin the restatement to torchaudio's librosa-compatible filter bank and torch.stft."""
    import torchaudio
    from oracle import mel_oracle as M
    fb = M.mel_filterbank()
    fb_ta = torchaudio.functional.melscale_fbanks(513, 80.0, 7600.0, 80, 22050, norm="slaney", mel_scale="slaney").T.numpy()
    assert np.abs(fb - fb_ta).max() < 2e-7
    for w in _signals():
        st = torch.stft(torch.from_numpy(w), 1024, 256, 1024, torch.hann_window(1024, periodic=True), center=True, pad_mode="constant",
                        return_complex=True).abs().numpy()
        spc = M.stft_mag(w)
        assert spc.shape == st.shape == (513, 1 + len(w) // 256)
        assert np.abs(spc - st).max() < 1e-5 * max(1.0, spc.max())
        wp, mel = M.wav2mel(w)
        assert mel.shape == (80, 1 + len(w) // 256) and wp.shape == (mel.shape[1] * 256,)
        assert mel.min() >= -6.001


def test_host_filter_table_equals_oracle():
    from fastdiff_b200.mel import mel_filter_table
    from oracle import mel_oracle as M
    table, ranges = mel_filter_table()
    assert np.array_equal(table, M.mel_filterbank())
    assert np.array_equal(ranges, M.filterbank_ranges(M.mel_filterbank()))


def _check(engine, tol):
    from fastdiff_b200.mel import wav2mel
    from oracle import mel_oracle as M
    for w in _signals():
        wp, mel = wav2mel(engine, torch.from_numpy(w))
        wp_ref, mel_ref = M.wav2mel(w)
        assert np.array_equal(wp.cpu().numpy()[0], wp_ref)
        got = mel.cpu().numpy()[0]
        assert got.shape == mel_ref.shape
        # compare in the linear domain relative to the frame's loudest band (fp32 FFT vs the reference's float64 rfft), and in the
        # log domain wherever the band is not buried 60 dB under the frame maximum
        lin, lin_ref = 10.0 ** got.astype(np.float64), 10.0 ** mel_ref.astype(np.float64)
        scale = np.maximum(lin_ref.max(axis=0, keepdims=True), 1e-6)
        assert (np.abs(lin - lin_ref) / scale).max() < tol
        loud = lin_ref > 1e-3 * scale
        assert np.abs(got - mel_ref)[loud].max() < 1e-3


def test_emulated_cuda_source_matches_oracle(emu_lib):
    from fastdiff_b200.engine import Engine
    _check(Engine(device="cpu", lib_path=emu_lib), 2e-6)


@gpu
def test_gpu_mel_frontend_matches_oracle(cuda_lib):
    from fastdiff_b200.engine import Engine
    _check(Engine(device="cuda:0"), 2e-6)
    # batch of 2 with the same content == single (independent items)
    from fastdiff_b200.mel import wav2mel
    w = torch.from_numpy(np.stack([_signals()[0][:20000], _signals()[1][:20000]]))
    eng = Engine(device="cuda:0")
    _, m2 = wav2mel(eng, w)
    _, m0 = wav2mel(eng, w[0])
    assert torch.equal(m2[0], m0[0])


def test_vocoder_wav2spec_matches_oracle(emu_lib, tmp_path):
    """`BaseVocoder.wav2spec` shape: (wav, mel [T,80]) from a wav FILE, through the emulated CUDA source; a synthetic signal and an
    excerpt of the reference's own example recording (egs/audios/LJ001-0001_gt.wav, stored under tests/golden)."""
    import os
    from scipy.io import wavfile
    from fastdiff_b200.engine import Engine
    from fastdiff_b200.plugin import FastDiffVocoder
    from oracle import mel_oracle as M
    eng = Engine(device="cpu", lib_path=emu_lib)
    pcm = (np.clip(_signals()[1], -1, 1) * 32767).astype(np.int16)
    fn = tmp_path / "a.wav"
    wavfile.write(fn, 22050, pcm)
    files = [str(fn), os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "LJ001-0001_gt_excerpt.wav")]
    for f in files:
        wav, mel = FastDiffVocoder.wav2spec(f, engine=eng)
        sr, data = wavfile.read(f)
        x = data.astype(np.float32) / 32768.0
        w_ref, mel_ref = M.wav2mel(x)
        assert mel.shape == (1 + len(x) // 256, 80) and wav.shape == (mel.shape[0] * 256,)
        assert np.array_equal(wav, w_ref)
        loud = 10.0 ** mel_ref > 1e-3 * (10.0 ** mel_ref).max(axis=0, keepdims=True)
        assert np.abs(mel.T - mel_ref)[loud].max() < 1e-3
    with pytest.raises(ValueError):
        wavfile.write(tmp_path / "b.wav", 16000, pcm)
        FastDiffVocoder.wav2spec(str(tmp_path / "b.wav"), engine=eng)
