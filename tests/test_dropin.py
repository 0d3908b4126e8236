"""SURVEY.md 8(f)1 -- the reference's OWN callers of the path drive the B200 implementation, unmodified:

  * `FastDiffTask.build_model / test_step` (modules/FastDiff/task/FastDiff.py:16-42, 60-119) from the reference YAML, fed by the
    reference's own inference data path: `.npy` mels in `test_mel_dir` -> `VocoderDataset.load_mel_inputs` -> `collater`
    (tasks/vocoder/dataset_utils.py:186-204, 100-160 -- which DROPS the last mel frame at inference, :114-125) -> `test_step` -> wav file;
  * the vocoder registry (vocoders/base_vocoder.py:3-40): `register_vocoder(FastDiffVocoder)`, `get_vocoder_cls(hparams)` by name and by
    dotted path, `spec2wav(mel [T, 80])` as tasks/tts/tts_base.py:254,284 call it.

The reference is imported from the checkout named by FD_REFERENCE_ROOT or from the bytecode build oracle/_ref that __graft_entry__.build()
makes of a reachable checkout (oracle/stage_reference.py); the task test reads the reference's YAML configs, so it needs the checkout.
Where neither is reachable (a GPU machine without the reference), these tests skip.
CPU variant: through the emulation build of the CUDA source; `-m gpu` variant: the real library on cuda:0."""
import os
import sys
import types

import numpy as np
import pytest
import torch

N4 = [3.2176e-04, 2.5743e-03, 2.5376e-02, 7.0414e-01]


def _reference(device, monkeypatch, configs=False):
    from oracle import refimport
    root = refimport.reference_checkout() if configs else refimport.reference_root()
    if root is None:
        pytest.skip("needs the reference's own code" + (" and YAML configs" if configs else "") + ": no checkout of it is reachable")
    refimport.stub_missing_deps()
    if device == "cpu":
        monkeypatch.setattr(torch.Tensor, "cuda", lambda self, *a, **k: self)
        monkeypatch.setattr(torch.nn.Module, "cuda", lambda self, *a, **k: self)
    else:
        refimport.shim_cuda_to_cpu(False)
    if root not in sys.path:
        sys.path.insert(0, root)
    monkeypatch.chdir(root)                                   # YAML base_config paths are relative
    return root


def _run_task(tmp_path, device, lib_path, synth, monkeypatch):
    import warnings
    _reference(device, monkeypatch, configs=True)
    from fastdiff_b200.synthetic import make_inputs
    from oracle import fastdiff_oracle as O
    mel_dir = tmp_path / "mels"
    mel_dir.mkdir()
    Tm = 3 if device == "cpu" else 41
    _, mel = make_inputs(1, Tm, 5)
    np.save(mel_dir / "utt0.npy", mel[0].t().contiguous().numpy())          # [T', 80] as the reference's mel files are
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from utils.hparams import hparams, set_hparams
        set_hparams(config="modules/FastDiff/config/FastDiff.yaml", exp_name="",
                    hparams_str=f"work_dir={tmp_path},N=4,test_mel_dir={mel_dir},use_wav=False", print_hparams=False)
        import fastdiff_b200 as fb
        from fastdiff_b200.plugin import patch_reference_task
        TaskCls = patch_reference_task()
        from tasks.vocoder.dataset_utils import VocoderDataset
        import utils as ref_utils
    assert hparams["task_cls"] == "modules.FastDiff.task.FastDiff.FastDiffTask"
    task = TaskCls()
    model = task.build_model()
    assert isinstance(model, fb.FastDiff) and task.diffusion_hyperparams["T"] == 1000
    sd, W = synth
    model.load_state_dict(sd)
    if device == "cpu":
        model._lib_path = lib_path
    else:
        task.cuda()
    task.trainer = types.SimpleNamespace(global_step=0)
    ds = VocoderDataset("test")                                              # the reference's own loader of `test_mel_dir`
    assert len(ds.sizes) == 1 and ds.sizes[0] == Tm
    batch = ds.collater([ds[0]])
    assert tuple(batch["mels"].shape) == (1, 80, Tm - 1) and batch["wavs"] == []     # the collater drops the last frame at inference
    assert torch.equal(batch["mels"][0], mel[0, :, : Tm - 1])
    if device != "cpu":
        batch = ref_utils.move_to_cuda(batch)
    torch.manual_seed(3)
    task.test_step(batch, 0)                                                 # unmodified reference code -> our sampler -> save_wav
    out = tmp_path / "generated_0_" / "utt0.npy_pred.wav"
    assert out.exists(), list((tmp_path / "generated_0_").iterdir())
    from scipy.io import wavfile
    sr, wav = wavfile.read(out)
    L = (Tm - 1) * 256
    assert sr == 22050 and wav.dtype == np.int16 and wav.shape[0] == L
    torch.manual_seed(3)
    dh = O.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
    ref = O.sample(W, (1, 1, L), dh, torch.FloatTensor(N4), mel[:, :, : Tm - 1])
    ref = (ref / ref.abs().max()).view(-1).numpy() * 32767
    assert np.abs(wav.astype(np.float64) - ref.astype(np.int16)).max() <= 2   # same waveform after the reference's peak-normalise + int16 cast


def _run_vocoder(device, lib_path, synth, monkeypatch):
    _reference(device, monkeypatch)
    from vocoders.base_vocoder import VOCODERS, get_vocoder_cls, register_vocoder
    from fastdiff_b200.plugin import FastDiffVocoder
    from fastdiff_b200.synthetic import make_inputs
    from oracle import fastdiff_oracle as O
    register_vocoder(FastDiffVocoder)                                        # vocoders/base_vocoder.py:6-9
    assert VOCODERS["FastDiffVocoder"] is FastDiffVocoder and VOCODERS["fastdiffvocoder"] is FastDiffVocoder
    assert get_vocoder_cls({"vocoder": "FastDiffVocoder"}) is FastDiffVocoder
    assert get_vocoder_cls({"vocoder": "fastdiff_b200.plugin.FastDiffVocoder"}) is FastDiffVocoder     # dotted path (:16-20)
    sd, W = synth
    Tm = 2 if device == "cpu" else 30
    _, mel = make_inputs(1, Tm, 6)
    voc = FastDiffVocoder(state_dict=None, device=device)
    if device == "cpu":
        voc.model._lib_path = lib_path
    voc.model.load_state_dict(sd)
    torch.manual_seed(4)
    wav = voc.spec2wav(mel[0].t().numpy())                                   # [T, 80] -> [T * hop], the BaseVocoder contract
    assert wav.shape == (Tm * 256,) and wav.dtype == np.float32
    torch.manual_seed(4)
    dh = O.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
    ref = O.sample(W, (1, 1, Tm * 256), dh, torch.FloatTensor(N4), mel).view(-1)
    assert np.abs(wav - ref.numpy()).max() < 5e-4
    torch.manual_seed(4)
    w16 = voc.spec2wav(mel[0].t().numpy(), int16=True)                       # only int16 leaves the device
    assert w16.dtype == np.int16 and w16.shape == (Tm * 256,)
    r = ref / ref.abs().max()
    a = r.numpy().copy()
    a *= 32767
    assert np.abs(w16.astype(np.int64) - a.astype(np.int16)).max() <= 2


def test_reference_task_from_mel_dir_cpu(tmp_path, emu_lib, synth, monkeypatch):
    _run_task(tmp_path, "cpu", emu_lib, synth, monkeypatch)


def test_reference_vocoder_registry_cpu(emu_lib, synth, monkeypatch):
    _run_vocoder("cpu", emu_lib, synth, monkeypatch)


@pytest.mark.gpu
def test_reference_task_from_mel_dir_gpu(tmp_path, cuda_lib, synth, monkeypatch):
    _run_task(tmp_path, "cuda", None, synth, monkeypatch)


@pytest.mark.gpu
def test_reference_vocoder_registry_gpu(cuda_lib, synth, monkeypatch):
    _run_vocoder("cuda", None, synth, monkeypatch)
