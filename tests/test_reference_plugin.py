"""Drop-in check with the UNMODIFIED reference task code (oracle/refimport.py: reference_checkout): `tasks/run.py`'s import chain resolves,
`FastDiffTask.build_model` builds the B200 model from the reference's own YAML hparams, and `test_step` drives our sampler
(through the CPU-emulated CUDA source, so this runs without a GPU) and writes the wav like the reference does."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import refimport

REF = refimport.reference_checkout()
pytestmark = pytest.mark.skipif(REF is None, reason="needs the reference's own task code and configs: no checkout of it is reachable")


def _stub_missing_deps():
    # the task-level chain imports packages that are not installed here (SURVEY.md 8c); none is used by test_step
    for name in ("chardet", "librosa", "librosa.filters", "resemblyzer"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["resemblyzer"].VoiceEncoder = object
    sys.modules["librosa"].filters = sys.modules["librosa.filters"]


def test_reference_task_runs_on_b200_path(tmp_path, emu_lib, synth, monkeypatch):
    _stub_missing_deps()
    torch.Tensor.cuda = lambda self, *a, **k: self          # no GPU here; the reference hard-codes .cuda()
    monkeypatch.setattr(torch.nn.Module, "cuda", lambda self, *a, **k: self)
    if REF not in sys.path:
        sys.path.insert(0, REF)
    monkeypatch.chdir(REF)                                   # YAML base_config paths are relative
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from utils.hparams import hparams, set_hparams
        set_hparams(config="modules/FastDiff/config/FastDiff.yaml", exp_name="", hparams_str=f"work_dir={tmp_path},N=4", print_hparams=False)
        import fastdiff_b200 as fb
        from fastdiff_b200.plugin import patch_reference_task
        TaskCls = patch_reference_task()
    assert hparams["task_cls"] == "modules.FastDiff.task.FastDiff.FastDiffTask"
    task = TaskCls()
    model = task.build_model()
    assert isinstance(model, fb.FastDiff)                    # built from the reference's hparams (task/FastDiff.py:17-29)
    assert task.diffusion_hyperparams["T"] == 1000
    sd, W = synth
    model.load_state_dict(sd)
    model._lib_path = emu_lib
    task.trainer = types.SimpleNamespace(global_step=0)
    Tm = 2
    from fastdiff_b200.synthetic import make_inputs
    _, mel = make_inputs(1, Tm, 5)
    sample = {"mels": mel, "wavs": [], "item_name": ["utt0"]}
    torch.manual_seed(3)
    task.test_step(sample, 0)                                # unmodified reference code -> our sampler -> save_wav
    out = tmp_path / "generated_0_" / "utt0_pred.wav"
    assert out.exists()
    from scipy.io import wavfile
    sr, wav = wavfile.read(out)
    assert sr == 22050 and wav.dtype == np.int16 and wav.shape[0] == Tm * 256
    # same waveform as the oracle with the same RNG stream, after the reference's peak normalisation + int16 cast
    from oracle import fastdiff_oracle as O
    torch.manual_seed(3)
    dh = O.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
    ref = O.sample(W, (1, 1, Tm * 256), dh, torch.FloatTensor([3.2176e-04, 2.5743e-03, 2.5376e-02, 7.0414e-01]), mel)
    ref = (ref / ref.abs().max()).view(-1).numpy() * 32767
    assert np.abs(wav.astype(np.float64) - ref.astype(np.int16)).max() <= 1
