"""Import the UNMODIFIED reference (test / benchmark infrastructure only -- never imported by ``fastdiff_b200/``).

``reference_root()`` = the checkout named by ``FD_REFERENCE_ROOT``, else the bytecode build ``oracle/_ref`` (oracle/stage_reference.py),
else None; ``reference_checkout()`` = a source checkout with the YAML configs: ``FD_REFERENCE_ROOT``, else the one ``oracle/_ref`` was
built from, if it is still reachable.  ``load(device)`` puts it on ``sys.path`` and returns the hot-path symbols.  The reference hard-codes ``.cuda()``
(util.py:68,91,217,427); for a CPU run ``torch.Tensor.cuda`` is shimmed to identity (SURVEY.md 8c) -- nothing else is touched.
The task-level import chain additionally needs packages that are absent from this image (chardet, librosa, resemblyzer); they are
stubbed with empty modules -- none of them is used by ``test_step`` / ``spec2wav``.
"""
from __future__ import annotations

import os
import sys
import types
import warnings

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILT = os.path.join(ROOT, "oracle", "_ref")
_orig_tensor_cuda = torch.Tensor.cuda


def reference_root():
    for c in (os.environ.get("FD_REFERENCE_ROOT"), BUILT):
        if c and os.path.isdir(os.path.join(c, "modules", "FastDiff", "module")):
            return c
    return None


def reference_checkout():
    c = os.environ.get("FD_REFERENCE_ROOT")
    if not c:
        try:
            with open(os.path.join(BUILT, "SOURCE")) as fh:
                c = fh.read().strip()
        except OSError:
            return None
    return c if os.path.isfile(os.path.join(c, "modules", "FastDiff", "config", "FastDiff.yaml")) else None


def shim_cuda_to_cpu(on: bool = True):
    """The reference's `.cuda()` calls become identities (CPU run) or are restored."""
    torch.Tensor.cuda = (lambda self, *a, **k: self) if on else _orig_tensor_cuda


# packages the reference's task / data-prep import chain pulls in that are absent from this image, with the attributes its
# `from X import name` statements need.  None of them is used by the code the tests run (test_step, the mel-dir loader, spec2wav).
_STUBS = {
    "chardet": (), "librosa": (), "librosa.filters": (), "resemblyzer": ("VoiceEncoder",), "parselmouth": (), "skimage": (),
    "skimage.transform": ("resize",), "webrtcvad": (), "pyloudnorm": (), "scipy.ndimage.morphology": ("binary_dilation",),
    "matplotlib": (), "matplotlib.pyplot": (), "h5py": (), "pyworld": (), "g2p_en": (), "soundfile": (), "pypinyin": (), "textgrid": (),
}


def stub_missing_deps():
    import importlib
    for name, attrs in _STUBS.items():
        if name in sys.modules:
            continue
        try:
            importlib.import_module(name)
        except Exception:
            mod = types.ModuleType(name)
            for a in attrs:
                setattr(mod, a, object)
            sys.modules[name] = mod
            if "." in name:
                parent, child = name.rsplit(".", 1)
                if parent in sys.modules and not hasattr(sys.modules[parent], child):
                    setattr(sys.modules[parent], child, mod)


def load(device: str = "cpu"):
    """-> namespace(root, FastDiff, sampling_given_noise_schedule, compute_hyperparams_given_schedule, util, modules)."""
    root = reference_root()
    if root is None:
        raise FileNotFoundError("reference not available: set FD_REFERENCE_ROOT to a checkout of it (oracle/stage_reference.py builds oracle/_ref)")
    if root not in sys.path:
        sys.path.insert(0, root)
    shim_cuda_to_cpu(device == "cpu")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from modules.FastDiff.module import modules as ref_modules
        from modules.FastDiff.module import util as ref_util
        from modules.FastDiff.module.FastDiff_model import FastDiff
    return types.SimpleNamespace(root=root, FastDiff=FastDiff, util=ref_util, modules=ref_modules,
                                 sampling_given_noise_schedule=ref_util.sampling_given_noise_schedule,
                                 compute_hyperparams_given_schedule=ref_util.compute_hyperparams_given_schedule)
