"""Pins the oracle and the host-side code to the UNMODIFIED reference: tests/golden/reference_cpu.npz holds the reference's own
outputs (CPU, fp32) for the inputs below, recorded by tests/golden/make_golden.py."""
import os

import numpy as np
import pytest
import torch

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LVC_STRIDE = 23          # make_golden.LVC_STRIDE


@pytest.fixture(scope="module")
def ref():
    return {k: torch.from_numpy(v) if v.dtype.kind == "f" else v for k, v in np.load(os.path.join(G, "reference_cpu.npz")).items()}


def test_denoiser_matches_reference(ref, synth):
    from fastdiff_b200.synthetic import make_inputs
    from oracle import fastdiff_oracle as O
    sd, W = synth
    for B, Tm, seed in ((2, 12, 0), (1, 1, 1), (3, 5, 2)):
        x, mel = make_inputs(B, Tm, seed)
        t = torch.tensor([7.413235, 498.0537, 23.46759][:B]).reshape(B, 1)
        o = O.denoise(W, x, mel, t)
        assert (ref[f"eps_{B}_{Tm}_{seed}"] - o).abs().max() < 2e-5


def test_lvc_closed_form_matches_reference(ref):
    from oracle import fastdiff_oracle as O
    torch.manual_seed(0)
    for hop, Tm in ((256, 3), (64, 5), (8, 7)):
        x = torch.randn(2, 32, hop * Tm)
        k = torch.randn(2, 32, 64, 3, Tm)
        b = torch.randn(2, 64, Tm)
        r = ref[f"lvc_{hop}_{Tm}"]
        assert (r - O.lvc(x, k, b, hop).flatten()[::LVC_STRIDE]).abs().max() < 5e-5


def test_sampler_matches_reference(ref, synth):
    from fastdiff_b200.synthetic import make_inputs
    from oracle import fastdiff_oracle as O
    sd, W = synth
    _, mel = make_inputs(1, 4, 5)
    dh = O.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
    sched = [3.2176e-04, 2.5743e-03, 2.5376e-02, 7.0414e-01]
    for ddim in (False, True):
        r = ref["seq_ddim" if ddim else "seq_ddpm"]
        torch.manual_seed(5)
        o = O.sample(W, (1, 1, 1024), dh, torch.FloatTensor(sched), mel, ddim=ddim, return_sequence=True)
        assert len(r) == len(o)
        for a, b in zip(r, o):
            assert (a - b).abs().max() < 1e-4


def test_host_tables_bit_identical_to_reference(ref):
    """The product's vectorised host prologue returns the very floats the reference's python loops return."""
    import fastdiff_b200 as fb
    g = np.load(os.path.join(G, "tables.npz"))
    beta = torch.linspace(1e-6, 0.01, 1000)
    b = fb.compute_hyperparams_given_schedule(beta.clone())
    assert torch.equal(torch.from_numpy(g["alpha"]), b["alpha"]) and torch.equal(torch.from_numpy(g["sigma"]), b["sigma"]) and b["T"] == 1000
    for al, step in zip(ref["map_alpha"].tolist(), ref["map_step"].tolist()):
        assert step == fb.map_noise_scale_to_time_step(torch.tensor(al), b["alpha"])
    st = torch.tensor([[0.0], [3.5], [999.0]])
    assert torch.equal(ref["embed"], fb.calc_diffusion_step_embedding(st, 128))


def test_state_dict_keys_match_reference(ref):
    import fastdiff_b200 as fb
    m = fb.FastDiff().state_dict()
    shapes = [tuple(int(d) for d in s.split(",")) for s in ref["sd_shapes"]]
    assert list(ref["sd_keys"]) == list(m.keys())
    assert all(tuple(m[k].shape) == s for k, s in zip(ref["sd_keys"], shapes))
    # a state dict of the reference's keys and shapes loads strictly, and the packer accepts it
    g = torch.Generator().manual_seed(0)
    r = {k: torch.randn(s, generator=g) * 0.1 for k, s in zip(ref["sd_keys"], shapes)}
    fb.FastDiff().load_state_dict(r, strict=True)
    from fastdiff_b200.weights import pack_state_dict
    assert pack_state_dict(r).nbytes > 60e6
