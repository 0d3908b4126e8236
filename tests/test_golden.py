"""Golden vectors = outputs of the unmodified reference (tests/golden/make_golden.py).  CPU: oracle and the emulated
CUDA source against them; GPU: the real CUDA path against them."""
import os

import numpy as np
import pytest
import torch

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
N4 = [3.2176e-04, 2.5743e-03, 2.5376e-02, 7.0414e-01]


def _load(name):
    return {k: torch.from_numpy(v) for k, v in np.load(os.path.join(G, name)).items()}


def test_oracle_vs_golden_denoise(synth):
    from oracle import fastdiff_oracle as O
    _, W = synth
    g = _load("denoise_b2_t12.npz")
    eps, inter = O.denoise(W, g["x"], g["mel"], g["t"], return_intermediates=True)
    assert (eps - g["eps"]).abs().max() < 2e-5
    for n in range(3):
        assert (inter[f"down{n}"] - g[f"down{n}"]).abs().max() < 1e-5
        lvc, want = (inter[f"lvc{n}"], g[f"lvc{n}"]) if n < 2 else (inter["lvc2"][:, :, ::4], g["lvc2_sub"])
        assert (lvc - want).abs().max() < 5e-5


def test_oracle_vs_golden_sampler(synth):
    from oracle import fastdiff_oracle as O
    _, W = synth
    g = _load("sample_n4_b1_t6.npz")
    dh = O.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
    for ddim, key in ((False, "seq_ddpm"), (True, "seq_ddim")):
        torch.manual_seed(int(g["seed"]))
        seq = O.sample(W, (1, 1, 6 * 256), dh, torch.FloatTensor(N4), g["mel"], ddim=ddim, return_sequence=True)
        assert (torch.stack(seq) - g[key]).abs().max() < 1e-4


def test_tables_vs_golden():
    """Weight-free known answers (SURVEY.md 8c): schedule tables and noise-scale -> step maps, bit for bit."""
    import fastdiff_b200 as fb
    from fastdiff_b200.sampler import build_steps
    from oracle import fastdiff_oracle as O
    from tests.golden.make_golden_schedules import N_SCHEDULES
    g = _load("tables.npz")
    for impl in (fb.compute_hyperparams_given_schedule, O.compute_hyperparams_given_schedule):
        dh = impl(torch.linspace(1e-6, 0.01, 1000))
        assert torch.equal(dh["alpha"], g["alpha"]) and torch.equal(dh["sigma"], g["sigma"])
    dh = fb.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
    for N, s in N_SCHEDULES.items():
        steps, fsteps = build_steps(dh, torch.FloatTensor(s))
        assert steps == g[f"steps_{N}"].tolist()
        _, _, sg, st = O.sampler_tables(torch.FloatTensor(s), dh["alpha"])
        assert st.tolist() == torch.FloatTensor(steps).tolist()
        assert [f.sigma for f in fsteps][::-1] == g[f"sigma_infer_{N}"].tolist()
    # values quoted in SURVEY.md 8(a)/(c)
    assert np.allclose(g["steps_4"].numpy(), [7.413235, 23.467590, 74.992283, 498.053687], atol=1e-5)
    assert np.allclose(g["steps_3"].numpy(), [3.630814, 42.111882, 429.112278], atol=1e-5)
    emb = fb.calc_diffusion_step_embedding(torch.tensor([[0.0], [7.413235], [498.0537], [999.0]]), 128)
    assert torch.equal(emb, g["embed_in"])
    assert (O.step_embedding(torch.tensor([[0.0], [7.413235], [498.0537], [999.0]])) - g["embed_in"]).abs().max() == 0


def test_emulated_cuda_source_vs_golden_denoise(synth, emu_lib):
    """The CUDA kernels' source, compiled for the CPU thread-emulator (tests/cudaemu), against the reference's output."""
    import fastdiff_b200 as fb
    sd, _ = synth
    g = _load("denoise_b2_t12.npz")
    net = fb.FastDiff().eval()
    net._lib_path = emu_lib
    net.load_state_dict(sd)
    eps = net((g["x"], g["mel"], g["t"]))
    assert (eps - g["eps"]).abs().max() < 5e-5
    eng = net.engine()
    for n, T in enumerate((768, 96, 12)):
        assert (eng.debug_read(f"down{n}", 2, 12).reshape(2, 32, T) - g[f"down{n}"]).abs().max() < 1e-5
        k = eng.debug_read(f"kernels{n}", 2, 12).reshape(2, 4, 32, 64, 3, 12)[:, :, ::8, ::8]
        assert (k - g[f"kernels{n}_sub"]).abs().max() < 2e-5
        assert (eng.debug_read(f"kbias{n}", 2, 12).reshape(2, 4, 64, 12) - g[f"kbias{n}"]).abs().max() < 2e-5
    assert (eng.debug_read("lvc2", 2, 12).reshape(2, 32, 3072)[:, :, ::4] - g["lvc2_sub"]).abs().max() < 1e-4


@pytest.mark.gpu
def test_cuda_vs_golden_denoise(synth, cuda_lib):
    import fastdiff_b200 as fb
    sd, _ = synth
    g = _load("denoise_b2_t12.npz")
    net = fb.FastDiff().to("cuda:0").eval()
    net.load_state_dict(sd)
    for mode in ("fp32_simt", None):
        net.mode = mode
        eps = net((g["x"].cuda(), g["mel"].cuda(), g["t"].cuda())).cpu()
        assert (eps - g["eps"]).abs().max() < 5e-5, mode
    eng = net.engine()
    for n, T in enumerate((768, 96, 12)):
        assert (eng.debug_read(f"down{n}", 2, 12).cpu().reshape(2, 32, T) - g[f"down{n}"]).abs().max() < 1e-5
        k = eng.debug_read(f"kernels{n}", 2, 12).cpu().reshape(2, 4, 32, 64, 3, 12)[:, :, ::8, ::8]
        assert (k - g[f"kernels{n}_sub"]).abs().max() < 2e-5
    assert (eng.debug_read("lvc2", 2, 12).cpu().reshape(2, 32, 3072)[:, :, ::4] - g["lvc2_sub"]).abs().max() < 1e-4


@pytest.mark.gpu
def test_cuda_vs_golden_sampler(synth, cuda_lib):
    import fastdiff_b200 as fb
    sd, _ = synth
    g = _load("sample_n4_b1_t6.npz")
    net = fb.FastDiff().to("cuda:0").eval()
    net.load_state_dict(sd)
    dh = fb.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
    for ddim, key in ((False, "seq_ddpm"), (True, "seq_ddim")):
        torch.manual_seed(int(g["seed"]))
        seq = fb.sampling_given_noise_schedule(net, (1, 1, 6 * 256), dh, torch.FloatTensor(N4), condition=g["mel"].cuda(), ddim=ddim,
                                               return_sequence=True)
        assert (torch.stack(seq).cpu() - g[key]).abs().max() < 5e-4
