"""SURVEY.md 8f.4 (second half): denoisers other than FastDiff that share the sampler.  fd_reverse_update (one reverse-step update as
one kernel) against the reference's eager operation sequence, bitwise, and the public sampler driving a foreign network against
what the reference's own sampler made of the same network (tests/golden/foreign_sampler.npz; CPU-emulated CUDA source)."""
import os

import numpy as np
import pytest
import torch

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class ForeignDenoiser(torch.nn.Module):
    """A denoiser that is not FastDiff, with the reference's `net((x, mel, diffusion_steps))` signature: elementwise in x, the first
    mel band held over each frame's 256 samples, and the step.  Every op is one exactly rounded product or sum, so the output has
    the same bits on any CPU (the stored sequence was recorded on another machine)."""

    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.tensor([0.3, -0.05, 1e-3]), requires_grad=False)

    def forward(self, data):
        x, mel, t = data
        band = mel[:, :1].repeat_interleave(256, dim=2)
        return self.w[0] * x + self.w[1] * band + self.w[2] * t.reshape(-1, 1, 1) * x


def foreign_sampler_input():
    """(size, mel, seed) of tests/golden/foreign_sampler.npz."""
    from fastdiff_b200.synthetic import make_inputs
    B, Tm = 2, 3
    return (B, 1, Tm * 256), make_inputs(B, Tm, 9)[1], 11


@pytest.fixture()
def emu_engine(emu_lib):
    from fastdiff_b200.engine import Engine
    return Engine(device="cpu", lib_path=emu_lib)


def _step(coef=0.151118, div=0.98723, sigma=0.051044, add_noise=1, c=(1.01, -0.16, 0.12)):
    from fastdiff_b200._lib import fd_step
    st = fd_step()
    st.t, st.coef_eps, st.div, st.sigma, st.add_noise = 74.99, coef, div, sigma, add_noise
    st.c1, st.c2, st.c3 = c
    return st


@pytest.mark.parametrize("n", [1, 3, 1024, 4099, 2 * 22016])
def test_reverse_update_is_the_reference_op_sequence_bitwise(emu_engine, n):
    """util.py:226-229: x -= coef*eps; x /= div; x = x + sigma*z  and  util.py:219-224: x = c1*x + c2*eps + c3*eps, every product
    and sum rounded to fp32 on its own (no FMA contraction), 0-dim fp32 coefficients as in the reference."""
    g = torch.Generator().manual_seed(n)
    x0, eps, z = (torch.randn(n, generator=g) * s for s in (3.0, 1.3, 1.0))
    st = _step()
    f = lambda v: torch.tensor(v, dtype=torch.float32)
    # stochastic rule, with and without the noise term, z given
    for add in (1, 0):
        st.add_noise = add
        want = x0.clone()
        want -= f(st.coef_eps) * eps
        want /= f(st.div)
        if add:
            want = want + f(st.sigma) * z
        x = x0.clone()
        seq = torch.empty_like(x)
        emu_engine.reverse_update(x, eps, st, z=z, seq=seq)
        assert torch.equal(x, want) and torch.equal(seq, want)
    # DDIM rule
    want = f(st.c1) * x0 + f(st.c2) * eps + f(st.c3) * eps
    x = x0.clone()
    emu_engine.reverse_update(x, eps, st, ddim=True)
    assert torch.equal(x, want)
    # unaligned views take the scalar path: same bits
    if n > 8:
        st.add_noise = 1
        xa = x0.clone()
        emu_engine.reverse_update(xa, eps, st, z=z)
        buf = torch.empty(n + 1)
        buf[1:] = x0
        xb, eb, zb = buf[1:], torch.empty(n + 1)[1:].copy_(eps), torch.empty(n + 1)[1:].copy_(z)
        emu_engine.reverse_update(xb, eb, st, z=zb)
        assert torch.equal(xa, xb)


def test_reverse_update_device_noise_is_the_sampler_stream(emu_engine):
    """z = NULL: the Philox4x32-10 draw keyed by (element, draw, seed) -- the generator fd_sample uses in device-noise mode."""
    n = 5000
    x0, eps = torch.randn(n), torch.randn(n)
    st = _step(coef=0.0, div=1.0, sigma=1.0)                 # x + z exactly
    a, b = x0.clone(), x0.clone()
    emu_engine.reverse_update(a, eps, st, seed=7, draw=1)
    emu_engine.reverse_update(b, eps, st, seed=7, draw=2)
    za, zb = a - x0, b - x0
    assert not torch.equal(za, zb)
    assert abs(za.mean().item()) < 0.06 and abs(za.std().item() - 1.0) < 0.05
    c = x0.clone()
    emu_engine.reverse_update(c, eps, st, seed=7, draw=1)
    assert torch.equal(a, c)                                  # a pure function of (element, draw, seed)


def test_reverse_update_rejects_bad_arguments(emu_engine):
    from fastdiff_b200._lib import FdError
    x = torch.zeros(8)
    with pytest.raises(ValueError):
        emu_engine.reverse_update(x, torch.zeros(9), _step())
    with pytest.raises(FdError, match="bad argument"):        # null pointers / count 0 through the raw C ABI
        emu_engine._check(emu_engine.lib.fd_reverse_update(emu_engine.h, None, None, None, None, 0, 0, 0, None, 0, None), "fd_reverse_update")


def test_foreign_network_needs_cuda():
    import fastdiff_b200 as fb
    net = torch.nn.Linear(2, 2)
    net.forward = lambda data: data[0]
    dh = fb.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
    with pytest.raises(RuntimeError, match="CUDA"):
        fb.sampling_given_noise_schedule(net, (1, 1, 256), dh, torch.FloatTensor([1e-4, 1e-2]), condition=torch.zeros(1, 80, 1))


@pytest.mark.parametrize("ddim", [False, True])
def test_sampler_drives_a_foreign_network_like_the_reference_sampler(emu_engine, monkeypatch, ddim):
    """ForeignDenoiser under OUR sampling_given_noise_schedule vs under the reference's (util.py:158-235): the same network, the same
    CPU RNG stream, every x_t of the sequence bit-identical."""
    import fastdiff_b200 as fb
    from fastdiff_b200 import sampler as S
    want = torch.from_numpy(np.load(os.path.join(G, "foreign_sampler.npz"))["seq_ddim" if ddim else "seq_ddpm"])
    net = ForeignDenoiser()
    size, mel, seed = foreign_sampler_input()
    sched = torch.FloatTensor([3.2176e-04, 2.5743e-03, 2.5376e-02, 7.0414e-01])
    monkeypatch.setitem(S._update_engines, "cpu", emu_engine)
    dh = fb.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
    torch.manual_seed(seed)
    got = fb.sampling_given_noise_schedule(net, size, dh, sched.clone(), condition=mel, ddim=ddim, return_sequence=True)
    assert len(got) == len(want) == 5
    for i in range(5):
        assert torch.equal(got[i], want[i]), i
    torch.manual_seed(seed)
    last = fb.sampling_given_noise_schedule(net, size, dh, sched.clone(), condition=mel, ddim=ddim)
    assert torch.equal(last, want[-1])


def _manual_loop(net, eng, x, mel, steps, noise=None, seed=0, ddim=False):
    """fd_denoise + fd_reverse_update per step: what the fused loop of fd_sample does, spelled out through the two public calls."""
    B = x.shape[0]
    draw = 0
    for st in steps:
        eps = eng.denoise(x, mel, torch.full((B,), st.t))
        z = None
        if st.add_noise and not ddim:
            z = noise[draw] if noise is not None else None
            draw += 1
        eng.reverse_update(x, eps, st, z=z, ddim=ddim, seed=seed, draw=draw)
    return x


@pytest.mark.parametrize("ddim", [False, True])
def test_fused_loop_equals_denoise_plus_reverse_update(synth, emu_lib, ddim):
    """fd_sample (final conv fused with the update, noise from the given draws or from Philox) == fd_denoise followed by
    fd_reverse_update, bitwise, for both update rules and both noise sources."""
    import fastdiff_b200 as fb
    from fastdiff_b200.sampler import build_steps
    from fastdiff_b200.synthetic import make_inputs
    sd, _ = synth
    net = fb.FastDiff().eval()
    net._lib_path = emu_lib
    net.load_state_dict(sd)
    eng = net.engine()
    B, Tm = 2, 2
    x0, mel = make_inputs(B, Tm, 8)
    dh = fb.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
    _, steps = build_steps(dh, torch.FloatTensor([3.2176e-04, 2.5743e-03, 2.5376e-02, 7.0414e-01]), ddim)
    noise = torch.randn(3, B, 1, Tm * 256)
    a = eng.sample(x0.clone(), mel, steps, noise=noise, ddim=ddim)
    b = _manual_loop(net, eng, x0.clone(), mel, steps, noise=noise, ddim=ddim)
    assert torch.equal(a, b)
    if not ddim:                                                                    # device noise: draw numbers 1, 2, 3
        a = eng.sample(x0.clone(), mel, steps, noise=None, seed=99)
        b = _manual_loop(net, eng, x0.clone(), mel, steps, noise=None, seed=99)
        assert torch.equal(a, b)
