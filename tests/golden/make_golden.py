"""Generates tests/golden/* from the UNMODIFIED reference (fp32, TF32 off).

    python tests/golden/make_golden.py [--out DIR]
    python tests/golden/make_golden.py --gpu [--out DIR]        # on a B200: reference_gpu.npz only

The reference is imported through oracle/refimport.py: the checkout named by FD_REFERENCE_ROOT, or the bytecode build oracle/_ref
that __graft_entry__.build() makes of a reachable checkout (oracle/stage_reference.py), which is how the ``--gpu`` part runs on a GPU
machine without the checkout.  The reference hard-codes
`.cuda()` (util.py:68,217,427); for the CPU part `torch.Tensor.cuda` is shimmed to identity so the whole path runs on the CPU
unmodified.  Weights are the seeded synthetic state dict (fastdiff_b200/synthetic.py, seed 1234, g_jitter 0.1) loaded into the
reference model with load_state_dict, and every input is drawn from a fixed seed, so the tests rebuild the same inputs.  Large
outputs are kept as a fixed strided sample (`flat[::stride]`, strides below); the tests compare the same sample.
"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from fastdiff_b200.synthetic import make_inputs, make_state_dict  # noqa: E402
from oracle import refimport  # noqa: E402
from tests.golden.make_golden_schedules import N_SCHEDULES  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
LVC_STRIDE = 23          # reference_cpu.npz lvc_*: flat[::23] of the LVC output
BATCH_STRIDE = 211       # reference_gpu.npz eps_8x861: flat[::211] of every item's eps
SEQ_STRIDE = 53          # reference_gpu.npz seq_*: flat[::53] of every x_t of the (2, 1, 25600) sequence
WAV_EXCERPT = (22050, 16384)   # LJ001-0001_gt_excerpt.wav: samples [22050, 22050 + 16384) of egs/audios/LJ001-0001_gt.wav


def _model(R, device):
    model = R.FastDiff().to(device).eval()
    model.load_state_dict(make_state_dict(1234, g_jitter=0.1))
    return model


def _save(out, name, arrays):
    np.savez_compressed(os.path.join(out, name), **{k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in arrays.items()})


def denoise_stages(R, out):
    """denoise_b2_t12.npz: eps and stage outputs of one forward, captured with forward hooks (tests/test_golden.py)."""
    torch.manual_seed(0)
    model = _model(R, "cpu")
    B, Tm = 2, 12
    x, mel = make_inputs(B, Tm, 3)
    t = torch.tensor([[7.413235], [498.0537]])
    cap = {}
    hooks = []
    for n in range(3):
        def down_hook(m, i, o, n=n):
            cap[f"down{n}"] = o.detach().clone()
        def lvc_hook(m, i, o, n=n):
            cap[f"lvc{n}"] = o.detach().clone()
        hooks.append(model.downsample[n].register_forward_hook(down_hook))
        hooks.append(model.lvc_blocks[n].register_forward_hook(lvc_hook))
        def kp_hook(m, i, o, n=n):
            cap[f"kernels{n}"] = o[0].detach().clone()
            cap[f"kbias{n}"] = o[1].detach().clone()
        hooks.append(model.lvc_blocks[n].kernel_predictor.register_forward_hook(kp_hook))
    with torch.no_grad():
        eps = model((x, mel, t))
    for h in hooks:
        h.remove()
    arrays = {"x": x, "mel": mel, "t": t, "eps": eps}
    for n in range(3):
        arrays[f"down{n}"] = cap[f"down{n}"]
        arrays[f"kbias{n}"] = cap[f"kbias{n}"]
        arrays[f"kernels{n}_sub"] = cap[f"kernels{n}"][:, :, ::8, ::8]  # (B,4,4,8,3,T') slice keeps the file small
        arrays[f"lvc{n}" if n < 2 else "lvc2_sub"] = cap[f"lvc{n}"] if n < 2 else cap["lvc2"][:, :, ::4]   # every 4th sample of the last block
    _save(out, "denoise_b2_t12.npz", arrays)
    return model


def sampler_and_tables(R, model, out):
    """sample_n4_b1_t6.npz (N=4 DDPM + DDIM, fixed CPU RNG seed, reference draw order) and tables.npz (weight-free known answers)."""
    B, Tm = 1, 6
    _, mel = make_inputs(B, Tm, 5)
    dh = R.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
    arrays = {"mel": mel, "seed": np.array(11)}
    for ddim in (False, True):
        torch.manual_seed(11)
        seq = R.sampling_given_noise_schedule(model, (B, 1, Tm * 256), dh, torch.FloatTensor(N_SCHEDULES[4]), condition=mel,
                                              ddim=ddim, return_sequence=True)
        arrays["seq_ddim" if ddim else "seq_ddpm"] = torch.stack(seq)
    _save(out, "sample_n4_b1_t6.npz", arrays)

    ka = {"alpha": dh["alpha"], "sigma": dh["sigma"]}
    for N, s in N_SCHEDULES.items():
        b = torch.FloatTensor(s)
        a = 1 - b
        sg = b + 0
        for n in range(1, len(b)):
            a[n] *= a[n - 1]
            sg[n] *= (1 - a[n - 1]) / (1 - a[n])
        a, sg = torch.sqrt(a), torch.sqrt(sg)
        ka[f"steps_{N}"] = np.array([R.util.map_noise_scale_to_time_step(a[n], dh["alpha"]) for n in range(len(b))], dtype=np.float64)
        ka[f"alpha_infer_{N}"] = a
        ka[f"sigma_infer_{N}"] = sg
    ka["embed_in"] = R.util.calc_diffusion_step_embedding(torch.tensor([[0.0], [7.413235], [498.0537], [999.0]]), 128)
    _save(out, "tables.npz", ka)


def reference_cpu(R, model, out):
    """reference_cpu.npz: what tests/test_oracle_vs_reference.py compares the oracle and the host code with."""
    arrays = {}
    for B, Tm, seed in ((2, 12, 0), (1, 1, 1), (3, 5, 2)):
        x, mel = make_inputs(B, Tm, seed)
        t = torch.tensor([7.413235, 498.0537, 23.46759][:B]).reshape(B, 1)
        with torch.no_grad():
            arrays[f"eps_{B}_{Tm}_{seed}"] = model((x, mel, t))
    blk = R.FastDiff().lvc_blocks[2]
    torch.manual_seed(0)
    for hop, Tm in ((256, 3), (64, 5), (8, 7)):
        x = torch.randn(2, 32, hop * Tm)
        k = torch.randn(2, 32, 64, 3, Tm)
        b = torch.randn(2, 64, Tm)
        arrays[f"lvc_{hop}_{Tm}"] = blk.location_variable_convolution(x, k, b, 1, hop).flatten()[::LVC_STRIDE]
    _, mel = make_inputs(1, 4, 5)
    dh = R.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
    for ddim in (False, True):
        torch.manual_seed(5)
        seq = R.sampling_given_noise_schedule(model, (1, 1, 1024), dh, torch.FloatTensor(N_SCHEDULES[4]), condition=mel, ddim=ddim,
                                              return_sequence=True)
        arrays["seq_ddim" if ddim else "seq_ddpm"] = torch.stack(seq)
    arrays["map_alpha"] = np.array([0.5, 0.9999, 0.05, 1.0, 0.0813796], dtype=np.float32)
    arrays["map_step"] = np.array([R.util.map_noise_scale_to_time_step(torch.tensor(al), dh["alpha"]) for al in arrays["map_alpha"]],
                                  dtype=np.float64)
    arrays["embed"] = R.util.calc_diffusion_step_embedding(torch.tensor([[0.0], [3.5], [999.0]]), 128)
    sd = R.FastDiff().state_dict()
    arrays["sd_keys"] = np.array(list(sd.keys()))
    arrays["sd_shapes"] = np.array([",".join(str(d) for d in v.shape) for v in sd.values()])
    _save(out, "reference_cpu.npz", arrays)


def foreign_sampler(R, out):
    """foreign_sampler.npz: the reference's sampler driving a network other than FastDiff (tests/test_foreign_denoiser.py)."""
    from tests.test_foreign_denoiser import ForeignDenoiser, foreign_sampler_input
    net = ForeignDenoiser()
    size, mel, seed = foreign_sampler_input()
    dh = R.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
    arrays = {}
    for ddim in (False, True):
        torch.manual_seed(seed)
        seq = R.sampling_given_noise_schedule(net, size, dh, torch.FloatTensor(N_SCHEDULES[4]), condition=mel, ddim=ddim,
                                              return_sequence=True)
        arrays["seq_ddim" if ddim else "seq_ddpm"] = torch.stack(seq)
    _save(out, "foreign_sampler.npz", arrays)


def wav_excerpt(root, out):
    """LJ001-0001_gt_excerpt.wav: 0.74 s of the reference's example recording (egs/audios), a real-speech mel front-end input."""
    from scipy.io import wavfile
    sr, data = wavfile.read(os.path.join(root, "egs", "audios", "LJ001-0001_gt.wav"))
    lo, n = WAV_EXCERPT
    wavfile.write(os.path.join(out, "LJ001-0001_gt_excerpt.wav"), sr, data[lo:lo + n])


def reference_gpu(out):
    """reference_gpu.npz: the reference on cuda:0 in eager fp32, TF32 off (tests/test_gpu_parity.py, `*_vs_reference_on_gpu`)."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    R = refimport.load("cuda")
    model = _model(R, "cuda")
    arrays = {}
    B, Tm = 8, 861
    x, mel = make_inputs(B, Tm, 32)
    t = torch.tensor([7.413235, 23.46759, 74.99228, 498.0537, 7.413235, 23.46759, 74.99228, 498.0537]).reshape(B, 1)
    with torch.no_grad():
        arrays["eps_8x861"] = model((x.cuda(), mel.cuda(), t.cuda())).reshape(B, -1)[:, ::BATCH_STRIDE]
    torch.cuda.empty_cache()
    B, Tm = 2, 100
    _, mel = make_inputs(B, Tm, 36)
    dh = R.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000).cuda())
    arrays["alpha"], arrays["sigma"] = dh["alpha"], dh["sigma"]
    for ddim in (False, True):
        torch.manual_seed(21)
        seq = R.sampling_given_noise_schedule(model, (B, 1, Tm * 256), dh, torch.FloatTensor(N_SCHEDULES[4]).cuda(), condition=mel.cuda(),
                                              ddim=ddim, return_sequence=True)
        arrays["seq_ddim" if ddim else "seq_ddpm"] = torch.stack([s.flatten()[::SEQ_STRIDE] for s in seq])
    arrays["device"] = np.array(torch.cuda.get_device_name(0))
    _save(out, "reference_gpu.npz", arrays)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpu", action="store_true", help="record reference_gpu.npz (needs a CUDA device)")
    ap.add_argument("--out", default=OUT)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    if args.gpu:
        reference_gpu(args.out)
    else:
        R = refimport.load("cpu")
        model = denoise_stages(R, args.out)
        sampler_and_tables(R, model, args.out)
        reference_cpu(R, model, args.out)
        foreign_sampler(R, args.out)
        wav_excerpt(R.root, args.out)
    for f in sorted(os.listdir(args.out)):
        if f.endswith((".npz", ".wav")):
            print(f, os.path.getsize(os.path.join(args.out, f)))


if __name__ == "__main__":
    main()
