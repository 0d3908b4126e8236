"""CPU oracle for the FastDiff reverse-diffusion sampling hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``fastdiff_b200/`` may import this
module; only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs do, and there only as the checker
or the CPU yardstick -- never as the thing that is measured as the product.

What it is: a functional restatement (own code, closed forms) of the
reference's algorithm for the path, written against ``torch`` CPU tensor ops
because the reference's arithmetic itself lives in ATen (oneDNN conv / MKL
GEMM); it is dtype-parametric so the same code gives an fp64 "truth" used to
anchor the stated fp32 tolerance.

Reference files restated (all under /root/reference):
  modules/FastDiff/module/FastDiff_model.py:74-102   FastDiff.forward
  modules/FastDiff/module/modules.py:127-138         DiffusionDBlock.forward
  modules/FastDiff/module/modules.py:190-253         TimeAware_LVCBlock.forward / LVC
  modules/FastDiff/module/modules.py:320-343         KernelPredictor.forward
  modules/FastDiff/module/util.py:158-235            sampling_given_noise_schedule
  modules/FastDiff/module/util.py:365-432            schedule helpers, step embedding

Pinning: the reference ships no tests or golden vectors for this path
(SURVEY.md section 4), so the oracle is pinned against the reference itself:
  * tests/golden/*.npz are outputs of the imported reference, produced by
    tests/golden/make_golden.py (committed), and are checked on any machine;
  * tests/test_oracle_vs_reference.py checks every function here against
    the reference's outputs for the same seeded inputs (reference_cpu.npz).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F

# Network constants of the only architecture the reference ships
# (modules/FastDiff/config/base.yaml:21-33); the oracle itself is generic.
DEFAULT_RATIOS = (8, 8, 4)


# ----------------------------------------------------------------------------
# weights
# ----------------------------------------------------------------------------
def fold_weight_norm(state_dict: Dict[str, torch.Tensor], dtype=torch.float32) -> Dict[str, torch.Tensor]:
    """name.weight_g/name.weight_v -> name.weight  (w = g * v / ||v||, norm per
    out-channel over the remaining dims; torch.nn.utils.weight_norm dim=0, which
    FastDiff_model.py:115-122 applies to every Conv1d).  Plain weights pass through."""
    out: Dict[str, torch.Tensor] = {}
    for k, v in state_dict.items():
        if k.endswith(".weight_g"):
            base = k[: -len(".weight_g")]
            g = v.to(dtype)
            vv = state_dict[base + ".weight_v"].to(dtype)
            nrm = vv.reshape(vv.shape[0], -1).norm(dim=1).reshape(-1, *([1] * (vv.dim() - 1)))
            out[base + ".weight"] = g * vv / nrm
        elif k.endswith(".weight_v"):
            continue
        else:
            out[k] = v.to(dtype)
    return out


# ----------------------------------------------------------------------------
# schedule helpers (util.py:365-404)
# ----------------------------------------------------------------------------
def compute_hyperparams_given_schedule(beta: torch.Tensor) -> dict:
    """util.py:365-390.  alpha_t = sqrt(prod_{s<=t}(1-beta_s)),
    sigma_t = sqrt(beta_t (1-abar_{t-1})/(1-abar_t)); sequential fp32 products
    exactly as the reference's in-place loop performs them."""
    T = len(beta)
    alpha = 1 - beta
    sigma = beta + 0
    for t in range(1, T):
        alpha[t] = alpha[t] * alpha[t - 1]
        sigma[t] = sigma[t] * ((1 - alpha[t - 1]) / (1 - alpha[t]))
    return {"T": T, "beta": beta, "alpha": torch.sqrt(alpha), "sigma": torch.sqrt(sigma)}


def map_noise_scale_to_time_step(alpha_infer, alpha) -> float:
    """util.py:394-404: clamp, else first bracketing interval, linear interpolation."""
    if alpha_infer < alpha[-1]:
        return len(alpha) - 1
    if alpha_infer > alpha[0]:
        return 0
    for t in range(len(alpha) - 1):
        if alpha[t + 1] <= alpha_infer <= alpha[t]:
            d = alpha[t] - alpha_infer
            d = d / (alpha[t] - alpha[t + 1])
            return t + d.item()
    return -1


def sampler_tables(inference_noise_schedule: torch.Tensor, alpha_train: torch.Tensor):
    """Host prologue of util.py:187-204 -> (beta_infer, alpha_infer, sigma_infer, steps_infer)."""
    beta_infer = inference_noise_schedule
    N = len(beta_infer)
    alpha_infer = 1 - beta_infer
    sigma_infer = beta_infer + 0
    for n in range(1, N):
        alpha_infer[n] = alpha_infer[n] * alpha_infer[n - 1]
        sigma_infer[n] = sigma_infer[n] * ((1 - alpha_infer[n - 1]) / (1 - alpha_infer[n]))
    alpha_infer = torch.sqrt(alpha_infer)
    sigma_infer = torch.sqrt(sigma_infer)
    steps = []
    for n in range(N):
        s = map_noise_scale_to_time_step(alpha_infer[n], alpha_train)
        if s >= 0:
            steps.append(s)
    return beta_infer, alpha_infer, sigma_infer, torch.FloatTensor(steps)


# ----------------------------------------------------------------------------
# denoiser pieces
# ----------------------------------------------------------------------------
def step_embedding(diffusion_steps: torch.Tensor, dim: int = 128) -> torch.Tensor:
    """util.py:407-432: [sin(t f_j), cos(t f_j)], f_j = exp(-j ln(1e4)/(half-1)).
    The frequency table is built in fp32 (torch.arange * python float -> fp32)."""
    assert dim % 2 == 0
    half = dim // 2
    c = np.log(10000) / (half - 1)
    f = torch.exp(torch.arange(half) * -c)  # fp32, like the reference
    a = diffusion_steps * f.to(diffusion_steps.dtype)
    return torch.cat((torch.sin(a), torch.cos(a)), 1)


def _swish(x):
    return x * torch.sigmoid(x)


def embed_mlp(W, t: torch.Tensor, dim_in: int = 128) -> torch.Tensor:
    """FastDiff_model.py:85-87."""
    e = step_embedding(t, dim_in)
    e = _swish(F.linear(e, W["fc_t1.weight"], W["fc_t1.bias"]))
    e = _swish(F.linear(e, W["fc_t2.weight"], W["fc_t2.bias"]))
    return e


def dblock(W, prefix: str, x: torch.Tensor, factor: int) -> torch.Tensor:
    """modules.py:127-138.  nearest interpolate to size L//f is x[..., ::f] (exact when f | L)."""
    size = x.shape[-1] // factor
    xs = x[..., ::factor][..., :size]
    res = F.conv1d(xs, W[f"{prefix}.residual_dense.weight"], W[f"{prefix}.residual_dense.bias"])
    h = xs
    for i, d in enumerate((1, 2, 4)):
        h = F.leaky_relu(h, 0.2)
        h = F.conv1d(h, W[f"{prefix}.conv.{i}.weight"], W[f"{prefix}.conv.{i}.bias"], padding=d, dilation=d)
    return h + res


def kernel_predictor(W, prefix: str, cond: torch.Tensor, layers=4, cin=32, cout=64, ksz=3):
    """modules.py:320-343 -> kernels (B,layers,cin,cout,ksz,T'), bias (B,layers,cout,T')."""
    B, _, Tm = cond.shape
    h = F.leaky_relu(F.conv1d(cond, W[f"{prefix}.input_conv.0.weight"], W[f"{prefix}.input_conv.0.bias"], padding=2), 0.1)
    r = h
    for idx in (1, 3, 6, 8, 11, 13):  # nn.Sequential slots that hold convs (others: Dropout p=0 / LeakyReLU)
        r = F.leaky_relu(
            F.conv1d(r, W[f"{prefix}.residual_conv.{idx}.weight"], W[f"{prefix}.residual_conv.{idx}.bias"], padding=1), 0.1
        )
    h = h + r
    k = F.conv1d(h, W[f"{prefix}.kernel_conv.weight"], W[f"{prefix}.kernel_conv.bias"], padding=1)
    b = F.conv1d(h, W[f"{prefix}.bias_conv.weight"], W[f"{prefix}.bias_conv.bias"], padding=1)
    return k.reshape(B, layers, cin, cout, ksz, Tm), b.reshape(B, layers, cout, Tm)


def lvc(x: torch.Tensor, kernel: torch.Tensor, bias: torch.Tensor, hop: int) -> torch.Tensor:
    """modules.py:220-253 at dilation 1 (the only value the reference passes, :216):
    out[b,o,t] = bias[b,o,t//hop] + sum_{i,k} xpad[b,i,t+k] * kernel[b,i,o,k,t//hop],
    xpad = x zero-padded by (ksz-1)/2 at both sequence ends.
    Evaluated the way the reference evaluates it -- frame windows by `unfold`, taps by a second `unfold`, ONE einsum over
    (i, k) that ATen lowers to a batched GEMM -- so that this port costs the same ATen work as the reference when it serves as a
    CPU yardstick.  `lvc_taps` below is the independent closed form (three shifted einsums) the tests cross-check it with."""
    B, Ci, T = x.shape
    _, _, Co, K, Tm = kernel.shape
    assert T == Tm * hop, "length of (x, kernel) is not matched"
    p = (K - 1) // 2
    win = F.pad(x, (p, p)).unfold(2, hop + 2 * p, hop)          # (B, Ci, Tm, hop + K - 1): frame l sees its hop samples + halo
    win = win.unfold(3, K, 1)                                   # (B, Ci, Tm, hop, K): tap k of sample s
    out = torch.einsum("bilsk,biokl->bols", win, kernel)        # (B, Co, Tm, hop)
    out = out + bias.unsqueeze(-1)
    return out.reshape(B, Co, T)


def lvc_taps(x: torch.Tensor, kernel: torch.Tensor, bias: torch.Tensor, hop: int) -> torch.Tensor:
    """The same sum written tap by tap (no unfold): the cross-check of `lvc`."""
    B, Ci, T = x.shape
    _, _, Co, K, Tm = kernel.shape
    assert T == Tm * hop, "length of (x, kernel) is not matched"
    p = (K - 1) // 2
    xp = F.pad(x, (p, p))
    out = bias.unsqueeze(-1).expand(B, Co, Tm, hop).clone()
    for k in range(K):
        xs = xp[:, :, k : k + T].reshape(B, Ci, Tm, hop)
        out = out + torch.einsum("bils,biol->bols", xs, kernel[:, :, :, k, :])
    return out.reshape(B, Co, T)


def lvc_block(W, n: int, x, skip, mel, e, ratio: int, hop: int, layers=4, C=32):
    """modules.py:190-218."""
    p = f"lvc_blocks.{n}"
    noise = F.linear(e, W[f"{p}.fc_t.weight"], W[f"{p}.fc_t.bias"]).unsqueeze(-1)
    cond = mel + noise
    kernels, bias = kernel_predictor(W, f"{p}.kernel_predictor", cond, layers, C, 2 * C, 3)
    x = F.leaky_relu(x, 0.2)
    x = F.conv_transpose1d(
        x, W[f"{p}.upsample.weight"], W[f"{p}.upsample.bias"], stride=ratio,
        padding=ratio // 2 + ratio % 2, output_padding=ratio % 2,
    )
    for i in range(layers):
        x = x + skip  # reference does this in place, every layer
        y = F.leaky_relu(x, 0.2)
        d = 3 ** i
        y = F.conv1d(y, W[f"{p}.convs.{i}.weight"], W[f"{p}.convs.{i}.bias"], padding=d, dilation=d)
        y = F.leaky_relu(y, 0.2)
        y = lvc(y, kernels[:, i], bias[:, i], hop)
        x = x + torch.sigmoid(y[:, :C]) * torch.tanh(y[:, C:])
    return x


def denoise(W, x: torch.Tensor, mel: torch.Tensor, t: torch.Tensor, ratios: Sequence[int] = DEFAULT_RATIOS,
            return_intermediates: bool = False):
    """FastDiff.forward((x, mel, t)) -> eps.  W = folded weights (fold_weight_norm)."""
    inter = {}
    e = embed_mlp(W, t)
    inter["embed"] = e
    h = F.conv1d(x, W["first_audio_conv.weight"], W["first_audio_conv.bias"], padding=3)
    skips = []
    nb = len(ratios)
    for n in range(nb):
        skips.append(h)
        h = dblock(W, f"downsample.{n}", h, ratios[nb - n - 1])
        inter[f"down{n}"] = h
    hop = 1
    for n, skip in enumerate(reversed(skips)):
        hop *= ratios[n]
        h = lvc_block(W, n, h, skip, mel, e, ratios[n], hop)
        inter[f"lvc{n}"] = h
    out = F.conv1d(h, W["final_conv.0.weight"], W["final_conv.0.bias"], padding=3)
    if return_intermediates:
        return out, inter
    return out


# ----------------------------------------------------------------------------
# sampler (util.py:158-235)
# ----------------------------------------------------------------------------
def sample(W, size, diffusion_hyperparams, inference_noise_schedule, condition, ddim=False,
           return_sequence=False, noise: Optional[Sequence[torch.Tensor]] = None,
           ratios: Sequence[int] = DEFAULT_RATIOS):
    """The reverse loop.  ``noise`` (optional) = [x_T, z_{N-1}, ..., z_1] in the order the reference
    draws them; if None they are drawn from the CPU default generator in that same order."""
    T, alpha = diffusion_hyperparams["T"], diffusion_hyperparams["alpha"]
    assert len(alpha) == T
    assert len(size) == 3
    beta_infer, alpha_infer, sigma_infer, steps_infer = sampler_tables(inference_noise_schedule, alpha)
    N = len(steps_infer)
    draws = iter(noise) if noise is not None else None

    def draw():
        return next(draws) if draws is not None else torch.normal(0, 1, size=size)

    dt = W["fc_t1.weight"].dtype
    x = draw().to(dt)
    xs = [x.clone()]
    for n in range(N - 1, -1, -1):
        t = (steps_infer[n] * torch.ones((size[0], 1))).to(dt)
        eps = denoise(W, x, condition, t, ratios)
        if ddim:
            alpha_next = alpha_infer[n] / (1 - beta_infer[n]).sqrt()
            c1 = alpha_next / alpha_infer[n]
            c2 = -(1 - alpha_infer[n] ** 2.0).sqrt() * c1
            c3 = (1 - alpha_next ** 2.0).sqrt()
            x = c1 * x + c2 * eps + c3 * eps
        else:
            x = x - beta_infer[n] / torch.sqrt(1 - alpha_infer[n] ** 2.0) * eps
            x = x / torch.sqrt(1 - beta_infer[n])
            if n > 0:
                x = x + sigma_infer[n] * draw().to(dt)
        xs.append(x.clone())
    return xs if return_sequence else x
