"""CPU emulation of precision mode 3 ("f16s"): the HiFi-GAN generator with fp16 activations in memory.

TEST INFRASTRUCTURE ONLY, like ``vc_oracle``: it predicts, on a machine without a GPU, what the fp16-storage
generator computes, rounding exactly where the kernels round (include/ovc.h, mode 3):

* conv_pre reads fp32 ``z_hat * mask``; its operand is rounded to fp16, its output stored as fp16;
* every conv from conv_pre to the last ResBlock multiplies fp16 operands by fp16 weights (one pass) and
  accumulates in fp32; a conv's operand is ``fp16(lrelu(x))``, computed in fp32 from the fp16 input;
* bias, residual add, MRF accumulation and the 1/3 are fp32 math, and every store rounds to fp16 (RN):
  a ResBlock conv2 stores ``fp16(conv + bias + residual)``, the MRF sum ``fp16(xs + v)`` after branch 1 and
  ``fp16((xs + v) * (1/3))`` after branch 2;
* conv_post reads fp16, applies lrelu(0.01) in fp32, accumulates in fp32 and applies tanh (fp32 output).

Weights and shapes are ``vc_oracle``'s; ``vc_oracle.generator`` is the fp32 reference this is compared with.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn.functional as F

from oracle import vc_oracle as V


def f16(x: torch.Tensor) -> torch.Tensor:
    """Round to fp16 (nearest even) and back to fp32."""
    return x.to(torch.float16).to(torch.float32)


def _lrelu16(x: torch.Tensor, slope: float) -> torch.Tensor:
    # the kernels' leaky_relu is max(x, x * slope) in fp32, bit-identical to the select for 0 <= slope <= 1
    return f16(torch.maximum(x, x * slope))


def generator_f16s(sd: V.StateDict, z: torch.Tensor, g: torch.Tensor, hp: Optional[dict] = None,
                   taps: Optional[dict] = None) -> torch.Tensor:
    """The generator of ``vc_oracle.generator`` under the mode-3 rounding contract.  ``z`` is the fp32
    ``z_hat * mask`` [B, 192, T], ``g`` the speaker embedding [B, gin, 1].  Returns o [B, 1, 256 T] (fp32)."""
    m = (hp or V.DEFAULT_HPARAMS)["model"]
    ks, ds = m["resblock_kernel_sizes"], m["resblock_dilation_sizes"]
    sd = {k: v.float() for k, v in sd.items()}
    z, g = z.float(), g.float()
    # conv_pre + cond(g): one bias vector per utterance (fp32), one fp16 pass, fp16 store
    bias = sd["dec.conv_pre.bias"][None, :, None] + F.conv1d(g, sd["dec.cond.weight"], sd["dec.cond.bias"])
    x = f16(F.conv1d(f16(z), f16(sd["dec.conv_pre.weight"]), None, padding=3) + bias)
    if taps is not None:
        taps["dec.pre"] = x
    for i, (u, k) in enumerate(zip(m["upsample_rates"], m["upsample_kernel_sizes"])):
        x = f16(F.conv_transpose1d(_lrelu16(x, V.LRELU_SLOPE), f16(V._w(sd, f"dec.ups.{i}")), sd[f"dec.ups.{i}.bias"],
                                   stride=u, padding=(k - u) // 2))
        if taps is not None:
            taps[f"dec.ups{i}"] = x
        xs = None
        for j in range(len(ks)):
            p = f"dec.resblocks.{i * len(ks) + j}"
            r = x
            for n, d in enumerate(ds[j]):
                xt = f16(F.conv1d(_lrelu16(r, V.LRELU_SLOPE), f16(V._w(sd, f"{p}.convs1.{n}")), sd[f"{p}.convs1.{n}.bias"],
                                  dilation=d, padding=d * (ks[j] - 1) // 2))
                v = F.conv1d(_lrelu16(xt, V.LRELU_SLOPE), f16(V._w(sd, f"{p}.convs2.{n}")), sd[f"{p}.convs2.{n}.bias"],
                             padding=(ks[j] - 1) // 2) + r
                if n < len(ds[j]) - 1:
                    r = f16(v)
                elif xs is None:
                    xs = f16(v)
                elif j < len(ks) - 1:
                    xs = f16(xs + v)
                else:
                    xs = f16((xs + v) * (1.0 / len(ks)))   # the kernels multiply by the fp32 1/3
        x = xs
        if taps is not None:
            taps[f"dec.stage{i}"] = x
    x = torch.maximum(x, x * 0.01)   # leaky_relu(0.01), models.py:287, on the fp16 activations
    return torch.tanh(F.conv1d(x, sd["dec.conv_post.weight"], None, padding=3))


def snr_db(got: torch.Tensor, ref: torch.Tensor) -> float:
    """10 log10(|ref|^2 / |got - ref|^2), in float64."""
    got, ref = torch.as_tensor(got).double(), torch.as_tensor(ref).double()
    err = (got - ref).pow(2).sum().item()
    return float("inf") if err == 0 else 10.0 * torch.log10(ref.pow(2).sum() / err).item()
