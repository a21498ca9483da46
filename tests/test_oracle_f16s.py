"""The fp16-storage generator contract (precision "f16s"), emulated on the CPU against the reference's outputs.

``oracle.f16_storage.generator_f16s`` rounds where the GPU kernels of mode 3 round.  Run on the reference's own
z_hat, its output must stay within the mode's accuracy gate (o SNR >= 50 dB) of the reference's o_hat: this
predicts the GPU gate without a GPU."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import f16_storage as H
from oracle import tts_oracle as T
from oracle import vc_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")
GATE_DB = 50.0


def load(name):
    d = np.load(os.path.join(GOLD, name + ".npz"))
    return d, json.loads(str(d["meta"]))


@pytest.mark.parametrize("name", ["vc_b1_t24", "vc_b1_t67", "vc_b2_padded"])
def test_vc_generator_f16s_snr(name, synthetic_sd):
    d, c = load(name)
    _, lengths, _, gt, _ = O.synthetic_inputs(c["B"], c["T"], c["seed"], lengths=c["lengths"])
    mask = torch.from_numpy(d["mask"])
    with torch.no_grad():
        o = H.generator_f16s(synthetic_sd, torch.from_numpy(d["z_hat"]) * mask, gt)
    snr = H.snr_db(o, torch.from_numpy(d["o_hat"]))
    print(name, f"{snr:.1f} dB")
    assert snr >= GATE_DB, snr


def test_tts_generator_f16s_snr():
    d, c = load("tts_b1_t37")
    sd = T.synthetic_tts_state_dict()
    _, _, sid, _ = T.synthetic_tts_inputs(c["B"], c["T"], c["seed"])
    g = torch.nn.functional.embedding(sid, sd["emb_g.weight"]).unsqueeze(-1)
    with torch.no_grad():
        o = H.generator_f16s(sd, torch.from_numpy(d["z"]), g)
    snr = H.snr_db(o, torch.from_numpy(d["o"]))
    print(f"tts_b1_t37 {snr:.1f} dB")
    assert snr >= GATE_DB, snr


def test_f16_rounding_points(synthetic_sd):
    """Every stored activation is exactly representable in fp16, and the emulation differs from fp32."""
    d, c = load("vc_b1_t24")
    _, _, _, gt, _ = O.synthetic_inputs(c["B"], c["T"], c["seed"])
    taps = {}
    with torch.no_grad():
        o = H.generator_f16s(synthetic_sd, torch.from_numpy(d["z_hat"]), gt, taps=taps)
    assert sorted(taps) == sorted(["dec.pre"] + [f"dec.{k}{i}" for k in ("ups", "stage") for i in range(4)])
    for name, t in taps.items():
        assert torch.equal(t, H.f16(t)), name
    assert o.dtype == torch.float32 and not torch.equal(o, torch.from_numpy(d["o_hat"]))
