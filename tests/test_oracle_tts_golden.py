"""The TTS-front-half oracle against vectors produced by the REAL reference
(oracle/make_golden_tts.py: SynthesizerTrn.infer, TextEncoder, both duration predictors)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import tts_oracle as T
from oracle.golden import Golden

GOLD = os.path.join(os.path.dirname(__file__), "golden")
CASES = ["tts_b1_t37", "tts_b2_padded", "tts_b1_t121_tails"]
# max |oracle - reference| per tensor.  The goldens are the reference's fp32 output on one CPU; on a CPU with another vector
# width or thread count the oracle's fp32 sums round differently, by up to a few times the reference's own fp32 noise floor
# (fp32 vs fp64 twin, floor_* in golden/REPORT_tts.json).  Where that floor is large -- logw_sdp 4.8e-5 (amplified by the
# spline inverses), z_p / z 8.8e-6, x 1.9e-6 -- the bound is about 4x it; on the other tensors the floor is <= 1.6e-6.
TOL = {"x": 8e-6, "m_p": 4e-6, "logs_p": 4e-6, "logw_sdp": 2e-4, "logw_dp": 4e-6, "z_p": 4e-5, "z": 4e-5}


def load(name):
    d = Golden(os.path.join(GOLD, name + ".npz"))
    return d, json.loads(str(d["meta"]))


def run_case(sd, c, **over):
    tokens, lengths, sid, noise_w = T.synthetic_tts_inputs(c["B"], c["T"], c["seed"], c["lengths"])
    noise = torch.randn(c["B"], 192, 40 * c["T"] + 64, generator=torch.Generator().manual_seed(30_000 + c["seed"]))
    kw = dict(noise_scale=c["noise_scale"], length_scale=c["length_scale"], noise_scale_w=c["noise_scale_w"],
              sdp_ratio=c["sdp_ratio"])
    kw.update(over)
    with torch.no_grad():
        return T.tts_infer(sd, tokens, lengths, sid, noise_w, noise, **kw)


@pytest.fixture(scope="module")
def tts_sd():
    return T.synthetic_tts_state_dict()


@pytest.mark.parametrize("name", CASES)
def test_infer_matches_reference(name, tts_sd):
    d, c = load(name)
    r = run_case(tts_sd, c)
    for key in ("x", "m_p", "logs_p", "logw_sdp", "logw_dp", "z_p", "z"):
        err = np.abs(d.pick(key, r[key].numpy()) - d[key]).max()
        assert err < TOL[key], (key, err)
    assert np.array_equal(r["w_ceil"][:, 0].numpy(), d["w_ceil"])
    assert np.array_equal(r["y_lengths"].numpy(), d["y_lengths"])
    assert r["o"].shape == d.shape("o")
    assert np.abs(d.pick("o", r["o"].numpy()) - d["o"]).max() < 1e-6


def test_spline_inverse_undoes_forward():
    """transforms.py:161-176 vs :188-207: the two branches are inverses on [-B, B], identity outside."""
    g = torch.Generator().manual_seed(5)
    x = 7 * (2 * torch.rand(4000, generator=g) - 1)
    uw, uh, ud = (torch.randn(4000, n, generator=g) for n in (10, 10, 9))
    y = T.rq_spline(x.double(), uw.double(), uh.double(), ud.double(), False, 5.0)
    back = T.rq_spline(y, uw.double(), uh.double(), ud.double(), True, 5.0)
    assert (back - x.double()).abs().max() < 1e-9
    out = x.abs() > 5
    assert torch.equal(y[out], x.double()[out]) and (torch.diff(y[torch.argsort(x)]) >= 0).sum() > 0


def test_ragged_equals_solo(tts_sd):
    """Per-utterance decode (what B=1 tts() calls give) for item 1 of the padded batch."""
    d, c = load("tts_b2_padded")
    r = run_case(tts_sd, c, ragged=True)
    tokens, lengths, sid, noise_w = T.synthetic_tts_inputs(c["B"], c["T"], c["seed"], c["lengths"])
    n = int(lengths[1])
    noise = torch.randn(c["B"], 192, 40 * c["T"] + 64, generator=torch.Generator().manual_seed(30_000 + c["seed"]))
    with torch.no_grad():
        solo = T.tts_infer(tts_sd, tokens[1:2, :n], lengths[1:2], sid[1:2], noise_w[1:2, :, :n], noise[1:2],
                           noise_scale=c["noise_scale"], length_scale=c["length_scale"],
                           noise_scale_w=c["noise_scale_w"], sdp_ratio=c["sdp_ratio"])
    ny = int(solo["y_lengths"][0])
    assert ny == int(r["y_lengths"][1])
    assert (solo["o"][0, 0] - r["o"][1, 0, :ny * 256]).abs().max() < 2e-6
