"""-m gpu: the bits of the tensor-core conv kernels, pinned.

Every tensor-core kernel (tcconv_kernel<128|64|32>, tcconv_wide_kernel, tcpair_kernel<64|32>) is reached by one of the
cases below: ragged and padded batches large enough for the sequential schedule (which fuses the conv pairs), the same
batch with the pair kernel off and with each kernel of the 128-column layers forced, a small call on the
concurrent-branch schedule, and a TTS call whose dense layers run through the same kernels.  Per case the SHA-256 of
every output and a few seeded sample values are compared with tests/golden/tc_bits.json.  Kernel changes that are
meant to keep the arithmetic must keep these bits.  Regenerate the fixture (only when a change of the arithmetic is
intended) with

    python tests/test_gpu_tc_bits.py

The second test checks that the retired tuning options are refused.
"""
import hashlib
import json
import os
import re
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURE = os.path.join(HERE, "golden", "tc_bits.json")
KERNELS = {"PAIR_N64", "PAIR_N32", "TC3_N128", "TC3_N64", "TC3_N32"}
N_SAMPLE = 8


def _digest(t):
    a = t.detach().contiguous().cpu().numpy()
    idx = np.random.default_rng(0).integers(0, a.size, N_SAMPLE)
    return {"shape": list(a.shape), "sha256": hashlib.sha256(a.tobytes()).hexdigest(),
            "sample": [float(v) for v in a.reshape(-1)[idx]]}


def _cases():
    """{name: (model, options, run)}: run() returns {tensor name: tensor}.  Options are set before and reset after."""
    from conftest import get_native, get_native_tts
    from oracle import tts_oracle as TO
    from oracle import vc_oracle as O
    m = get_native(False)
    dev = m.device

    def vc(B, T, lens, seed, ragged):
        spec, lengths, gs, gt, noise = (t.to(dev) for t in O.synthetic_inputs(B, T, seed, lengths=lens))

        def run():
            o, lat = m.native.voice_conversion(spec, lengths, gs, gt, noise=noise, tau=0.3, ragged=ragged)
            return {"o_hat": o, "z": lat[0], "z_p": lat[1], "z_hat": lat[2]}
        return run

    big = vc(3, 300, [300, 211, 37], 11, True)            # B * T > 512: sequential schedule, conv pairs fused
    cases = {
        "vc_b3_t300_f16x3": (m, {"precision": "f16x3"}, big),
        "vc_b3_t300_f16": (m, {"precision": "f16"}, big),
        "vc_b3_t300_f16x3_nopair": (m, {"precision": "f16x3", "pair": 0}, big),
        "vc_b3_t300_f16x3_wide0": (m, {"precision": "f16x3", "wide_variant": 0}, big),
        "vc_b3_t300_f16x3_wide2": (m, {"precision": "f16x3", "wide_variant": 2}, big),
        "vc_b3_t300_f16x3_padded": (m, {"precision": "f16x3"}, vc(3, 300, [300, 211, 37], 11, False)),
        "vc_b2_t48_f16x3": (m, {"precision": "f16x3"}, vc(2, 48, [48, 31], 3, True)),   # concurrent branches
    }

    t = get_native_tts()
    tokens, lengths, sid, noise_w = TO.synthetic_tts_inputs(2, 37, 9, [37, 22])

    def tts():
        o, _, y_mask, (z, z_p, _, _) = t.infer(tokens, lengths, sid=sid, noise_w=noise_w, noise_scale=0.667,
                                               noise_scale_w=0.6, sdp_ratio=0.2, seed=5, ragged=True)
        return {"o": o, "y_mask": y_mask, "z": z, "z_p": z_p}
    cases["tts_b2_t37_f16x3"] = (t, {"precision": "f16x3"}, tts)
    return cases


def _with_options(model, opts, fn):
    nat = model.native
    nat.set_option("graph", 0)
    try:
        for k, v in opts.items():
            nat.set_precision(v) if k == "precision" else nat.set_option(k, v)
        out = fn()
        torch.cuda.synchronize()
        return out
    finally:
        nat.set_precision(model.precision)
        nat.set_option("pair", 1)
        nat.set_option("wide_variant", 3)
        nat.set_option("graph", 1)


def record():
    """{case: {tensor: digest}} of unprofiled calls (profiling turns the concurrent-branch schedule off)."""
    return {name: {k: _digest(v) for k, v in _with_options(m, opts, run).items()}
            for name, (m, opts, run) in _cases().items()}


def launched_kernels():
    """Kernels of every tensor-core launch the cases make, from a separate profiled pass.  A per-launch profile name
    carries the kernel's column count: P<C>k<k>d<d> is tcpair_kernel<C> (PAIR_N<C>), T<TN>c<Cin>k<k>d<d> a conv of
    tcconv_kernel<TN> or, at TN = 128, tcconv_wide_kernel (TC3_N<TN>)."""
    names = set()
    for m, opts, run in _cases().values():
        nat = m.native
        nat.profile_enable(True)
        try:
            _with_options(m, opts, run)
            for rec in nat.profile_detail():
                hit = re.fullmatch(r"([PT])(\d+)(c\d+)?k\d+d\d+", rec[0])
                if hit:
                    names.add(("PAIR_N" if hit[1] == "P" else "TC3_N") + hit[2])
        finally:
            nat.profile_enable(False)
    return names


def test_tc_bits_match_fixture():
    with open(FIXTURE) as f:
        want = json.load(f)
    got = json.loads(json.dumps(record()))
    assert sorted(got) == sorted(want)
    for case in want:
        assert got[case] == want[case], case
    missing = KERNELS - launched_kernels()
    assert not missing, f"the cases no longer launch {sorted(missing)}"


def test_retired_options_are_refused():
    """OVC_OPT_ACT_TMA (4) and OVC_OPT_TUNE (6) are retired, and so is wide_variant 1 (256-step tiles)."""
    from conftest import get_native
    from openvoice_b200._native import _check
    nat = get_native(False).native
    for key in (4, 6):
        for value in (0, 1):
            with pytest.raises(ValueError, match="retired"):
                _check(nat.lib, nat.lib.ovc_set_option(nat.handle, key, value), "ovc_set_option")
    with pytest.raises(ValueError):
        nat.set_option("wide_variant", 1)
    for wv in (0, 2, 3):
        nat.set_option("wide_variant", wv)


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(HERE))
    rec = record()
    with open(FIXTURE, "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"wrote {FIXTURE}: {len(rec)} cases")
