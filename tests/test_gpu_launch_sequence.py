"""-m gpu: what the host library enqueues, pinned.

The launch list of every entry point -- per launch the profile record (kernel name, family, algorithmic flops and
bytes), the profile totals, ovc_last_launch_count and the debug taps -- is compared with
tests/golden/launch_sequence.json.  Host-side changes to the launch code must leave all of it as it is: bench.py's
roofline leg and tools/layer_report.py read these records.  Regenerate the fixture (only when a change to the launch
sequence is intended) with

    python tests/test_gpu_launch_sequence.py

The second test checks how finalize reports a broken checkpoint: a missing tensor raises OvcError, a mis-shaped one
ValueError, and both messages name the tensor.
"""
import copy
import json
import os
import re
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURE = os.path.join(HERE, "golden", "launch_sequence.json")
VC_TAPS = ["cond", "enc.pre", "enc.wn", "dec.pre"] + [f"dec.{s}{i}" for i in range(4) for s in ("ups", "stage")]
TTS_TAPS = ["tts.layer0", "tts.x", "tts.stats", "tts.sdp_cond", "tts.logw_sdp", "tts.logw_dp"]


def _profiled(nat, fn):
    """Run fn with profiling on: per-launch records (without times), totals, launch count."""
    nat.profile_enable(True)
    try:
        fn()
        torch.cuda.synchronize()
        detail = [[name, fl, by, fam] for name, _, fl, by, fam in nat.profile_detail()]
        tot = nat.profile_read()
    finally:
        nat.profile_enable(False)
    return {"detail": detail, "launches": tot["launches"], "flops": tot["flops"], "bytes": tot["bytes"],
            "last_launch_count": nat.last_launch_count}


def _taps(nat, names):
    """{name: [B, C, T, pitch]} of the named debug taps, None for a tap the last call did not write."""
    import ctypes as C
    out = {}
    for name in names:
        shape = (C.c_int64 * 4)()
        rc = nat.lib.ovc_debug_fetch(nat.handle, name.encode(), None, 0, shape)
        out[name] = [int(v) for v in shape] if rc >= 0 else None
    return out


def record():
    from conftest import get_native, get_native_tts
    from oracle import tts_oracle as TO
    from oracle import vc_oracle as O
    rec = {}

    m = get_native(False)
    nat = m.native
    dev = m.device
    nat.set_option("graph", 0)
    try:
        def vc(B, T, lens, seed):
            spec, lengths, gs, gt, noise = O.synthetic_inputs(B, T, seed, lengths=lens)
            args = [t.to(dev) for t in (spec, lengths, gs, gt, noise)]
            return lambda: nat.voice_conversion(*args[:4], noise=args[4], tau=0.3, ragged=True)

        small = vc(2, 48, [48, 31], 3)
        for mode in ("fp32", "f16x3", "f16"):
            nat.set_precision(mode)
            rec[f"vc_b2_t48_{mode}"] = _profiled(nat, small)
        nat.set_precision("f16x3")
        nat.set_option("pair", 0)
        rec["vc_b2_t48_f16x3_nopair"] = _profiled(nat, small)
        nat.set_option("pair", 1)
        rec["vc_b2_t300_f16x3"] = _profiled(nat, vc(2, 300, [300, 211], 4))
        small()                                   # profiling off: the concurrent-branch schedule
        torch.cuda.synchronize()
        rec["vc_b2_t48_f16x3_branches_launch_count"] = nat.last_launch_count

        L = 22050
        wav = (torch.rand(2, L, generator=torch.Generator().manual_seed(3)) - 0.5).to(dev)
        wlen = torch.tensor([L, L - 3000], dtype=torch.int64, device=dev)
        g1 = 0.1 * torch.randn(2, 256, generator=torch.Generator().manual_seed(4)).to(dev)
        g2 = 0.1 * torch.randn(2, 256, generator=torch.Generator().manual_seed(5)).to(dev)
        rec["convert_waveform_b2_f16x3"] = _profiled(nat, lambda: nat.convert_waveform(wav, wlen, g1, g2, tau=0.3, seed=7))

        nat.debug_enable(True)
        try:
            for mode in ("fp32", "f16x3"):
                nat.set_precision(mode)
                small()
                torch.cuda.synchronize()
                rec[f"taps_vc_{mode}"] = _taps(nat, VC_TAPS)
        finally:
            nat.debug_enable(False)
    finally:
        nat.set_precision(m.precision)
        nat.set_option("graph", 1)

    t = get_native_tts()
    nat = t.native
    dev = t.device
    tokens, lengths, sid, noise_w = TO.synthetic_tts_inputs(2, 37, 9, [37, 22])
    targs = [x.to(dev) for x in (tokens, lengths, sid, noise_w)]
    state = {}

    def encode():
        state["yl"] = nat.tts_encode(*targs[:3], noise_w=targs[3], noise_scale_w=0.6, length_scale=1.0, sdp_ratio=0.2)[0]

    def decode():
        nat.tts_decode(2, int(state["yl"].max()), dev, seed=5, noise_scale=0.667, ragged=True)

    try:
        for simple in (0, 1):
            nat.set_option("tts_simple", simple)
            rec[f"tts_encode_simple{simple}"] = _profiled(nat, encode)
        nat.set_option("tts_simple", 0)
        rec["tts_decode"] = _profiled(nat, decode)
        nat.debug_enable(True)
        encode()
        decode()
        torch.cuda.synchronize()
        rec["taps_tts"] = _taps(nat, TTS_TAPS + VC_TAPS)
    finally:
        nat.set_option("tts_simple", 0)
        nat.debug_enable(False)
    return rec


def test_launch_sequence_matches_fixture():
    with open(FIXTURE) as f:
        want = json.load(f)
    got = json.loads(json.dumps(record()))        # same float repr / list types as the fixture
    assert sorted(got) == sorted(want)
    for k in want:
        if isinstance(want[k], dict) and "detail" in want[k]:
            for i, (g, w) in enumerate(zip(got[k]["detail"], want[k]["detail"])):
                assert g == w, (k, i, g, w)
        assert got[k] == want[k], k


def _sd(tts):
    from oracle import tts_oracle as TO
    from oracle import vc_oracle as O
    return TO.synthetic_tts_state_dict() if tts else O.synthetic_state_dict(1234)


@pytest.fixture(scope="module")
def checkpoints():
    return {False: _sd(False), True: _sd(True)}


BROKEN = [   # (key, wrong shape, TTS checkpoint)
    ("enc_q.enc.in_layers.3.weight_v", (384, 192, 3), False),
    ("flow.flows.2.enc.cond_layer.weight_v", (1536, 128, 1), False),
    ("dec.resblocks.4.convs2.1.weight_v", (128, 128, 3), False),
    ("ref_enc.gru.weight_hh_l0", (384, 64), False),
    ("sdp.flows.3.proj.weight", (29, 192, 3), True),
]


@pytest.mark.parametrize("key,shape,tts", BROKEN)
def test_checkpoint_errors_name_the_tensor(key, shape, tts, checkpoints):
    """A fresh context per case: a failed finalize leaves its context unfinalized."""
    from oracle import tts_oracle as TO
    from oracle import vc_oracle as O
    from openvoice_b200._native import OvcError
    from openvoice_b200.api import NativeSynthesizer
    from openvoice_b200.utils import HParams
    hp = copy.deepcopy(O.DEFAULT_HPARAMS)
    if tts:
        hp["data"]["n_speakers"] = TO.TTS_HPARAMS["n_speakers"]
    sd = checkpoints[tts]
    assert key in sd and tuple(sd[key].shape) != shape
    dropped = {k: v for k, v in sd.items() if k != key}
    with pytest.raises(OvcError, match=re.escape(key)):
        NativeSynthesizer(HParams(**hp), "cuda:0").load_state_dict(dropped)
    bad = dict(sd)
    bad[key] = torch.zeros(shape)
    with pytest.raises(ValueError, match=re.escape(key)):
        NativeSynthesizer(HParams(**hp), "cuda:0").load_state_dict(bad)


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(HERE))
    rec = record()
    with open(FIXTURE, "w") as f:
        json.dump(rec, f, indent=0, sort_keys=True)
        f.write("\n")
    print(f"wrote {FIXTURE}: {len(rec)} records")
