"""Generate tests/golden/tts_*.npz by running the REAL reference ``SynthesizerTrn.infer``.

Run in the build container only (``python oracle/make_golden_tts.py``).  Same method as
``make_golden.py``: the reference ships no golden vectors, so the TTS front half (SURVEY.md
section 8 rows a12 / a13 / f3) is pinned on outputs of the reference's own modules --
``SynthesizerTrn.infer`` (openvoice/models.py:467-490) with ``TextEncoder``,
``StochasticDurationPredictor(reverse=True)``, ``DurationPredictor``, ``generate_path`` --
on the seeded synthetic V1-style checkpoint of ``tts_oracle``.  The two RNG draws on the path
(models.py:173 ``torch.randn``, :487 ``torch.randn_like``) are replaced by injected tensors.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.dont_write_bytecode = True

import vc_oracle as V  # noqa: E402
import tts_oracle as T  # noqa: E402
import golden as G  # noqa: E402
from make_golden import import_reference, maxdiff  # noqa: E402


class injected_rng:
    def __init__(self, noise_w, noise):
        self.noise_w, self.noise = noise_w, noise

    def __enter__(self):
        self.o1, self.o2 = torch.randn, torch.randn_like
        torch.randn = lambda *s, **k: self.noise_w.clone()
        torch.randn_like = lambda x, **k: self.noise[:, :, :x.shape[2]].to(x.dtype)

    def __exit__(self, *a):
        torch.randn, torch.randn_like = self.o1, self.o2


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)
    api, mel, models = import_reference()
    hp = V.DEFAULT_HPARAMS
    tts = T.TTS_HPARAMS
    sd = T.synthetic_tts_state_dict()
    model = models.SynthesizerTrn(tts["n_vocab"], hp["data"]["filter_length"] // 2 + 1,
                                  n_speakers=tts["n_speakers"], **hp["model"]).eval()
    ref_sd = model.state_dict()
    schema = T.tts_state_dict_schema()
    for k, shp in schema.items():
        assert k in ref_sd and tuple(ref_sd[k].shape) == tuple(shp), (k, shp)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    assert all(k.startswith("sdp.post_") for k in missing), missing   # training-only members
    model64 = models.SynthesizerTrn(tts["n_vocab"], hp["data"]["filter_length"] // 2 + 1,
                                    n_speakers=tts["n_speakers"], **hp["model"]).eval()
    model64.load_state_dict(sd, strict=False)
    model64.double()

    outdir = os.path.join(ROOT, "tests", "golden")
    report = {}
    cases = [
        ("tts_b1_t37", dict(B=1, T=37, seed=1, lengths=None, noise_scale=0.667, noise_scale_w=0.6, length_scale=1.0, sdp_ratio=0.2)),
        ("tts_b2_padded", dict(B=2, T=50, seed=2, lengths=[50, 31], noise_scale=0.667, noise_scale_w=0.6, length_scale=1.0, sdp_ratio=0.2)),
        ("tts_b1_t121_tails", dict(B=1, T=121, seed=3, lengths=None, noise_scale=0.5, noise_scale_w=2.5, length_scale=1.3, sdp_ratio=0.3)),
    ]
    for name, c in cases:
        tokens, lengths, sid, noise_w = T.synthetic_tts_inputs(c["B"], c["T"], c["seed"], c["lengths"])
        noise = torch.randn(c["B"], 192, 40 * c["T"] + 64, generator=torch.Generator().manual_seed(30_000 + c["seed"]))
        kw = dict(noise_scale=c["noise_scale"], length_scale=c["length_scale"], noise_scale_w=c["noise_scale_w"],
                  sdp_ratio=c["sdp_ratio"])
        with torch.no_grad(), injected_rng(noise_w, noise):
            o, attn, y_mask, (z, z_p, m_y, logs_y) = model.infer(tokens, lengths, sid=sid, **kw)
            x, m_p, logs_p, x_mask = model.enc_p(tokens, lengths)
            g = model.emb_g(sid).unsqueeze(-1)
            logw_s = model.sdp(x, x_mask, g=g, reverse=True, noise_scale=c["noise_scale_w"])
            logw_d = model.dp(x, x_mask, g=g)
        w_ceil = attn[:, 0].sum(1)                         # [B,T]: frames per token
        y_lengths = y_mask[:, 0].sum(1).long()
        with torch.no_grad():
            r = T.tts_infer(sd, tokens, lengths, sid, noise_w, noise, hp=hp, tts=tts, **kw)
        d = dict(x=maxdiff(x, r["x"]), m_p=maxdiff(m_p, r["m_p"]), logs_p=maxdiff(logs_p, r["logs_p"]),
                 logw_sdp=maxdiff(logw_s, r["logw_sdp"]), logw_dp=maxdiff(logw_d, r["logw_dp"]),
                 w_ceil=maxdiff(w_ceil, r["w_ceil"][:, 0]), y_lengths=maxdiff(y_lengths.float(), r["y_lengths"].float()),
                 z_p=maxdiff(z_p, r["z_p"]), z=maxdiff(z, r["z"]), o=maxdiff(o, r["o"]),
                 frames=[int(v) for v in y_lengths],
                 outside_tail=int(((noise_w * c["noise_scale_w"]).abs() > 5).sum()))
        # fp64 twin of the reference = the noise floor of its own fp32 arithmetic (floor_*).  A CPU with another vector
        # width or thread count rounds the fp32 oracle differently, so the oracle's tolerances are set from these floors.
        with torch.no_grad(), injected_rng(noise_w.double(), noise.double()):
            o64, _, _, (z64, z_p64, _, _) = model64.infer(tokens, lengths, sid=sid, **kw)
            x64, m_p64, logs_p64, x_mask64 = model64.enc_p(tokens, lengths)
            g64 = model64.emb_g(sid).unsqueeze(-1)
            logw_s64 = model64.sdp(x64, x_mask64, g=g64, reverse=True, noise_scale=c["noise_scale_w"])
            logw_d64 = model64.dp(x64, x_mask64, g=g64)
        for k, a, b in (("x", x, x64), ("m_p", m_p, m_p64), ("logs_p", logs_p, logs_p64), ("logw_sdp", logw_s, logw_s64),
                        ("logw_dp", logw_d, logw_d64), ("z_p", z_p, z_p64), ("z", z, z64), ("o", o, o64)):
            d["floor_" + k] = maxdiff(a.double(), b)
        report[name] = d
        arrays = dict(x=x.numpy(), m_p=m_p.numpy(), logs_p=logs_p.numpy(), logw_sdp=logw_s.numpy(), logw_dp=logw_d.numpy(),
                      w_ceil=w_ceil.numpy(), y_lengths=y_lengths.numpy(), z_p=z_p.numpy(), z=z.numpy(), o=o.numpy(),
                      meta=np.array(json.dumps(c)))
        if name == "tts_b1_t121_tails":     # 723 frames: whole z_p / z / o would take the file to 2 MB
            arrays = G.sample(arrays, ("z_p", "z", "o"), 0.25)
        np.savez_compressed(os.path.join(outdir, name + ".npz"), **arrays)
    with open(os.path.join(outdir, "REPORT_tts.json"), "w") as f:
        json.dump(report, f, indent=1, sort_keys=True)
    print(json.dumps(report, indent=1, sort_keys=True))


if __name__ == "__main__":
    main()
