#!/usr/bin/env python
"""Parity of the tensor-core path vs the CPU oracle, stage by stage, for every tiling of the wide kernel."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
from oracle import vc_oracle as O
from openvoice_b200.api import NativeSynthesizer
from openvoice_b200.utils import HParams


def rel(a, b):
    b = np.asarray(b, np.float64)
    return float(np.abs(np.asarray(a, np.float64) - b).max() / (np.sqrt((b ** 2).mean()) + 1e-30))


def per_tile(a, b, tile):
    """max error / rms per block of `tile` time steps (arrays [B, C, T]); nan -> 9.9"""
    b = np.asarray(b, np.float64)
    e = np.abs(np.asarray(a, np.float64) - b)
    e[np.isnan(e)] = 9.9 * np.sqrt((b ** 2).mean())
    e = e.max(axis=(0, 1)) / np.sqrt((b ** 2).mean())
    return " ".join(f"{e[i:i + tile].max():.0e}" for i in range(0, len(e), tile))


def first_bad(a, b):
    """first time index where the error exceeds 1e-3 * rms (arrays [B, C, T])"""
    b = np.asarray(b, np.float64)
    e = np.abs(np.asarray(a, np.float64) - b)
    e[np.isnan(e)] = 1e9
    bad = np.where(e.max(axis=(0, 1)) > 1e-3 * np.sqrt((b ** 2).mean()))[0]
    return (int(bad[0]), int(bad[-1]), len(bad)) if len(bad) else None


sd = O.synthetic_state_dict(1234)
m = NativeSynthesizer(HParams(**O.DEFAULT_HPARAMS), "cuda:0")
m.load_state_dict(sd)
T = int(sys.argv[1]) if len(sys.argv) > 1 else 300
B, lens = 2, [T, T - 29]
spec, lengths, gs, gt, noise = O.synthetic_inputs(B, T, 3, lengths=lens)
taps = {}
with torch.no_grad():
    ro, _, (rz, rzp, rzh) = O.voice_conversion(sd, spec, lengths, gs, gt, noise, 0.3, taps=taps)
summary = {}
names = ["enc.wn", "dec.pre", "dec.ups0", "dec.stage0", "dec.ups1", "dec.stage1", "dec.ups2", "dec.stage2", "dec.ups3", "dec.stage3"]
for mode, wv, pair in (("fp32", 0, 0), ("f16x3", 3, 0), ("f16x3", 3, 1), ("f16x3", 0, 0), ("f16x3", 2, 0), ("f16", 3, 0), ("f16", 3, 1)):
    m.native.set_precision(mode)
    m.native.set_option("wide_variant", wv)
    m.native.set_option("pair", pair)
    m.native.debug_enable(True)
    o, _, lat = m.voice_conversion(spec.cuda(), lengths.cuda(), gs.cuda(), gt.cuda(), tau=0.3, noise=noise.cuda(), ragged=False)
    torch.cuda.synchronize()
    print(mode, "wide_variant", wv, "pair", pair, "o_hat", f"{rel(o.cpu().numpy(), ro.numpy()):.3e}", "z", f"{rel(lat[0].cpu().numpy(), rz.numpy()):.3e}",
          "z_hat", f"{rel(lat[2].cpu().numpy(), rzh.numpy()):.3e}")
    for name in names:
        if name not in taps:
            continue
        got = m.native.debug_fetch(name)
        print("   ", name, f"{rel(got, taps[name].numpy()):.3e}", "first/last/count bad t:", first_bad(got, taps[name].numpy()), "of", got.shape[-1])
        if name in ("dec.ups0", "dec.stage0", "dec.ups1") and mode != "fp32":
            print("        per 128-step tile:", per_tile(got, taps[name].numpy(), 128)[:600])
    m.native.debug_enable(False)
    o2, _, _ = m.voice_conversion(spec.cuda(), lengths.cuda(), gs.cuda(), gt.cuda(), tau=0.3, noise=noise.cuda(), ragged=True)
    with torch.no_grad():
        qo, _, _ = O.voice_conversion_ragged(sd, spec, lengths, gs, gt, noise, 0.3)
    e2 = rel(o2.cpu().numpy(), qo.numpy())
    print("    ragged o_hat", f"{e2:.3e}")
    summary[f"{mode}:{wv}:{pair}"] = max(rel(o.cpu().numpy(), ro.numpy()), e2)
import json
for k in summary:
    if not np.isfinite(summary[k]):
        summary[k] = 1e9
json.dump(summary, open(os.path.join(ROOT, "gpurun_out", "tc_check_summary.json"), "w"))
print("tc_check done", summary)
