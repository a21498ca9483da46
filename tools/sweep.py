#!/usr/bin/env python
"""BASELINE.json configs[4]: length x batch sweep of ToneColorConverter.convert_batch on one GPU (host arrays in, host
arrays out, launches of at most --max-batch utterances), audio-seconds per second.

  python tools/sweep.py [--json out.json] [--points "1x1,1x3,1x10,1x30,8x3,8x10,32x10,64x30,128x10,256x3,256x30"]
"""
import argparse
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", default="1x1,1x3,1x10,1x30,8x3,8x10,32x10,64x30,128x10,256x3,256x30")
    ap.add_argument("--max-batch", type=int, default=64)
    ap.add_argument("--precision", default="f16x3")
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    from oracle import vc_oracle as O
    from openvoice_b200.api import ToneColorConverter

    with tempfile.TemporaryDirectory() as td:
        cfg = os.path.join(td, "config.json")
        json.dump(O.DEFAULT_HPARAMS, open(cfg, "w"))
        conv = ToneColorConverter(cfg, device="cuda:0", enable_watermark=False, precision=args.precision)
    conv.model.load_state_dict(O.synthetic_state_dict(1234))
    gen = torch.Generator().manual_seed(0)
    src, tgt = 0.1 * torch.randn(1, 256, 1, generator=gen), 0.1 * torch.randn(1, 256, 1, generator=gen)
    rows = []
    for pt in args.points.split(","):
        B, secs = pt.split("x")
        B, secs = int(B), float(secs)
        L = int(round(secs * 22050))
        rng = np.random.default_rng(B * 1000 + int(secs))
        waves = [(0.5 * (2 * rng.random(L, dtype=np.float32) - 1)).astype(np.float32) for _ in range(B)]
        audio_s = B * (L // 256 * 256) / 22050
        reps = 3 if audio_s > 200 else 8
        for _ in range(2):
            conv.convert_batch(waves, src, tgt, tau=0.3, max_batch=args.max_batch)
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            out = conv.convert_batch(waves, src, tgt, tau=0.3, max_batch=args.max_batch)
            ts.append(time.perf_counter() - t0)
        assert len(out) == B and np.isfinite(out[-1]).all()
        ms = 1e3 * float(np.median(ts))
        nat = conv.model.native
        # device workspace of one chunk of max_batch utterances (T = L // 256 frames), in this precision mode
        ws_gb = nat.lib.ovc_workspace_floats(nat.handle, min(B, args.max_batch), L // 256) * 4e-9
        rows.append({"batch": B, "secs": secs, "ms": ms, "audio_s_per_s": audio_s / (ms * 1e-3),
                     "launches_last_chunk": int(nat.last_launch_count), "graph_replays": int(nat.graph_replays),
                     "workspace_gb": ws_gb})
        print(f"B={B:4d} x {secs:5.1f} s: {ms:9.2f} ms  {rows[-1]['audio_s_per_s']:9.1f} audio-s/s  workspace {ws_gb:6.2f} GB",
              flush=True)
    res = {"what": f"ToneColorConverter.convert_batch, host numpy in / out, max_batch {args.max_batch}, {args.precision}, "
                   "median wall time, one B200", "points": rows}
    if args.json:
        json.dump(res, open(args.json, "w"), indent=1)


if __name__ == "__main__":
    main()
