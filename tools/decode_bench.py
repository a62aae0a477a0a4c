"""Decode throughput of lm_decode_frames on a CT-sized series (needs one GPU).

    python tools/decode_bench.py [--slices 300] [--size 512] [--iters 10] [--out decode_bench.json]

A seeded CT-like series (oracle.synth.phantom) is encoded as JPEG Lossless (predictor 1, the .4.70 syntax) and as RLE
Lossless.  For each codec: one lm_decode_frames call for the whole series, timed after warm-up with CUDA events and a
host clock (the call copies the compressed bytes in, decodes, copies the samples out and synchronises), and a kernel
breakdown from torch.profiler in a separate call.  Then read_dicoms on the series written as files, and LMInferer.apply
on the decoded volume for scale.  The card's name and power limit are recorded in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from collections import defaultdict

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # the numbers stay, but say that the card could not be read
        q = "unknown (%s)" % e
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--slices", type=int, default=300)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default="decode_bench.json")
    a = ap.parse_args()

    import torch
    from lungmask_b200 import LMInferer, _native, io as lio
    from oracle import dicom_codecs as dc, synth

    vol = synth.phantom(a.slices, a.size, a.size, seed=7)
    t0 = time.perf_counter()
    enc = {"jpeg_lossless_p1": [dc.jpeg_lossless_encode(s, P=16, predictor=1) for s in vol]}
    t_jpeg = time.perf_counter() - t0
    t0 = time.perf_counter()
    enc["rle"] = [dc.rle_encode(s) for s in vol]
    t_rle = time.perf_counter() - t0
    res = {"card": card(), "slices": a.slices, "rows": a.size, "cols": a.size, "iters": a.iters,
           "encode_s": {"jpeg_lossless_p1": round(t_jpeg, 2), "rle": round(t_rle, 2)}, "codecs": {}}
    out_bytes = vol.size * 2
    for name, streams in enc.items():
        codec = 2 if name == "rle" else 1
        frames = np.zeros(len(streams), _native.FRAME_DTYPE)
        off = 0
        for i, s in enumerate(streams):
            frames[i] = (off, len(s), codec, a.size, a.size, 1)
            off += len(s)
        data = b"".join(streams)
        arrays, status = _native.decode_frames(data, frames, 0)          # warm-up + correctness
        assert not status.any(), status
        assert np.array_equal(np.stack(arrays).view(np.int16), vol), name
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.iters)]
        wall = []
        for e0, e1 in ev:
            t0 = time.perf_counter()
            e0.record()
            _native.decode_frames(data, frames, 0)
            e1.record()
            e1.synchronize()
            wall.append(time.perf_counter() - t0)
        ms = sorted(e0.elapsed_time(e1) for e0, e1 in ev)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            _native.decode_frames(data, frames, 0)
        kern = defaultdict(lambda: [0.0, 0])
        for e in prof.events():
            if e.device_type.name == "CUDA":
                k = e.name.split("(")[0].replace("void ", "").replace("lm_decode::", "")
                kern[k][0] += e.device_time_total / 1000.0 if hasattr(e, "device_time_total") else e.cuda_time_total / 1000.0
                kern[k][1] += 1
        med = ms[len(ms) // 2]
        res["codecs"][name] = {
            "compressed_MB": round(len(data) / 1e6, 2), "ratio": round(out_bytes / len(data), 3),
            "ms_per_series_median": round(med, 3), "ms_min": round(ms[0], 3), "ms_max": round(ms[-1], 3),
            "host_wall_ms_median": round(sorted(wall)[len(wall) // 2] * 1e3, 3),
            "decoded_GBps": round(out_bytes / (med * 1e-3) / 1e9, 2),
            "kernels_ms": {k: [round(v[0], 3), v[1]] for k, v in sorted(kern.items(), key=lambda kv: -kv[1][0])},
        }
        print(name, json.dumps(res["codecs"][name]), flush=True)

    with tempfile.TemporaryDirectory() as tmp:
        for name, streams in enc.items():
            d = os.path.join(tmp, name)
            os.makedirs(d)
            syntax = dc.RLE_LOSSLESS if name == "rle" else dc.JPEG_LOSSLESS_SV1
            for k, s in enumerate(streams):
                dc.write_encapsulated(os.path.join(d, "im%04d.dcm" % k), s, syntax, a.size, a.size, "1.2.826.1",
                                      (0.0, 0.0, 1.25 * k))
            lio.read_dicoms(d)                                            # warm (page cache, module)
            t0 = time.perf_counter()
            v = lio.read_dicoms(d)[0]
            res["codecs"][name]["read_dicoms_s"] = round(time.perf_counter() - t0, 3)
            assert np.array_equal(v.array, vol)
        w = os.path.join(tmp, "w.pth")
        torch.save(synth.random_state_dict(3, seed=13, head_gain=0.3), w)
        inf = LMInferer(modelpath=w, tqdm_disable=True, batch_size=20)
        inf.apply(vol)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        inf.apply(vol)
        res["lminferer_apply_s"] = round(time.perf_counter() - t0, 3)
    print(json.dumps(res))
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
