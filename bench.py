#!/usr/bin/env python
"""bench.py — CT slices/sec @256x256 through the B200 engine, per the driver contract.

    python bench.py --gpus N --steps K --warmup W              # this repo's engine, BASELINE config C2 (the headline)
    python bench.py --config C3|C4|C5 ...                       # the other BASELINE.json configurations
    python bench.py --mode shard --gpus N ...                   # ONE volume's slices sharded over the N GPUs (latency)
    python bench.py --impl reference ...                        # the CPU port of the reference path (oracle) on host cores

One "step" = one full pass of the hot path (preprocess -> U-Net forward -> postprocess -> reshape) over the
configuration's synthetic int16 CT volume(s) on every GPU:
    C2  R231 (3 classes), one 300-slice 256x256 volume, reference batch_size 20           (BASELINE configs[1], default)
    C3  LTRCLobes (6 classes), one 512-slice volume, batch_size 32                          (configs[2])
    C4  LTRCLobes_R231 fusion: two models + spare-label fusion + post-processing, 300 slices (configs[3])
    C5  R231 throughput: 64 volumes x 512 slices over 8 GPUs = 8 volumes per GPU and step  (configs[4])
`value` is measured with the volume(s) already resident in HBM (lm_apply_volume_dev / lm_apply_fused_dev), `e2e`
through the public API (LMInferer.apply) with a pinned host input and a host output, copies inside the timed region.
Multi-GPU, --mode replica (default): one process per GPU, every rank segments its own volume(s) per step (volumes are
independent objects -> weak scaling, no data-path collective) and the uint8 label volumes are all-gathered over NCCL
at the end of each step as the north-star asks.  --mode shard: every rank holds the same volume and computes a
contiguous slab of its slices; the engine all-gathers the argmax slabs itself (CUDA-IPC peer stores, csrc/shard.cu)
and every rank post-processes the whole volume -> strong scaling of one volume's latency.
The line also carries the parity of the run: Dice / argmax flips / differing voxels of the engine against the CPU
oracle on the bounded sample the CPU baseline is timed on.
--dump-outputs DIR writes what the timed path returned in its last timed step (rank 0's label volumes) as
DIR/<name>.npy in float32, so that two builds run with the same arguments (same seeded volumes and weights) can be
compared output for output.
"""
import argparse
import json
import os
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL's version / debug lines must not precede the JSON line on stdout
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RES = 256
S_VOL = 300  # C2 (kept as a module constant: tests import it)
STEM_GFLOP = 0.0755
CONFIGS = {
    # K: classes of the (base) model; fill: classes of the fill model (fusion); S: slices per volume; vols: volumes per GPU and step
    "C2": dict(K=3, fill=None, S=300, batch=20, vols=1, gflop=96.20,
               desc="R231 (3-class) 300-slice 256x256 int16 synthetic CT volume per GPU, batch_size=20 (engine waves of %d slices)"),
    "C3": dict(K=6, fill=None, S=512, batch=32, vols=1, gflop=96.23,
               desc="LTRCLobes (6-class) 512-slice 256x256 int16 synthetic CT volume per GPU, batch_size=32 (engine waves of %d slices)"),
    "C4": dict(K=6, fill=3, S=300, batch=20, vols=1, gflop=96.23 + 96.20,
               desc="LTRCLobes_R231 fusion (6-class base + 3-class fill model, spare-label fusion, post-processing at original "
                    "resolution) on a 300-slice 256x256 int16 synthetic CT volume per GPU"),
    "C5": dict(K=3, fill=None, S=512, batch=20, vols=8, gflop=96.20,
               desc="R231 throughput: 8 volumes x 512 slices (256x256 int16, synthetic) per GPU and step = 64 volumes over 8 GPUs"),
}
WEIGHT_SEEDS = {3: 7, 6: 8}
# mean dram__bytes_read.sum + dram__bytes_write.sum per conv_tc_kernel launch: taken from the newest committed ncu --set full
# summary that tools/ncu_summarize.py wrote (profiles/*conv_traffic.json: per-layer table of one full 37-slice wave)
TRAFFIC_FALLBACK = (188.7e6, "profiles/r01_ncu_summary_v5.md (4 launches of a 37-slice wave, layers down2/down3)")
DUMP_BYTES = 64 * 10**6   # --dump-outputs writes at most this much in all


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def dump_outputs(out_dir, outputs):
    """Writes every {name: array} as out_dir/<name>.npy in float32.  An output larger than its share of DUMP_BYTES is
    written as a fixed sample instead: its values at seeded random flat indices, in index order, as a 1-D array."""
    os.makedirs(out_dir, exist_ok=True)
    share = (DUMP_BYTES // len(outputs) - 4096) // 4   # float32 elements per file, room left for the .npy header
    for name, a in outputs.items():
        a = np.asarray(a)
        if a.size > share:
            idx = np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))
            log("dump %s: %d of %d values of shape %s (seeded sample)" % (name, share, a.size, a.shape))
            a = a.ravel()[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def rank_info():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def conv_traffic():
    """(mean DRAM bytes per conv launch, source) from the newest per-layer table under profiles/."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_conv_traffic.json")))
    if files:
        try:
            d = json.load(open(files[-1]))
            return float(d["mean_bytes_per_launch"]), os.path.relpath(files[-1], ROOT) + " (%d launches of one wave)" % d["launches"]
        except Exception:
            pass
    return TRAFFIC_FALLBACK


def get_weights(K, seed, steps=60):
    """Seeded 'trained-looking' synthetic weights with the reference's layout (no network for the released .pth)."""
    import torch
    from oracle import synth
    path = "/tmp/lm_b200_synth_K%d_s%d_t%d_r%s.pth" % (K, seed, steps, os.environ.get("LOCAL_RANK", "0"))
    if os.path.exists(path):
        return torch.load(path, map_location="cpu")
    t0 = time.time()
    sd = synth.train_state_dict(K, seed=seed, steps=steps, log=log)
    torch.save(sd, path)
    log("synthetic weights trained in %.1fs" % (time.time() - t0))
    return sd


class ClockSampler(threading.Thread):
    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.samples, self.reasons, self.stop_flag = gpu_index, [], set(), False
        self.max_mhz = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.2)

    def result(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


def _cpu_threads():
    import torch
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use the host's cores.  torch's own default is one
    # thread per physical core (64 on the GPU box: 128 hyper-threads measured 2.7x slower), so restore that.
    if torch.get_num_threads() == 1 and (os.cpu_count() or 1) > 2:
        torch.set_num_threads(max(1, (os.cpu_count() or 2) // 2))
    return torch.get_num_threads()


def cpu_port(cfg, sds, sample, taps=None):
    """The oracle port of the reference path (mask.py:141-232) on the host cores, on `sample`; returns (seconds, output)."""
    from oracle import restate
    _cpu_threads()
    t0 = time.perf_counter()
    if cfg["fill"] is None:
        out = restate.inference(sample, sds[0], batch_size=cfg["batch"], taps=taps)
    else:
        out = restate.apply(sample, sds[0], fill_sd=sds[1], batch_size=cfg["batch"])
    return time.perf_counter() - t0, out


def dice_min(a, b):
    out = []
    for v in np.union1d(np.unique(a), np.unique(b)):
        if v == 0:
            continue
        x, y = a == v, b == v
        out.append(2.0 * float((x & y).sum()) / max(1, int(x.sum() + y.sum())))
    return min(out) if out else 1.0


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path = oracle port (the reference is
    pure Python over torch/scipy; its third-party natives skimage/fill_voids are restated in oracle/standins)."""
    rank, _, world = rank_info()
    if rank != 0:
        return
    import torch
    from oracle import synth
    cfg = CONFIGS[args.config]
    sds = [get_weights(cfg["K"], WEIGHT_SEEDS[cfg["K"]])] + ([get_weights(cfg["fill"], WEIGHT_SEEDS[cfg["fill"]])] if cfg["fill"] else [])
    vol = synth.phantom(cfg["S"], seed=100)
    n = cfg["batch"] if cfg["fill"] is None else max(4, cfg["batch"] // 2)  # bounded sample per step: one reference batch
    sample = vol[:n]
    for _ in range(args.warmup):
        cpu_port(cfg, sds, sample)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        _, out = cpu_port(cfg, sds, sample)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"labels": out})
    v = n * args.steps / dt
    cores = torch.get_num_threads()
    line = {"impl": "reference", "metric": "CT slices/sec @256x256 (%s)" % ("R231" if args.config in ("C2", "C5") else args.config), "value": v, "unit": "slices/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["desc"].replace("%d", "37"), "config": args.config, "sample": "first %d slices of the volume per step" % n},
            "cpu_baseline": {"value": v, "unit": "slices/s", "cores": cores, "kind": "port",
                             "sample": "%d slices per step (oracle port of mask.py:141-232 on host cores)" % n},
            "e2e": {"value": v, "unit": "slices/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_engine(args):
    import torch
    import torch.distributed as dist
    rank, local_rank, world = rank_info()
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from lungmask_b200 import LMInferer
    from lungmask_b200 import parallel
    from lungmask_b200.logger import logger as lm_logger
    from oracle import synth
    import logging
    lm_logger.setLevel(logging.WARNING)   # the reference logs "Apply: ..." to stdout; stdout carries the JSON line here

    cfg = CONFIGS[args.config]
    shard = args.mode == "shard"
    K, S, nv = cfg["K"], cfg["S"], (1 if shard else cfg["vols"])
    fused = cfg["fill"] is not None
    if shard and fused:
        raise SystemExit("--mode shard covers the single-model path (C2 / C3 / C5 volumes)")
    sds = [get_weights(K, WEIGHT_SEEDS[K])] + ([get_weights(cfg["fill"], WEIGHT_SEEDS[cfg["fill"]])] if fused else [])
    paths = []
    for i, sd in enumerate(sds):
        p = "/tmp/lm_b200_bench_%s_%d_rank%d.pth" % (args.config, i, local_rank)
        torch.save(sd, p)
        paths.append(p)
    if fused:
        inferer = LMInferer(modelname="LTRCLobes", modelpath=paths[0], fillmodel="R231", fillmodel_path=paths[1],
                            batch_size=cfg["batch"], tqdm_disable=True, device=local_rank)
    else:
        inferer = LMInferer(modelname="R231", modelpath=paths[0], batch_size=cfg["batch"], tqdm_disable=True, device=local_rank)
    eng = inferer.engine
    eng.set_option("time_convs", 1)
    if shard:
        parallel.connect(eng, rank, world, S)

    # shard mode: the SAME volume on every rank; replica mode: every rank (and volume slot) its own phantom
    vols = [synth.phantom(S, seed=100 + (0 if shard else rank * nv + i)) for i in range(nv)]
    d_vols = [torch.from_numpy(v).cuda() for v in vols]
    d_outs = [torch.empty(v.shape, dtype=torch.uint8, device="cuda") for v in vols]
    gathered = torch.empty((world, nv) + vols[0].shape, dtype=torch.uint8, device="cuda") if (world > 1 and not shard) else None
    h_vols = [torch.from_numpy(v).pin_memory().numpy() for v in vols]
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_dev(i):
        if shard:
            eng.apply_volume_sharded_dev(0, d_vols[i].data_ptr(), vols[i].shape, d_outs[i].data_ptr())
        elif fused:
            eng.apply_fused_dev(0, 1, d_vols[i].data_ptr(), vols[i].shape, d_outs[i].data_ptr())
        else:
            eng.apply_volume_dev(0, d_vols[i].data_ptr(), vols[i].shape, d_outs[i].data_ptr())

    stage, acc = {}, {"conv_ms": 0.0, "conv_launches": 0, "launches": 0}

    def step_dev(record):
        for i in range(nv):
            one_dev(i)
            if record:
                t = eng.last_timings()
                acc["launches"] += t["kernel_launches"]
                cm, cl = eng.last_conv_timing()
                acc["conv_ms"] += cm
                acc["conv_launches"] += cl
                for k in ("preprocess", "forward", "postprocess", "reshape"):
                    stage[k] = stage.get(k, 0.0) + t[k]
        if gathered is not None:
            dist.all_gather_into_tensor(gathered, torch.stack(d_outs) if nv > 1 else d_outs[0].unsqueeze(0))
            torch.cuda.synchronize()

    # ---- device-resident throughput (value) ------------------------------------------------------------
    for _ in range(args.warmup):
        step_dev(False)
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_dev(True)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    sampler.stop_flag = True
    last_step = {"labels_vol%d" % i: d.cpu().numpy() for i, d in enumerate(d_outs)} if (args.dump_outputs and rank == 0) else None
    # every engine call ends with a stream synchronisation, so the bracketed wall time between the two synchronised
    # barriers IS the device-side duration of the K steps
    step_ms = wall_ms / args.steps
    if world > 1:
        tt = torch.tensor([step_ms], device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        step_ms = float(tt.item())
    slices_per_step = S if shard else world * nv * S
    value = slices_per_step / (step_ms * 1e-3)

    # ---- end to end through the public API (host in / host out) ----------------------------------------
    eng.set_option("time_convs", 0)
    res = None

    def step_e2e():
        out = None
        for i in range(nv):
            if shard:  # every rank copies its slab in; rank 0 reads the whole result back
                out = parallel.apply_sharded_device(eng, 0, h_vols[i], want_output=(rank == 0))
            else:
                out = inferer.apply(h_vols[i])
            if out is not None:
                _ = int(out[::37].sum())  # read the result on the host
        return out

    for _ in range(max(1, args.warmup // 2)):
        res = step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = step_e2e()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    if world > 1:
        tt = torch.tensor([e2e_ms], device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_ms = float(tt.item())
    e2e_value = slices_per_step / (e2e_ms * 1e-3)
    same = bool(np.array_equal(res, d_outs[nv - 1].cpu().numpy())) if res is not None else None
    if shard:
        lo, hi = parallel.shard_range(S, rank, world)
        h2d, d2h = (hi - lo) * RES * RES * 2, (S * RES * RES if rank == 0 else 0)
    else:
        h2d, d2h = nv * int(vols[0].nbytes), nv * int(vols[0].size)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (cuBLAS bf16, kernel timed inside a long step)" if peaks else "fallback 1.4 PFLOP/s sustained"
        my_slices = (parallel.shard_range(S, 0, world)[1] if shard else nv * S)
        flops_timed = (cfg["gflop"] - STEM_GFLOP * (2 if fused else 1)) * 1e9 * my_slices * args.steps  # rank 0's convolutions
        achieved = flops_timed / (acc["conv_ms"] * 1e-3) / 1e12 if acc["conv_ms"] > 0 else None
        traffic, traffic_src = conv_traffic()
        # CPU baseline + parity: the oracle port on this box's host cores on a bounded sample, the engine on the same sample
        n_cpu = 16 if not fused else 8
        sample = vols[0][:n_cpu]
        taps = {} if not fused else None
        cpu_s, want = cpu_port(cfg, sds, sample, taps=taps)
        cores = _cpu_threads()
        eng2 = inferer.engine
        got = eng2.apply_fused(0, 1, sample) if fused else eng2.apply_volume(0, sample)
        parity = {"sample": "first %d slices of the step's volume, engine vs CPU oracle on the same sub-volume" % n_cpu,
                  "dice": dice_min(got, want), "voxels_differing": int((got != want).sum()), "voxels": int(want.size)}
        if taps is not None:
            resized, _ = eng2.preprocess(sample)
            labels, scores = eng2.forward(0, resized, return_scores=True)
            parity["label_flips"] = int((labels != taps["labels"]).sum())
            parity["max_abs_score_err"] = float(np.abs(scores - taps["scores"]).max())
            parity["preprocess_bit_exact"] = bool(np.array_equal(resized, taps["resized"]))
        line = {
            "metric": "CT slices/sec @256x256 (%s)" % ("R231" if args.config in ("C2", "C5") else args.config),
            "value": value, "unit": "slices/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": "strong" if shard else "weak", "vs_baseline": None,
            "dtype": "f16x3 (fp32-class: every fp32 value is an fp16 hi + scaled fp16 lo pair, 3 exact products per MAC, fp32 accumulate)",
            "data": "synthetic",
            "dice": parity["dice"], "label_flips": parity.get("label_flips"),
            "config": {"workload": cfg["desc"].replace("%d", str(inferer.wave_slices)), "config": args.config, "mode": args.mode, "volumes_per_step_per_gpu": nv,
                       "slices_per_step": slices_per_step,
                       "l2": "inputs larger than L2: %d MB volume, ~%d GB of activations per %d-slice wave" % (vols[0].nbytes >> 20, round(0.16 * inferer.wave_slices), inferer.wave_slices),
                       "weights": "seeded synthetic state_dict, 60 Adam steps on phantoms (released .pth needs network)",
                       "stage_ms_per_step": {k: v / args.steps for k, v in stage.items()},
                       "engine_env_options": {k: os.environ[k] for k in sorted(os.environ) if k.startswith("LM_") and k != "LM_TEST_EXPERIMENTAL"},
                       "e2e_matches_device_path": same, "parity": parity},
            "e2e": {"value": e2e_value, "unit": "slices/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(acc["launches"]),
            "clocks": sampler.result(),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "conv_tc kernels (tcgen05 kind::f16, 3 products per algorithmic MAC => ceiling 1/3 of the bf16 peak)",
                         "launches_timed": int(acc["conv_launches"]), "avg_launch_ms": acc["conv_ms"] / max(1, acc["conv_launches"]),
                         "peak_source": peak_src, "algorithmic_flops_per_step": flops_timed / args.steps},
            "cpu_baseline": {"value": n_cpu / cpu_s, "unit": "slices/s", "cores": cores, "kind": "port",
                             "sample": "first %d slices of the same volume, full path (oracle port of mask.py:141-232)" % n_cpu},
        }
        print(json.dumps(line), flush=True)
        if last_step is not None:
            dump_outputs(args.dump_outputs, last_step)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--mode", default="replica", choices=["replica", "shard"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_engine(args)


if __name__ == "__main__":
    main()
