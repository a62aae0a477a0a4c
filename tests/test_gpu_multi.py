"""Two (or four) GPUs, one process each: one volume's slices sharded over the ranks (SURVEY.md 8e).  The engine's own
device-side gather (CUDA-IPC mapped gather blocks, slab pushed over NVLink, csrc/shard.cu) must give every rank the
single-GPU result bit for bit, and so must the stage-level path with an NCCL all_gather_into_tensor.  Skipped on
boxes with one GPU (the driver's round-end GPU test box); run with `gpurun --gpus 2`."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    sys.path.insert(0, ROOT)
    try:
        import torch
        import torch.distributed as dist
        from lungmask_b200 import _native
        from lungmask_b200.mask import NativeModel
        from lungmask_b200.parallel import apply_sharded, apply_sharded_device, connect
        from oracle import synth
        torch.cuda.set_device(rank)
        dist.init_process_group("cpu:gloo,cuda:nccl", rank=rank, world_size=world)
        eng = _native.Engine(device=rank, batch_capacity=8)
        m = NativeModel(synth.random_state_dict(3, seed=5, head_gain=0.3))
        eng.load_weights(0, m.blob, m.n_classes)
        connect(eng, rank, world, 64)
        ok = True
        for S, shape in ((21, (150, 170)), (3, (256, 256)), (1, (64, 80))):   # odd split, one slice per rank + idle rank, single slice
            vol = synth.phantom(S, shape[0], shape[1], seed=40 + S)
            want = eng.apply_volume(0, vol)                       # the whole volume on this rank's GPU
            got = apply_sharded_device(eng, 0, vol)               # engine gather (P2P pushes + epoch flags)
            got2 = apply_sharded_device(eng, 0, vol)              # again: epochs advance, blocks are reused
            via_nccl = apply_sharded(eng, 0, vol, rank, world, device="cuda:%d" % rank)
            raw = apply_sharded_device(eng, 0, vol, postprocess=False)
            ok = ok and np.array_equal(got, want) and np.array_equal(got2, want) and np.array_equal(via_nccl, want)
            ok = ok and np.array_equal(raw, eng.apply_volume(0, vol, postprocess=False))
            eng.set_option("shard_slab_ccl", 0)           # every rank labels the whole gathered volume instead
            ok = ok and np.array_equal(apply_sharded_device(eng, 0, vol), want)
            eng.set_option("shard_slab_ccl", 1)
        q.put((rank, bool(ok), ""))
        dist.barrier()
        dist.destroy_process_group()
        eng.close()
    except Exception as ex:  # report instead of leaving the parent waiting
        import traceback
        q.put((rank, False, traceback.format_exc()[-1500:]))


def test_sharded_volume_equals_single_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    import torch.multiprocessing as mp
    world = int(os.environ.get("LM_TEST_WORLD", min(torch.cuda.device_count(), 4)))   # 2 ranks, or 4 on a box with >= 4 GPUs
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=120)
    print("world size", world)
    assert sorted((r, ok) for r, ok, _ in res) == [(r, True) for r in range(world)], [msg for _, _, msg in res]


def test_shard_world_one_is_the_plain_path(engine):
    """world = 1: no peers, no pushes; lm_apply_volume_sharded must equal lm_apply_volume (runs on any GPU box)."""
    from lungmask_b200.mask import NativeModel
    from oracle import synth
    m = NativeModel(synth.random_state_dict(3, seed=5, head_gain=0.3))
    engine.load_weights(0, m.blob, m.n_classes)
    engine.shard_init(0, 1, 16)
    vol = synth.phantom(5, 180, 200, seed=12)
    assert np.array_equal(engine.apply_volume_sharded(0, vol), engine.apply_volume(0, vol))
    assert np.array_equal(engine.apply_volume_sharded(0, vol, postprocess=False), engine.apply_volume(0, vol, postprocess=False))
    with pytest.raises(Exception):
        engine.apply_volume_sharded(0, synth.phantom(17, 64, 64, seed=1))   # beyond the gather capacity
    # slab-sharded 3-D labelling: virtual slabs on one GPU (each labelled on its own, boundaries joined afterwards) must
    # reproduce the whole-volume labelling, hence the same post-processing, bit for bit - also without slab labelling
    vol = synth.phantom(13, 150, 170, seed=14)
    want = engine.apply_volume(0, vol)
    for slabs in (2, 3, 8, 13):
        engine.set_option("shard_test_slabs", slabs)
        try:
            assert np.array_equal(engine.apply_volume_sharded(0, vol), want), slabs
        finally:
            engine.set_option("shard_test_slabs", 0)
    engine.set_option("shard_slab_ccl", 0)
    try:
        assert np.array_equal(engine.apply_volume_sharded(0, vol), want)
    finally:
        engine.set_option("shard_slab_ccl", 1)
