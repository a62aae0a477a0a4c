"""Host-side logic that needs no GPU: the C-ABI library loads and exports every symbol the header declares,
the state_dict -> blob packing, argument validation of the reference-compatible surface, slice sharding,
and a world_size-2 gloo run of the multi-rank path."""
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from lungmask_b200 import _native
    header = open(os.path.join(ROOT, "include", "lungmask_b200.h")).read()
    declared = set(re.findall(r"LM_API\s+[\w\s\*]+?\b(lm_[a-z_0-9]+)\s*\(", header))
    assert len(declared) >= 20
    L = _native.lib()
    for name in declared:
        assert hasattr(L, name), name
    assert declared == set(_native.EXPORTS)


def test_blob_packing_matches_native_size():
    from lungmask_b200 import _native
    from lungmask_b200.mask import NativeModel
    from oracle import synth
    for K in (3, 6):
        sd = synth.random_state_dict(K, seed=1, calibrate_on=np.zeros((1, 256, 256), np.float32) + 0.5)
        m = NativeModel(sd)
        assert m.n_classes == K
        assert m.blob.size == _native.lib().lm_weight_blob_floats(K)
        live = sum(int(np.prod(s)) for k, s, kind in synth.schema(K) if kind in ("conv_w", "conv_b", "bn_w", "bn_b", "bn_mean", "bn_var"))
        assert m.blob.size == live
    bad = dict(sd)
    del bad["up_path.2.up.1.bias"]
    with pytest.raises(KeyError):
        NativeModel(bad)


def test_no_silent_cpu_fallback():
    from lungmask_b200 import LMInferer, _native
    with pytest.raises(AssertionError):
        LMInferer(modelname="NotAModel")
    with pytest.raises(AssertionError):
        LMInferer(modelname="R231", fillmodel="nope")
    if not torch.cuda.is_available():
        with pytest.raises(_native.NativeError):
            _native.Engine(0, 2)


def test_volume_dtype_rules():
    from lungmask_b200.mask import _to_engine_volume, _to_int16_volume
    v = np.array([[[-3000, 0, 70000]]], dtype=np.int32)
    assert _to_int16_volume(v).tolist() == [[[-1024, 0, 600]]]
    assert _to_engine_volume(v).dtype == np.int16
    for dt in (np.float32, np.float64):          # float volumes keep their dtype (the reference computes in it)
        assert _to_engine_volume(v.astype(dt)).dtype == dt
    assert _to_engine_volume(v.astype(np.float16)).dtype == np.float32
    with pytest.raises(TypeError):
        _to_int16_volume(v.astype(np.float64))
    with pytest.raises(ValueError):
        _to_engine_volume(np.zeros((4, 4), np.int16))


def test_normalisation_in_fp32_is_exact():
    """mask.py:168 divides in float64 and casts to fp32 (mask.py:178-182); the stem kernels divide the two exactly
    representable integers in fp32 (IEEE, round to nearest): the same bits for EVERY int16 input, not only [-1024, 600]."""
    hu = np.minimum(np.arange(-32768, 32768, dtype=np.int64), 600)
    i = hu + 1024
    assert np.array_equal((i.astype(np.float64) / 1624.0).astype(np.float32), i.astype(np.float32) / np.float32(1624.0))


def test_native_binding_refuses_lossy_conversions():
    from lungmask_b200._native import _as
    assert _as(np.array([[1, 2]], dtype=np.int64), np.int32).dtype == np.int32        # fits: converted
    assert _as(np.array([True, False]), np.uint8).tolist() == [1, 0]
    with pytest.raises(TypeError):
        _as(np.array([40000], dtype=np.int32), np.int16)                                # would wrap
    with pytest.raises(TypeError):
        _as(np.array([1.5], dtype=np.float32), np.int16)                                # would truncate
    with pytest.raises(ValueError):
        _as(np.zeros((2, 2), np.int16), np.int16, 3)


def test_cli_flags_match_reference():
    from lungmask_b200.__main__ import build_parser
    p = build_parser()
    a = p.parse_args([__file__, "out.nii", "--modelname", "LTRCLobes_R231", "--nopostprocess", "--batchsize", "7", "--noprogress", "--cpu", "--removemetadata"])
    assert a.modelname == "LTRCLobes_R231" and a.nopostprocess and a.batchsize == 7 and a.noprogress and a.cpu
    with pytest.raises(SystemExit):
        p.parse_args(["/definitely/not/here", "out"])


def test_shard_ranges_cover_and_do_not_overlap():
    from lungmask_b200.parallel import shard_range
    for S in (1, 5, 300, 512):
        for world in (1, 2, 3, 8):
            rs = [shard_range(S, r, world) for r in range(world)]
            assert rs[0][0] == 0 and rs[-1][1] == S
            assert all(a[1] == b[0] for a, b in zip(rs, rs[1:]))


def _gloo_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from lungmask_b200.parallel import apply_sharded
    from oracle import restate, synth
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sd = synth.random_state_dict(3, seed=3, calibrate_on=np.full((1, 256, 256), 0.4, np.float32))

    class OracleEngine:  # same stage methods as lungmask_b200._native.Engine, computed by the CPU oracle
        def preprocess(self, vol):
            r, b = restate.preprocess(vol, resolution=[256, 256])
            return r, np.asarray(b, dtype=np.int32).reshape(-1, 4)

        def forward(self, slot, resized):
            return restate.forward_volume(restate.normalise(resized), sd, batch_size=2)

        def postprocess(self, labels):
            return restate.postprocessing(labels)

        def reshape_masks(self, masks, boxes, H, W):
            return np.asarray([restate.reshape_mask(masks[i], boxes[i], (H, W)) for i in range(len(masks))], dtype=np.uint8)

    vol = synth.phantom(3, 96, 112, seed=11)
    out = apply_sharded(OracleEngine(), 0, vol, rank, world)
    want = restate.inference(vol, sd, batch_size=2)
    q.put((rank, bool(np.array_equal(out, want))))
    dist.destroy_process_group()


def test_two_rank_gloo_matches_single_rank():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]


def _connect_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from lungmask_b200.parallel import connect
    dist.init_process_group("gloo", rank=rank, world_size=world)

    class FakeEngine:  # records the collective protocol of lungmask_b200.parallel.connect
        def shard_init(self, r, w, n):
            self.init = (r, w, n)

        def shard_export(self):
            return bytes([rank]) * 64

        def shard_connect(self, handles):
            self.handles = handles

    e = connect(FakeEngine(), rank, world, 300)
    ok = e.init == (rank, world, 300) and e.handles == [bytes([r]) * 64 for r in range(world)]
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_shard_connect_exchanges_handles_in_rank_order():
    """world_size-2 gloo run of the handle exchange behind the engine's device-side gather (csrc/shard.cu)."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + os.getpid() % 2000
    procs = [ctx.Process(target=_connect_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]


def test_lungmask_alias_package_resolves_to_engine_mirror():
    import importlib
    for k in [k for k in sys.modules if k == "lungmask" or k.startswith("lungmask.")]:
        del sys.modules[k]
    lm = importlib.import_module("lungmask")
    import lungmask_b200
    assert lm.LMInferer is lungmask_b200.LMInferer
    from lungmask.mask import MODEL_URLS, get_model  # noqa: F401
    from lungmask.utils import bbox_3D, postprocessing, preprocess  # noqa: F401
    assert set(MODEL_URLS) == {"R231", "LTRCLobes", "R231CovidWeb"} and MODEL_URLS["LTRCLobes"][1] == 6
    m = np.zeros((10, 10, 10), dtype=np.uint8)
    m[2:8, 3:7, 4:6] = 1
    assert tuple(bbox_3D(m, margin=2)) == (0, 10, 1, 9, 2, 8)


def test_upsample_cell_corners_are_the_rows_the_formula_names():
    """forward_misc.cu upsample2x_kernel indexes the four loaded corners statically.  That is exact iff, for every
    output row y of a 2x bilinear upsample (align_corners=False, PyTorch's formula), the pair (i0, i1) the formula names
    equals the pair (ya, yb) the cell containing y loads - frame cells included (the same holds per column)."""
    f32 = np.float32
    for h in range(1, 40):
        for y in range(2 * h):
            s = max(f32(0.5) * (f32(y) + f32(0.5)) - f32(0.5), f32(0.0))        # up_axis()
            i0 = int(s)
            i1 = i0 + (1 if i0 < h - 1 else 0)
            ci = -1 if y == 0 else (y - 1) // 2                                   # the cell rows are 2 ci + 1 and 2 ci + 2
            assert y - (2 * ci + 1) in (0, 1) and -1 <= ci <= h - 1
            ya = 0 if ci < 0 else ci
            yb = ya + 1 if ya + 1 < h else h - 1
            assert (i0, i1) == (ya, yb), (h, y)
