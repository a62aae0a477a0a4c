"""GPU parity of the U-Net forward and of the whole path (C ABI) against the CPU oracle."""
import numpy as np
import pytest

from oracle import restate, synth
from _parity import explain_fused, explain_inference, fmt

pytestmark = pytest.mark.gpu

TOL_SCORES = 1e-4   # north_star: pre-argmax float scores within 1e-4 (absolute)


def _blob(sd):
    from lungmask_b200.mask import NativeModel
    return NativeModel(sd)


@pytest.fixture(scope="module")
def models():
    # head gain 0.3 keeps the scores in about [-10, 0] like a trained net (SURVEY App. A); the 1e-4 bound is absolute
    return {K: synth.random_state_dict(K, seed=10 + K, head_gain=0.3) for K in (3, 6)}


@pytest.mark.parametrize("K", [3, 6])
def test_forward_scores_and_labels(engine, models, K):
    sd = models[K]
    m = _blob(sd)
    engine.load_weights(0, m.blob, m.n_classes)
    vol = synth.phantom(5, seed=21)
    resized, _ = restate.preprocess(vol, resolution=[256, 256])
    want_labels, want_scores = restate.forward_volume(restate.normalise(resized), sd, batch_size=2, return_scores=True)
    labels, scores = engine.forward(0, resized, return_scores=True)
    err = np.abs(scores - want_scores)
    print("K=%d max|dscore|=%.3e mean=%.3e score range [%.2f, %.2f]" % (K, err.max(), err.mean(), want_scores.min(), want_scores.max()))
    assert err.max() <= TOL_SCORES
    # labels: identical wherever the oracle's top-2 margin exceeds the tolerance (near-ties are undecidable in fp32)
    top2 = np.sort(want_scores, axis=1)[:, -2:]
    margin = top2[:, 1] - top2[:, 0]
    diff = labels != want_labels
    print("label flips: %d of %d; pixels with margin<2e-4: %d" % (diff.sum(), diff.size, (margin < 2 * TOL_SCORES).sum()))
    assert not np.any(diff & (margin > 2 * TOL_SCORES))
    assert diff.sum() <= (margin <= 2 * TOL_SCORES).sum()


def test_forward_batch_invariance(engine, models):
    m = _blob(models[3])
    engine.load_weights(0, m.blob, m.n_classes)
    vol = synth.phantom(7, seed=4)   # 7 slices over a capacity-4 engine: waves of 4 + 3
    resized, _ = restate.preprocess(vol, resolution=[256, 256])
    a = engine.forward(0, resized)
    b = np.concatenate([engine.forward(0, resized[i:i + 1]) for i in range(7)])
    assert np.array_equal(a, b)


def test_apply_volume_end_to_end(engine, models):
    """lm_apply_volume against restate.inference with the every-voxel-explained protocol of tests/_parity.py
    (north_star: labels bit-exact, scores within 1e-4)."""
    sd = models[3]
    m = _blob(sd)
    engine.load_weights(0, m.blob, m.n_classes)
    vol = synth.phantom(6, 300, 414, seed=8)
    rep = explain_inference(engine, 0, vol, sd, batch=3)
    print("end to end: " + fmt(rep))
    t = engine.last_timings()
    assert t["kernel_launches"] > 30
    rep = explain_inference(engine, 0, vol, sd, batch=3, postprocess=False)   # LMInferer(volume_postprocessing=False)
    print("end to end, no post-processing: " + fmt(rep))


@pytest.mark.parametrize("postprocess", [True, False])
def test_apply_fused(engine, models, postprocess):
    """LMInferer.apply with a fill model (mask.py:223-232): both inner inferences explained, the fusion glue
    (lm_fuse) and the original-resolution post-processing bit-exact in isolation, the fused volume explained by the
    inner results.  volume_postprocessing=False reaches the inner inferences only (mask.py:191-194)."""
    m6, m3 = _blob(models[6]), _blob(models[3])
    engine.load_weights(0, m6.blob, m6.n_classes)
    engine.load_weights(1, m3.blob, m3.n_classes)
    vol = synth.phantom(4, 200, 216, seed=9)
    rep = explain_fused(engine, 0, 1, vol, models[6], models[3], batch=2, postprocess=postprocess)
    print("fused (volume_postprocessing=%s): %s" % (postprocess, fmt(rep)))


def test_fuse_kernel_edge_cases(engine):
    """lm_fuse alone (mask.py:228-230) on crafted inputs: the spare value is uint8 arithmetic (255 + 1 wraps to 0)."""
    rng = np.random.default_rng(11)
    for top in (5, 254, 255):
        res_l = rng.integers(0, 3, size=(3, 40, 56)).astype(np.uint8)
        res_l[res_l == 2] = top
        res_r = rng.integers(0, 3, size=res_l.shape).astype(np.uint8)
        want, spare = restate.fuse_pre(res_l, res_r)
        got, gspare = engine.fuse(res_l, res_r)
        assert gspare == int(spare) and np.array_equal(got, want), top


def test_lminferer_fused_honours_volume_postprocessing(tmp_path, models):
    """ADVICE r1: LMInferer(fillmodel=..., volume_postprocessing=False) must differ from the default exactly as the
    reference does (inner post-processing skipped, fusion post-processing kept)."""
    import torch
    from lungmask_b200 import LMInferer
    p6, p3 = str(tmp_path / "l.pth"), str(tmp_path / "r.pth")
    torch.save(models[6], p6)
    torch.save(models[3], p3)
    vol = synth.phantom(4, 200, 216, seed=9)
    outs = {}
    for vp in (True, False):
        inf = LMInferer(modelname="LTRCLobes", modelpath=p6, fillmodel="R231", fillmodel_path=p3, batch_size=4,
                        volume_postprocessing=vp, tqdm_disable=True)
        outs[vp] = inf.apply(vol)
        assert np.array_equal(outs[vp], inf.engine.apply_fused(0, 1, vol, postprocess=vp))
        inf.engine.close()
    assert not np.array_equal(outs[True], outs[False])


def test_lminferer_surface(tmp_path, models):
    """LMInferer keeps the reference's constructor / apply contract (mask.py:72-139,212-232)."""
    import torch
    from lungmask_b200 import LMInferer
    p = str(tmp_path / "synthetic_r231.pth")
    torch.save(models[3], p)
    with pytest.raises(AssertionError):
        LMInferer(modelname="nope", modelpath=p)
    with pytest.raises(RuntimeError):
        LMInferer(modelpath=p, force_cpu=True)
    inf = LMInferer(modelname="LTRCLobes", modelpath=p, batch_size=4, tqdm_disable=True)  # class count comes from the file
    assert inf.modelname == "synthetic_r231.pth" and inf.model.n_classes == 3
    vol = synth.phantom(3, seed=2)
    before = vol.copy()
    out = inf.apply(vol)
    assert out.dtype == np.uint8 and out.shape == vol.shape and np.array_equal(vol, before)
    assert out.max() <= 2
    out32 = inf.apply(vol.astype(np.int32))
    assert np.array_equal(out, out32)
    # float volumes: integral values give the integer result only up to the missing rounding of the resampled slices
    outf = inf.apply(vol.astype(np.float32))
    assert outf.shape == vol.shape and outf.dtype == np.uint8 and (outf != out).mean() < 0.01


def test_activation_taps(engine, models):
    """Layer-by-layer parity: every block output of the engine against the oracle's (relative to the
    tensor's own scale), which localises a wiring bug to one layer and documents where error accumulates."""
    import torch
    sd = models[3]
    m = _blob(sd)
    engine.load_weights(0, m.blob, m.n_classes)
    vol = synth.phantom(2, seed=33)
    resized, _ = restate.preprocess(vol, resolution=[256, 256])
    taps = {}
    with torch.inference_mode():
        restate.unet_forward(torch.as_tensor(restate.normalise(resized)[:, None], dtype=torch.float32), sd, taps=taps)
    engine.forward(0, resized)
    ids = {"S0": 1, "P0": 2, "S1": 4, "P1": 5, "S2": 7, "P2": 8, "S3": 10, "P3": 11, "B4": 13, "U0": 15, "E0": 17,
           "U1": 19, "E1": 21, "U2": 23, "E2": 25, "U3": 27}
    worst = 0.0
    for name, aid in ids.items():
        got = engine.read_activation(aid, 2)
        want = taps[name].permute(0, 2, 3, 1).numpy()
        rel = float(np.abs(got - want).max() / (np.abs(want).max() + 1e-12))
        print("%-3s max|d|/max|x| = %.3e" % (name, rel))
        worst = max(worst, rel)
    assert worst < 2e-5


def test_default_wave_matches_small_waves(engine, models, tmp_path):
    """LMInferer's default 37-slice forward wave (one full wave + a 2-slice tail) gives bit-identical labels to
    the capacity-4 engine: the engine is batch-invariant, so the reference's batch_size only bounds memory."""
    import torch
    from lungmask_b200 import LMInferer
    p = str(tmp_path / "w3.pth")
    torch.save(models[3], p)
    inf = LMInferer(modelpath=p, tqdm_disable=True)
    assert inf.wave_slices == 37 and inf.batch_size == 20
    vol = synth.phantom(39, seed=77)
    m = _blob(models[3])
    engine.load_weights(0, m.blob, m.n_classes)
    assert np.array_equal(inf.apply(vol), engine.apply_volume(0, vol))


def test_sharded_path_equals_whole_volume(engine, models):
    """lungmask_b200.parallel.apply_sharded (stage-level C-ABI calls + gather) on one rank == lm_apply_volume."""
    from lungmask_b200.parallel import apply_sharded
    m = _blob(models[3])
    engine.load_weights(0, m.blob, m.n_classes)
    vol = synth.phantom(5, 180, 200, seed=12)
    assert np.array_equal(apply_sharded(engine, 0, vol, 0, 1), engine.apply_volume(0, vol))


@pytest.mark.parametrize("code", ["RAS", "PLI", "SAL"])
def test_orientation_on_device(engine, models, code, tmp_path):
    """f2: lm_apply_volume_oriented == re-orient with numpy, run the LPS path, orient back (mask.py:157-164,204-208),
    single model and fusion (whose post-processing runs in the NATIVE orientation, mask.py:225-232)."""
    from lungmask_b200 import orient
    m6, m3 = _blob(models[6]), _blob(models[3])
    engine.load_weights(0, m6.blob, m6.n_classes)
    engine.load_weights(1, m3.blob, m3.n_classes)
    lps = synth.phantom(5, 120, 136, seed=17)
    native = orient.from_lps(lps, code)
    perm, flip = orient.array_transform_to_lps(code)
    assert np.array_equal(orient.to_lps(native, code), lps)
    got = engine.apply_volume_oriented(1, native, perm, flip)
    assert got.shape == native.shape
    assert np.array_equal(got, orient.from_lps(engine.apply_volume(1, lps), code))
    res_l = orient.from_lps(engine.apply_volume(0, lps), code)
    res_r = orient.from_lps(engine.apply_volume(1, lps), code)
    pre, spare = engine.fuse(res_l, res_r)
    want_fused = engine.postprocess(pre, spare=[spare])             # native-orientation fusion, stage by stage
    assert np.array_equal(engine.apply_volume_oriented(0, native, perm, flip, slot_fill=1), want_fused)
    assert np.array_equal(want_fused, restate.fuse(res_l, res_r))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_float_volumes(engine, models, dtype):
    """ADVICE r1: the reference accepts float volumes and keeps their dtype through utils.preprocess (no rounding of the
    resampled slices) and the normalisation of mask.py:167-168.  Pre-processing + normalisation bit-exact, end to end
    explained like the integer path."""
    sd = models[3]
    m = _blob(sd)
    engine.load_weights(0, m.blob, m.n_classes)
    rng = np.random.default_rng(3)
    vol = (synth.phantom(4, 200, 216, seed=19).astype(np.float64) + rng.uniform(-0.4, 0.4, size=(4, 200, 216))).astype(dtype)
    tv, boxes = restate.preprocess(vol, resolution=[256, 256])
    assert tv.dtype == dtype
    want_norm = restate.normalise(tv).astype(np.float32)        # the cast of mask.py:178-182
    norm, gboxes = engine.preprocess_float(vol)
    assert np.array_equal(gboxes.astype(np.int64), np.asarray(boxes, dtype=np.int64).reshape(-1, 4))
    assert np.array_equal(norm, want_norm)
    want = restate.inference(vol, sd, batch_size=2)
    got = engine.apply_volume_float(0, vol)
    d = int((got != want).sum())
    print("%s volume: voxels differing %d of %d" % (np.dtype(dtype).name, d, want.size))
    # explained: the oracle's integer stages on the engine's own labels reproduce the engine's output
    labels = engine.apply_volume_float(0, vol, postprocess=False)
    raw = restate.inference(vol, sd, batch_size=2, volume_postprocessing=False)
    assert (labels != raw).mean() < 2e-3 and d <= 5e-3 * want.size


def test_graph_replay_matches_plain_launches(models):
    """A volume's forward is captured once as a CUDA graph and replayed; results must equal launching every kernel
    (lm_set_option("graphs", 0)), also after the configuration changes (new weights -> new capture)."""
    from lungmask_b200 import _native
    eng = _native.Engine(device=0, batch_capacity=3)
    try:
        vol = synth.phantom(7, 150, 170, seed=23)      # 3 + 3 + 1 slices
        for K in (3, 6):
            m = _blob(models[K])
            eng.load_weights(0, m.blob, m.n_classes)
            eng.set_option("graphs", 0)
            plain = eng.apply_volume(0, vol)
            eng.set_option("graphs", 1)
            first = eng.apply_volume(0, vol)           # captures
            again = eng.apply_volume(0, vol)           # replays
            assert np.array_equal(plain, first) and np.array_equal(plain, again)
    finally:
        eng.close()


@pytest.mark.parametrize("key", ["stem_v2", "upsample_v2", "cta_pairs", "weight_mcast", "dual_issue", "bn64_mask"])
def test_removed_kernel_options_are_unknown_keys(engine, key):
    """The forward has one stem, one upsample and one convolution kernel: the options that once selected alternatives are
    rejected like any other unknown key instead of being accepted and ignored."""
    from lungmask_b200 import _native
    with pytest.raises(_native.NativeError, match="unknown key " + key):
        engine.set_option(key, 0)
