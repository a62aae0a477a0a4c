"""Validates the oracle against the reference ITSELF: tests/golden/reference.json and reference_forward.npz hold what
the unmodified reference (imported with the stand-ins of oracle/standins.py) computed on the inputs below, written by
oracle/make_golden.py.  Runs anywhere (no GPU, no reference tree)."""
import json
import os

import numpy as np
import pytest

from oracle import make_golden, restate, synth

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ref():
    return json.load(open(os.path.join(GOLD, "reference.json")))


def test_reference_known_answer_tests_through_standins():
    """tests/test_utils.py:58-63,73-107,124-159 of the reference, verbatim assertions, on the restatement and the
    stand-ins it calls."""
    m = np.zeros((10, 10, 10), dtype=np.uint8)
    m[2:8, 3:7, 4:6] = 1
    assert tuple(restate.bbox_3D(m, margin=2)) == (0, 10, 1, 9, 2, 8)
    img = np.full((10, 10), dtype=np.int16, fill_value=-1000)
    img[2:8, 3:7] = 1
    img[9, 9] = 1
    assert np.sum(restate.simple_bodymask(img)) == 24
    cropped, bb = restate.crop_and_resize(img, width=20, height=20)
    assert tuple(bb) == (2, 3, 8, 7) and cropped.shape == (20, 20) and np.sum(cropped) == 400
    out = restate.reshape_mask(np.full((10, 10), dtype=np.uint8, fill_value=1), (2, 2, 22, 22), origsize=(30, 30))
    assert out.shape == (30, 30) and np.sum(out) == 400
    li = np.zeros((1, 6, 6), dtype=np.uint8)
    li[0] = np.asarray([[0, 0, 0, 0, 0, 0], [0, 1, 1, 2, 2, 0], [0, 2, 0, 3, 1, 0], [0, 4, 4, 4, 0, 0], [0, 4, 0, 4, 0, 0], [0, 4, 4, 4, 0, 0]])
    gt = [[0, 0, 0, 0, 0, 0], [0, 1, 1, 2, 2, 0], [0, 1, 0, 3, 2, 0], [0, 4, 4, 4, 0, 0], [0, 4, 0, 4, 0, 0], [0, 4, 4, 4, 0, 0]]
    vol = np.tile(li, (2, 1, 1))
    assert np.all(restate.postprocessing(vol, spare=[], skip_below=1)[0] == gt)
    assert restate.postprocessing(vol, spare=[3], skip_below=1)[0][2, 3] == 2
    assert restate.postprocessing(vol, spare=[3], skip_below=3)[0][2, 1] == 0


def test_state_dict_schema_is_the_reference_layout(ref):
    for K in (3, 6):
        rsd = ref["state_dict_layout"][str(K)]
        sch = synth.schema(K)
        assert [k for k, _, _ in sch] == [k for k, _ in rsd]
        assert all(tuple(s) == tuple(r) for (_, s, _), (_, r) in zip(sch, rsd))
        assert len(sch) == 227


@pytest.mark.parametrize("shape,seed", make_golden.REF_PRE_CASES)
def test_preprocess_equals_reference(ref, shape, seed):
    want = ref["preprocess"][make_golden.case_key(shape, seed)]
    r, br = restate.preprocess(synth.phantom(*shape, seed=seed), resolution=[256, 256])
    assert make_golden.digest(r) == want["digest"] and np.array_equal(np.asarray(br), np.asarray(want["boxes"]))


@pytest.mark.parametrize("S,K,seed", make_golden.REF_POST_CASES)
def test_postprocessing_equals_reference(ref, S, K, seed):
    want = ref["postprocess"][make_golden.case_key(S, K, seed)]
    lab = synth.label_noise_volume(S, K, seed=seed, speckle=2e-3)
    assert make_golden.digest(restate.postprocessing(lab)) == want["plain"]
    assert make_golden.digest(restate.postprocessing(lab, spare=[K - 1])) == want["spare"]


def test_forward_and_apply_equal_reference(ref):
    f = make_golden.REF_FORWARD
    g = np.load(os.path.join(GOLD, "reference_forward.npz"))
    vol = synth.phantom(*f["volume"], seed=f["volume_seed"])
    taps = {}
    with make_golden.single_thread():
        sd = synth.random_state_dict(f["K"], seed=f["weights_seed"])
        labels = restate.inference(vol, sd, batch_size=f["batch_size"], taps=taps)
    assert np.array_equal(labels, g["apply"])
    assert np.array_equal(taps["scores"][:, :, 3::8, 5::8], g["scores_sample"])
    assert make_golden.digest(taps["scores"]) == ref["forward_scores"]


def test_preprocess_equals_reference_on_ragged_and_noisy_volumes(ref):
    """slices smaller than the 128 x 128 thumbnail, non-square and odd sizes, volumes without a clear body"""
    vols = make_golden.ragged_volumes()
    assert len(vols) == len(ref["preprocess_ragged"])
    for vol, want in zip(vols, ref["preprocess_ragged"]):
        assert list(vol.shape) == want["shape"]
        r, br = restate.preprocess(vol, resolution=[256, 256])
        assert make_golden.digest(r) == want["digest"] and np.array_equal(np.asarray(br), np.asarray(want["boxes"])), vol.shape


def test_postprocessing_equals_reference_sweep(ref):
    """random sizes, class counts and speckle levels x the spare / skip_below combinations of utils.py:272"""
    cases = list(make_golden.postprocessing_sweep())
    assert len(cases) == len(ref["postprocess_sweep"])
    for (seed, lab, spare, skip), want in zip(cases, ref["postprocess_sweep"]):
        assert (seed, list(spare), skip) == (want["seed"], want["spare"], want["skip_below"])
        out = restate.postprocessing(lab.copy(), spare=list(spare), skip_below=skip)
        assert make_golden.digest(out) == want["digest"], (seed, lab.shape, spare, skip)
