"""Generates tests/golden/* from the UNMODIFIED reference (imported from /root/reference through
oracle.ref_loader).  Run in the build container only:  python -m oracle.make_golden

Fixtures (small, committed):
  ct_slice_512.npz   pixel data of the reference's tests/testdata/0.dcm (int16 512x512), the only real CT
                     slice available offline (SURVEY.md section 4)
  preprocess.json    utils.preprocess(resolution=[256,256]) on seeded inputs: boxes + CRC32 of every slice
  postprocess.npz    utils.postprocessing on seeded label volumes (inputs + outputs, several spare lists)
  forward.npz        resunet.UNet (get_model configuration) scores on one phantom slice, sub-sampled,
                     for seeded synthetic state_dicts (K = 3 and 6)
  e2e.json           LMInferer(force_cpu=True).apply label histograms for seeded weights / volumes
  fusion.npz         LMInferer(modelname K=6, fillmodel K=3, force_cpu=True): the two inner _inference results
                     (res_l, res_r) and apply() for volume_postprocessing True / False (mask.py:223-232), plus
                     the single-model apply() volumes behind e2e.json's histograms
  reference.json     what tests/test_oracle_reference.py compares oracle.restate with: the UNet state_dict layout,
                     and digests of utils.preprocess / utils.postprocessing outputs and of the UNet scores on
                     the inputs below
  reference_forward.npz  LMInferer(force_cpu=True).apply labels and a sub-sample of the UNet scores for that test
"""
import contextlib
import hashlib
import json
import os
import tempfile
import zlib

import numpy as np
import torch

from . import ref_loader, restate, synth

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

PRE_CASES = [("ct", None, None), ("phantom", (4, 256, 256), 0), ("phantom", (3, 300, 414), 1), ("phantom", (2, 97, 200), 2),
             ("phantom", (2, 512, 512), 3), ("phantom", (2, 64, 64), 4), ("phantom", (2, 14, 27), 6)]
POST_CASES = [(12, 3, 0, 2e-3), (9, 6, 1, 2e-3), (1, 3, 2, 2e-3), (2, 6, 3, 1e-3)]
# inputs of tests/test_oracle_reference.py (reference.json, reference_forward.npz)
REF_PRE_CASES = [((3, 256, 256), 0), ((2, 300, 414), 1), ((2, 97, 200), 2), ((2, 40, 52), 3)]
REF_POST_CASES = [(8, 3, 0), (5, 6, 1), (1, 3, 2)]
REF_FORWARD = dict(K=3, weights_seed=13, volume=(3, 200, 216), volume_seed=5, batch_size=2)


def pre_input(kind, shape, seed):
    if kind == "ct":
        ct = np.load(os.path.join(GOLD, "ct_slice_512.npz"))["slice"]
        return np.stack([ct, ct[::-1].copy(), np.roll(ct, 37, 1), ct.T.copy()])
    return synth.phantom(*shape, seed=seed)


def digest(a):
    """dtype, shape and SHA-256 of an array's bytes: equal digests <=> bit-identical arrays."""
    a = np.ascontiguousarray(a)
    return "%s%s:%s" % (a.dtype.str, list(a.shape), hashlib.sha256(a.tobytes()).hexdigest())


@contextlib.contextmanager
def single_thread():
    """torch's CPU convolutions sum in an order that depends on the thread count: bit-identical scores across
    machines need the same count, so the forward behind reference_forward.npz runs on one thread, here and in the test."""
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        yield
    finally:
        torch.set_num_threads(n)


def case_key(*args):
    return "/".join("x".join(map(str, a)) if isinstance(a, tuple) else str(a) for a in args)


def ragged_volumes():
    """slices smaller than the 128 x 128 thumbnail, non-square and odd sizes, volumes without a clear body"""
    shapes = [(2, 17, 23), (1, 128, 128), (2, 129, 127), (1, 64, 300), (2, 511, 513), (1, 33, 33), (2, 200, 100), (1, 12, 12),
              (2, 256, 255), (1, 150, 400)]
    vols = [synth.phantom(*sh, seed=50 + i) for i, sh in enumerate(shapes)]
    rng = np.random.default_rng(0)
    vols += [rng.normal(-400, 400, size=(2, 90 + 7 * i, 110 + 5 * i)).astype(np.int16) for i in range(6)]
    return vols


def postprocessing_sweep():
    """random sizes, class counts and speckle levels x the spare / skip_below combinations of utils.py:272;
    yields (seed, label volume, spare, skip_below)"""
    rng = np.random.default_rng(0)
    for seed in range(10, 22):
        S, K = int(rng.integers(1, 7)), int(rng.choice([3, 6]))
        lab = synth.label_noise_volume(S, K, seed=seed, speckle=float(rng.choice([5e-4, 2e-3, 1e-2])), H=int(rng.choice([48, 64, 96])),
                                       W=int(rng.choice([48, 80, 128])))
        for spare, skip in (([], 3), ([K - 1], 3), ([], 1), ([1], 2)):
            yield seed, lab, spare, skip


def write_reference_checks(ref):
    """reference.json and reference_forward.npz: the reference's own results on the inputs above."""
    pre = {}
    for shape, seed in REF_PRE_CASES:
        out, boxes = ref.utils.preprocess(synth.phantom(*shape, seed=seed), resolution=[256, 256])
        pre[case_key(shape, seed)] = {"digest": digest(out), "boxes": np.asarray(boxes).tolist()}
    ragged = []
    for vol in ragged_volumes():
        out, boxes = ref.utils.preprocess(vol, resolution=[256, 256])
        ragged.append({"shape": list(vol.shape), "digest": digest(out), "boxes": np.asarray(boxes).tolist()})
    post = {}
    for S, K, seed in REF_POST_CASES:
        lab = synth.label_noise_volume(S, K, seed=seed, speckle=2e-3)
        post[case_key(S, K, seed)] = {"plain": digest(ref.utils.postprocessing(lab, disable_tqdm=True)),
                                      "spare": digest(ref.utils.postprocessing(lab, spare=[K - 1], disable_tqdm=True))}
    sweep = []
    for seed, lab, spare, skip in postprocessing_sweep():
        out = ref.utils.postprocessing(lab.copy(), spare=list(spare), disable_tqdm=True, skip_below=skip)
        sweep.append({"seed": seed, "spare": list(spare), "skip_below": skip, "digest": digest(out)})
    schema = {}
    for K in (3, 6):
        m = ref.resunet.UNet(n_classes=K, padding=True, depth=5, up_mode="upsample", batch_norm=True, residual=False)
        schema[str(K)] = [[k, list(v.shape)] for k, v in m.state_dict().items()]

    f = REF_FORWARD
    vol = synth.phantom(*f["volume"], seed=f["volume_seed"])
    with single_thread():
        sd = synth.random_state_dict(f["K"], seed=f["weights_seed"])   # BN calibration is a torch forward too
        p = os.path.join(tempfile.gettempdir(), "golden_reference_forward.pth")
        torch.save(sd, p)
        inf = ref.mask.LMInferer(modelname="R231", modelpath=p, force_cpu=True, batch_size=f["batch_size"], tqdm_disable=True)
        labels = inf.apply(vol)
        resized, _ = ref.utils.preprocess(vol, resolution=[256, 256])
        x = torch.as_tensor(restate.normalise(resized)[:, None], dtype=torch.float32)
        with torch.inference_mode():
            scores = inf.model(x).numpy()
    json.dump({"preprocess": pre, "preprocess_ragged": ragged, "postprocess": post, "postprocess_sweep": sweep,
               "state_dict_layout": schema, "forward_scores": digest(scores)},
              open(os.path.join(GOLD, "reference.json"), "w"), indent=1)
    np.savez_compressed(os.path.join(GOLD, "reference_forward.npz"), apply=labels, scores_sample=scores[:, :, 3::8, 5::8].copy())


def main():
    ref = ref_loader.load()
    os.makedirs(GOLD, exist_ok=True)
    b = open(os.path.join(ref_loader.REFERENCE_ROOT, "tests", "testdata", "0.dcm"), "rb").read()
    np.savez_compressed(os.path.join(GOLD, "ct_slice_512.npz"), slice=np.frombuffer(b[-524288:], "<i2").reshape(512, 512))

    pre = []
    for kind, shape, seed in PRE_CASES:
        vol = pre_input(kind, shape, seed)
        out, boxes = ref.utils.preprocess(vol, resolution=[256, 256])
        pre.append({"kind": kind, "shape": shape, "seed": seed, "boxes": np.asarray(boxes).astype(int).tolist(),
                    "crc32": [int(zlib.crc32(np.ascontiguousarray(s).tobytes())) for s in out], "dtype": str(out.dtype)})
    json.dump(pre, open(os.path.join(GOLD, "preprocess.json"), "w"), indent=1)

    post = {}
    for i, (S, K, seed, sp) in enumerate(POST_CASES):
        lab = synth.label_noise_volume(S, K, seed=seed, speckle=sp)
        post[f"in{i}"] = lab
        post[f"out{i}_plain"] = ref.utils.postprocessing(lab, disable_tqdm=True)
        post[f"out{i}_spare"] = ref.utils.postprocessing(lab, spare=[K - 1], disable_tqdm=True)
        post[f"out{i}_skip1"] = ref.utils.postprocessing(lab, skip_below=1, disable_tqdm=True)
    np.savez_compressed(os.path.join(GOLD, "postprocess.npz"), **post)

    fwd, e2e, fus, paths = {}, [], {}, {}
    for K in (3, 6):
        sd = synth.random_state_dict(K, seed=10 + K)
        model = ref.resunet.UNet(n_classes=K, padding=True, depth=5, up_mode="upsample", batch_norm=True, residual=False)
        model.load_state_dict(sd)
        model.eval()
        vol = synth.phantom(2, seed=21)
        tv, _ = ref.utils.preprocess(vol, resolution=[256, 256])
        x = torch.as_tensor(np.divide(tv + 1024, 1624)[:, None], dtype=torch.float32)
        with torch.inference_mode():
            y = model(x).numpy()
        fwd[f"scores_K{K}"] = y[:, :, 3::8, 5::8].copy()
        p = os.path.join(tempfile.gettempdir(), f"golden_K{K}.pth")
        torch.save(sd, p)
        paths[K] = p
        inf = ref.mask.LMInferer(modelname="R231", modelpath=p, force_cpu=True, batch_size=2, tqdm_disable=True)
        v2 = synth.phantom(4, 200, 216, seed=30 + K)
        out = inf.apply(v2)
        fus[f"apply_K{K}"] = out
        e2e.append({"K": K, "weights_seed": 10 + K, "volume": [4, 200, 216], "volume_seed": 30 + K,
                    "histogram": np.bincount(out.ravel(), minlength=K).tolist()})
    # fusion (mask.py:223-232): base = the K=6 weights, fill = the K=3 weights, on the K=6 e2e volume
    vf = synth.phantom(4, 200, 216, seed=36)
    for vp in (True, False):
        inf = ref.mask.LMInferer(modelname="LTRCLobes", modelpath=paths[6], fillmodel="R231", fillmodel_path=paths[3],
                                 force_cpu=True, batch_size=2, volume_postprocessing=vp, tqdm_disable=True)
        tag = "pp" if vp else "nopp"
        fus[f"res_l_{tag}"] = inf._inference(vf, inf.model)
        fus[f"res_r_{tag}"] = inf._inference(vf, inf.fillmodelm)
        fus[f"fused_{tag}"] = inf.apply(vf)
    np.savez_compressed(os.path.join(GOLD, "fusion.npz"), **fus)
    np.savez_compressed(os.path.join(GOLD, "forward.npz"), **fwd)
    json.dump(e2e, open(os.path.join(GOLD, "e2e.json"), "w"), indent=1)
    write_reference_checks(ref)
    print("golden fixtures written to", GOLD)


if __name__ == "__main__":
    main()
