#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the UNMODIFIED reference (oracle/_ref, built by
oracle/build_ref.sh from /root/reference) on small seeded inputs.

Run from the repo root in the build container (where /root/reference exists):

    bash oracle/build_ref.sh && python tests/golden/make_golden.py

The fixtures pin the oracle (tests/test_oracle.py) and the CUDA path (tests/test_gpu_*.py); they
travel to the GPU box, /root/reference does not.  Inputs are stored next to outputs so a drift in
the synthetic generator cannot silently move the goal posts.
"""
import gzip
import math
import os
import struct
import sys

import numpy as np
from numpy.random import RandomState
from scipy.stats.mstats import zscore
from sklearn import svm
from sklearn.linear_model import LogisticRegression

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import reference  # noqa: E402
from brainiak_b200.fcma import synthetic  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
REF_TESTS = "/root/reference/tests"


def ref_create_epoch(prng, row=12, col=5):
    # same construction as reference tests/fcma/test_voxel_selection.py:27-36
    mat = prng.rand(row, col).astype(np.float32)
    mat = zscore(mat, axis=0, ddof=0)
    mat = np.nan_to_num(mat)
    mat = mat / math.sqrt(mat.shape[0])
    return mat


def svc():
    return svm.SVC(kernel="precomputed", shrinking=False, C=1, gamma="auto")


def stages_all(vs, V, unit):
    raws, norms, kerns = [], [], []
    for s in range(0, V, unit):
        n = min(unit, V - s)
        r, z, k = reference.voxel_block_stages(vs, (s, n))
        raws.append(r), norms.append(z), kerns.append(k)
    return np.concatenate(raws), np.concatenate(norms), np.concatenate(kerns)


def accs(results, n):
    out = np.zeros(n)
    for vid, a in results:
        out[vid] = a
    return out


def gen_vs_small(m):
    """The reference's own voxel-selection test inputs (test_voxel_selection.py:40-130)."""
    prng = RandomState(1234567890)
    raw = [ref_create_epoch(prng) for _ in range(8)]
    labels = [0, 1, 0, 1, 0, 1, 0, 1]
    vs = m.VoxelSelector(labels, 4, 2, raw, voxel_unit=1, process_num=0)
    fake_corr = prng.rand(1, 4, 5).astype(np.float32)
    scipy_norm = vs._correlation_normalization(fake_corr.copy())
    cpp_norm = fake_corr.copy()
    m.fcma_extension.normalization(cpp_norm, 4)
    r, z, k = stages_all(vs, 5, 1)
    acc_svm = accs(reference.run_voxel_selection(vs, svc()), 5)
    acc_lr = accs(reference.run_voxel_selection(vs, LogisticRegression()), 5)
    # two masks (test_voxel_selection.py:101-130)
    prng = RandomState(1234567890)
    raw1 = [ref_create_epoch(prng) for _ in range(8)]
    raw2 = [ref_create_epoch(prng) for _ in range(8)]
    vs2 = m.VoxelSelector(labels, 4, 2, raw1, raw_data2=raw2, voxel_unit=1, process_num=0)
    r2, z2, k2 = stages_all(vs2, 5, 1)
    acc2_svm = accs(reference.run_voxel_selection(vs2, svc()), 5)
    acc2_lr = accs(reference.run_voxel_selection(vs2, LogisticRegression()), 5)
    np.savez_compressed(
        os.path.join(OUT, "vs_small.npz"),
        raw=np.stack(raw), labels=np.array(labels), fake_corr=fake_corr,
        scipy_norm=scipy_norm, cpp_norm=cpp_norm,
        corr_raw=r, corr_norm=z, kernels=k, acc_svm=acc_svm, acc_lr=acc_lr,
        raw1=np.stack(raw1), raw2=np.stack(raw2), corr_raw2=r2, corr_norm2=z2, kernels2=k2,
        acc2_svm=acc2_svm, acc2_lr=acc2_lr)
    print("vs_small: svm", (8 * acc_svm).astype(int), "lr", (8 * acc_lr).astype(int),
          "| two masks svm", (8 * acc2_svm).astype(int), "lr", (8 * acc2_lr).astype(int))


def gen_vs_mid(m):
    """Mid-size seeded case: ragged task, eps that leaves trailing epochs, two masks."""
    V, T, E, eps = 160, 24, 10, 4        # E=10, eps=4 -> 2 subjects + 2 untouched trailing epochs
    raw, labels = synthetic.make_epochs(V, T, E, informative=16)
    vs = m.VoxelSelector(labels, eps, 2, raw, voxel_unit=37, process_num=0)
    task = (40, 37)
    r, z, k = reference.voxel_block_stages(vs, task)
    V1, V2 = 96, 136
    d1, d2, labels2 = synthetic.make_two_masks(V1, V2, 20, 8)
    vs2 = m.VoxelSelector(labels2, 4, 2, d1, raw_data2=d2, voxel_unit=29, process_num=0)
    task2 = (58, 29)
    r2, z2, k2 = reference.voxel_block_stages(vs2, task2)
    # full run on a case with planted signal: accuracies for every voxel
    Vf, Tf, Ef, epsf = 128, 40, 16, 4
    rawf, labelsf = synthetic.make_epochs(Vf, Tf, Ef, informative=12, signal=1.0)
    vsf = m.VoxelSelector(labelsf, epsf, 4, rawf, voxel_unit=32, process_num=0)
    accf = accs(reference.run_voxel_selection(vsf, svc()), Vf)
    _, _, kf = stages_all(vsf, Vf, 32)
    np.savez_compressed(
        os.path.join(OUT, "vs_mid.npz"),
        raw=np.stack(raw), labels=np.array(labels), eps=eps, task=np.array(task),
        corr_raw=r, corr_norm=z, kernels=k,
        d1=np.stack(d1), d2=np.stack(d2), labels2=np.array(labels2), task2=np.array(task2),
        corr_raw2=r2, corr_norm2=z2, kernels2=k2)
    # the full run in a file of its own: each fixture stays under 1 MB
    np.savez_compressed(
        os.path.join(OUT, "vs_mid_run.npz"),
        rawf=np.stack(rawf), labelsf=np.array(labelsf), epsf=epsf, accf=accf, kernelsf=kf)
    print("vs_mid: top voxels", np.argsort(-accf, kind="stable")[:12], "acc", np.sort(accf)[-12:])


def ref_clf_epoch(prng, idx, num_voxels):
    # reference tests/fcma/test_classification.py:28-40
    mat = prng.rand(12, num_voxels).astype(np.float32)
    if idx % 2 == 0:
        mat = np.sort(mat, axis=0)
    mat = zscore(mat, axis=0, ddof=0)
    mat = np.nan_to_num(mat)
    mat = mat / math.sqrt(mat.shape[0])
    return mat


def gen_clf(m):
    prng = RandomState(1234567890)
    d5 = [ref_clf_epoch(prng, i, 5) for i in range(20)]
    d6 = [ref_clf_epoch(prng, i, 6) for i in range(20)]
    labels = [0, 1] * 10
    out = dict(d5=np.stack(d5), d6=np.stack(d6), labels=np.array(labels))
    for tag, a, b in (("one", d5, d5), ("two", d5, d6)):
        # full-kernel fit (classifier.py:350-424), predict with recomputation
        clf = m.Classifier(svc(), epochs_per_subj=4)
        clf.fit(list(zip(a[:12], b[:12])), labels[:12])
        out[tag + "_train_features"] = clf.training_data_.copy()
        out[tag + "_num_digits"] = clf.num_digits_
        test = list(zip(a[12:], b[12:]))
        out[tag + "_decision"] = clf.decision_function(test)
        out[tag + "_predict"] = clf.predict(test)
        out[tag + "_test_sim"] = clf.test_data_.copy()
        # the kernel the fit used
        X1, X2 = (a[:12], b[:12]) if a[0].shape[1] >= b[0].shape[1] else (b[:12], a[:12])
        c2 = m.Classifier(svc(), epochs_per_subj=4)
        c2.num_voxels_ = X1[0].shape[1]
        c2.num_features_ = X1[0].shape[1] * X2[0].shape[1]
        c2.num_samples_ = 12
        K, _ = c2._compute_kernel_matrix_in_portion(X1, X2)
        out[tag + "_kernel12"] = K
        # portion mode (classifier.py:279-348) over all 20 samples
        clf = m.Classifier(svc(), num_processed_voxels=2, epochs_per_subj=4)
        clf.fit(list(zip(a, b)), labels, num_training_samples=12)
        out[tag + "_portion_decision"] = clf.decision_function()
        out[tag + "_portion_predict"] = clf.predict()
        out[tag + "_portion_test_sim"] = clf.test_data_.copy()
        out[tag + "_portion_num_digits"] = clf.num_digits_
        # logistic regression path (features, not kernels)
        clf = m.Classifier(LogisticRegression(), epochs_per_subj=4)
        clf.fit(list(zip(a[:12], b[:12])), labels[:12])
        out[tag + "_lr_decision"] = clf.decision_function(test)
        out[tag + "_lr_predict"] = clf.predict(test)
    # a larger kernel build with several portions and a ragged last portion
    V1, V2, T, E, eps = 90, 70, 16, 12, 4
    x1, x2, lab = synthetic.make_two_masks(V1, V2, T, E)
    c3 = m.Classifier(svc(), num_processed_voxels=32, epochs_per_subj=eps)
    c3.num_voxels_, c3.num_features_, c3.num_samples_ = V1, V1 * V2, E
    K3, _ = c3._compute_kernel_matrix_in_portion(x1, x2)
    out.update(big_x1=np.stack(x1), big_x2=np.stack(x2), big_kernel=K3,
               big_num_digits=c3.num_digits_, big_eps=eps, big_portion=32)
    np.savez_compressed(os.path.join(OUT, "clf.npz"), **out)
    print("clf: one", out["one_predict"], "two", out["two_predict"],
          "digits", out["one_num_digits"], out["big_num_digits"])


def gen_util(m):
    prng = RandomState(1234567890)   # reference tests/fcma/test_util.py:20-54
    mat1 = prng.rand(5, 10).astype(np.float32)
    mat2 = prng.rand(6, 10).astype(np.float32)
    c11 = m.util.compute_correlation(mat1, mat1)
    c12 = m.util.compute_correlation(mat1, mat2)
    mat1n = prng.rand(5, 10).astype(np.float32)
    mat2n = prng.rand(6, 10).astype(np.float32)
    mat1n[0, 0] = np.nan
    cn0 = m.util.compute_correlation(mat1n, mat2n, return_nans=False)
    cn1 = m.util.compute_correlation(mat1n, mat2n, return_nans=True)
    big1 = RandomState(7).randn(70, 45).astype(np.float32)
    big2 = RandomState(8).randn(33, 45).astype(np.float32)
    big2[5] = 3.0     # constant row -> zscore nan -> 0
    cb = m.util.compute_correlation(big1, big2)
    np.savez_compressed(os.path.join(OUT, "util.npz"), mat1=mat1, mat2=mat2, c11=c11, c12=c12,
                        mat1n=mat1n, mat2n=mat2n, cn0=cn0, cn1=cn1, big1=big1, big2=big2, cb=cb)
    print("util: ok")


def read_nifti(path):
    """Minimal NIfTI-1 reader (nibabel is absent): returns the data array in Fortran order."""
    with gzip.open(path, "rb") as f:
        buf = f.read()
    dim = struct.unpack_from("<8h", buf, 40)
    datatype, bitpix = struct.unpack_from("<hh", buf, 70)
    vox_offset = int(struct.unpack_from("<f", buf, 108)[0])
    slope, inter = struct.unpack_from("<ff", buf, 112)
    dt = {2: np.uint8, 4: np.int16, 8: np.int32, 16: np.float32, 64: np.float64,
          256: np.int8, 512: np.uint16}[datatype]
    shape = dim[1:1 + dim[0]]
    n = int(np.prod(shape))
    arr = np.frombuffer(buf, dtype=np.dtype(dt).newbyteorder("<"), count=n, offset=vox_offset)
    arr = arr.reshape(shape, order="F").astype(np.float64)
    if slope not in (0.0,) and not math.isnan(slope):
        arr = arr * slope + inter
    return arr


def gen_preproc(m):
    """Pins a14 (_separate_epochs) with the reference's own golden file
    tests/fcma/data/expected_raw_data.npy (test_preprocessing.py:31-43)."""
    d = os.path.join(REF_TESTS, "io", "data")
    mask = read_nifti(os.path.join(d, "mask.nii.gz")).astype(bool)
    subj = [read_nifti(os.path.join(d, "subject%d_bet.nii.gz" % s)) for s in (1, 2)]
    activity = [s.astype(np.float32)[mask] for s in subj]          # image.py:136-140
    epochs = np.load(os.path.join(d, "epoch_labels.npy"))          # [subj][cond][epoch][TR]
    expected = np.load(os.path.join(REF_TESTS, "fcma", "data", "expected_raw_data.npy"))
    raw, labels = m.preprocessing._separate_epochs(activity, list(epochs))
    for a, b in zip(raw, expected):
        assert np.allclose(a, b), "mini NIfTI reader disagrees with the reference golden file"
    # a seeded synthetic case incl. a constant voxel (std 0 -> nan -> 0) and unequal epoch lengths
    prng = RandomState(99)
    act = [prng.randn(50, 30).astype(np.float32) * 3 + 10 for _ in range(3)]
    act[1][7, :] = 2.5
    ep = np.zeros((3, 2, 3, 30), np.int8)
    for s in range(3):
        ep[s, 0, 0, 0:6] = 1
        ep[s, 1, 0, 6:13] = 1
        ep[s, 0, 1, 14:20] = 1
        ep[s, 1, 1, 21:30] = 1
    raw2, labels2 = m.preprocessing._separate_epochs(act, list(ep))
    np.savez_compressed(
        os.path.join(OUT, "preproc.npz"),
        activity=np.stack(activity), epochs=epochs, expected_raw_data=expected,
        ref_raw=np.stack(raw), labels=np.array(labels),
        act2=np.stack(act), ep2=ep, labels2=np.array(labels2),
        **{"raw2_%d" % i: r for i, r in enumerate(raw2)})
    print("preproc: %d voxels, %d epochs; synthetic %d epochs" %
          (activity[0].shape[0], len(raw), len(raw2)))


def gen_vs_sym(m):
    """One mask, more than two 256-row tiles: pins the symmetric pipeline (blocks on/above the diagonal, row pass +
    column pass) against the unmodified reference's kernels and accuracies for EVERY voxel."""
    V, T, E, eps = 560, 20, 8, 4
    raw, labels = synthetic.make_epochs(V, T, E, informative=10, signal=1.0, seed=20260921)
    vs = m.VoxelSelector(labels, eps, 2, raw, voxel_unit=40, process_num=0)
    acc = accs(reference.run_voxel_selection(vs, svc()), V)
    _, _, k = stages_all(vs, V, 40)
    np.savez_compressed(os.path.join(OUT, "vs_sym.npz"), raw=np.stack(raw), labels=np.array(labels), eps=eps,
                        folds=2, acc=acc, kernels=k)
    print("vs_sym: top voxels", np.argsort(-acc, kind="stable")[:10], "acc", np.sort(acc)[-10:])


def ref_rows(m, raw, labels, eps, folds, s0, n0, mask_self=False):
    """Rows [s0, s0+n0) through the reference's stages (voxelselector.py:492-509): shrunk kernels and cross-validation
    accuracies.  mask_self: zero the self column after its normaliser."""
    vs = m.VoxelSelector(labels, eps, folds, raw, voxel_unit=n0, process_num=0)
    clf = svm.SVC(kernel="precomputed", shrinking=False, C=1)
    corr = vs._correlation_computation((s0, n0))
    m.fcma_extension.normalization(corr, eps)
    if mask_self:
        for i in range(n0):
            corr[i, :, s0 + i] = 0
    K = vs._prepare_for_cross_validation(corr, clf)
    acc = np.array([a for _, a in vs._do_cross_validation(clf, K, (s0, n0))])
    return K, acc


def input_probe(raw, seed, n=64):
    """n seeded input values (epoch, TR, voxel): the tests regenerate these large inputs and check them against this."""
    rng = RandomState(seed)
    idx = np.stack([rng.randint(0, len(raw), n), rng.randint(0, raw[0].shape[0], n),
                    rng.randint(0, raw[0].shape[1], n)], axis=1)
    return idx, np.array([raw[e][t, v] for e, t, v in idx], np.float32)


def gen_vs_scale(m):
    """Sampled rows of the BASELINE config shapes (inputs too large to store: regenerated by the tests from
    synthetic.make_epochs and checked against a probe) and the result-level noise floor case."""
    out = {}
    # configs[1]: V = 30 000, T = 200, E = 16, eps = 8, 2 folds; first pass, a middle pass, the ragged tail
    V, T, E, eps = 30000, 200, 16, 8
    raw, labels = synthetic.make_epochs(V, T, E)
    out["c1_probe_idx"], out["c1_probe"] = input_probe(raw, 1)
    out["c1_rows"] = np.array([64, 15008, V - 32])
    ks, accs_ = zip(*[ref_rows(m, raw, labels, eps, 2, s0, 32) for s0 in out["c1_rows"]])
    out["c1_kernels"], out["c1_acc"] = np.stack(ks), np.stack(accs_)
    # configs[4] shape class: V = 20 000, T = 200, E = 32, eps = 8; kernels only (symmetric: upper triangle stored)
    V, T, E, eps = 20000, 200, 32, 8
    raw, labels = synthetic.make_epochs(V, T, E)
    out["c4_probe_idx"], out["c4_probe"] = input_probe(raw, 4)
    out["c4_rows"] = np.array([256, 10016, V - 32])
    ks = np.stack([ref_rows(m, raw, labels, eps, 4, s0, 32)[0] for s0 in out["c4_rows"]])
    assert np.array_equal(ks, ks.transpose(0, 1, 3, 2))
    iu = np.triu_indices(E)
    out["c4_kernels_triu"] = ks[:, :, iu[0], iu[1]]
    # noise floor: V = 768, T = 200, E = 32, eps = 8, 4 folds; every voxel, on the inputs, on TR-permuted inputs and with
    # the self column masked
    V, T, E, eps = 768, 200, 32, 8
    raw, labels = synthetic.make_epochs(V, T, E)
    out["nf_probe_idx"], out["nf_probe"] = input_probe(raw, 768)
    perm = RandomState(7).permutation(T)
    raw_p = [np.ascontiguousarray(x[perm]) for x in raw]
    out["nf_acc"] = ref_rows(m, raw, labels, eps, 4, 0, V)[1]
    out["nf_acc_perm"] = ref_rows(m, raw_p, labels, eps, 4, 0, V)[1]
    out["nf_acc_masked"] = ref_rows(m, raw, labels, eps, 4, 0, V, mask_self=True)[1]
    np.savez_compressed(os.path.join(OUT, "vs_scale.npz"), **out)
    print("vs_scale: noise floor %.3f" % np.mean(out["nf_acc"] != out["nf_acc_perm"]))


def main():
    m = reference.load()
    only = {"vs_sym": gen_vs_sym, "vs_scale": gen_vs_scale}
    if len(sys.argv) > 1 and sys.argv[1] in only:      # add this fixture without regenerating the others
        only[sys.argv[1]](m)
        return
    gen_vs_scale(m)
    gen_vs_sym(m)
    gen_vs_small(m)
    gen_vs_mid(m)
    gen_clf(m)
    gen_util(m)
    gen_preproc(m)


if __name__ == "__main__":
    main()
