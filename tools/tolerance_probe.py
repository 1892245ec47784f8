#!/usr/bin/env python
"""Measures the quantities behind the result-level assertions of tests/test_gpu_parity.py so that their bounds can be
set per precision (VERDICT round 1, weak item 3)."""
import os, sys, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sklearn import svm
from brainiak_b200.fcma.voxelselector import VoxelSelector
g = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "vs_mid_run.npz"))
raw = list(g["rawf"]); labels = [int(x) for x in g["labelsf"]]; ref = g["accf"]
clf = svm.SVC(kernel='precomputed', shrinking=False, C=1)
for prec in ("fp32", "fp16x3", "tf32x3", "bf16x3", "tf32", "bf16"):
    for ms in (False,):
        res = VoxelSelector(labels, int(g["epsf"]), 4, raw, voxel_unit=32, process_num=2, precision=prec).run(clf)
        acc = np.zeros(raw[0].shape[1])
        for v, a in res:
            acc[v] = a
        top_ref = set(int(v) for v in np.argsort(-ref, kind="stable")[:12])
        top_got = set(v for v, _ in res[:12])
        print("vs_mid %-7s identical %.4f  max|d acc| %.4f  top12 overlap %d  V=%d E=%d" % (prec, np.mean(acc == ref), np.max(np.abs(acc - ref)), len(top_ref & top_got), len(acc), len(raw)))
g = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "vs_sym.npz"))
raw, eps, folds = list(g["raw"]), int(g["eps"]), int(g["folds"]); labels = [int(x) for x in g["labels"]]
for prec in ("fp32", "tf32x3", "bf16x3", "tf32", "bf16"):
    res = VoxelSelector(labels, eps, folds, raw, process_num=0, block_rows=256, precision=prec).run(clf)
    acc = np.zeros(raw[0].shape[1])
    for v, a in res:
        acc[v] = a
    print("vs_sym %-7s identical %.4f  max|d acc| %.4f" % (prec, np.mean(acc == g["acc"]), np.max(np.abs(acc - g["acc"]))))
