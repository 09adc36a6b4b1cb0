"""Run by test_q_features_kernel.py::test_form_b_build_rows in a subprocess with DDZ_LIB set to the -DDDZ_PROB_FORM_B build:
ddz_q_features' rows against the float64 first layer (and the bfloat16 rows against the float32 ones, bit for bit) on
mid-game envs, a batch with finished envs and the edge positions, all four env classes, every width of the test file.
Form B marks the probability planes' ranks 0..12 (right-aligned rows, the reversed half of the tables) and leaves their two
joker ranks unmarked: both must occur in the input, or the form-B paths of the kernel are not exercised."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ddz_b200 as D
import test_q_features_kernel as K

assert D.native.lib.ddz_prob_form() == 1, "not the form-B build"
worst = 0.0
for cls, C in K.CLASSES:
    envs = (K.midgame_env(D, cls), K.finished_mix_env(D, cls), K.edge_env(D, cls))
    right_aligned = jokers = 0
    for W in K.WIDTHS:
        for env in envs:
            x, w = K.check_env(D, env, C, W, seed=W + C)
            worst = max(worst, w)
            if W == K.WIDTHS[0]:
                prob = x[:, C - 2:C]
                right_aligned += int(((prob[:, :, :13, 0] == 0) & (prob[:, :, :13, 3] > 0)).sum())
                jokers += int((prob[:, :, 13:, 0] > 0).sum())
    assert right_aligned > 0 and jokers > 0, (cls, right_aligned, jokers)
print("largest err/bound %.3g" % worst)
print("form B q features ok")
