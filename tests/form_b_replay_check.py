"""Run by test_packed_replay.py::test_form_b_build_gather in a subprocess with DDZ_LIB set to the -DDDZ_PROB_FORM_B build:
ddz_encode_face_gather against ddz_encode_face and ddz_encode_actions of that build (split and concatenated layouts, rows
outside the batch, guard memory) on fresh, mid-game, finished and payload-ingested envs of all four env classes.  Form B
right-aligns the probability planes' ranks 0..12: the check asserts that such rows occur, or the form-B nibbles are not read."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ddz_b200 as D
import test_packed_replay as T


class Golden:
    core_payloads = np.load(os.path.join(ROOT, "tests", "golden", "core_payloads.npz"))


assert D.native.lib.ddz_prob_form() == 1, "not the form-B build"
for cls, C in T.CLASSES:
    rng = np.random.default_rng(C)
    right_aligned = 0
    for env in (T.fresh_env(D, cls, 7), T.midgame_env(D, cls), T.finished_env(D, cls), T.payload_env(D, cls, Golden)):
        T.check_gather(D, env, rng, T.SIZES)
        prob = T.encode_face(D, env._state, env.VARIANT, env.B)[:, C - 2:C]
        right_aligned += int(((prob[:, :, :13, 0] == 0) & (prob[:, :, :13, 3] > 0)).sum())
    assert right_aligned > 0, cls
print("form B replay ok")
