"""Run by test_action_ids.py::test_form_b_build_ids in a subprocess with DDZ_LIB set to the -DDDZ_PROB_FORM_B build: that
build exports the id entry points (the binding checks every declared symbol at import), and ids, unranking and legal masks
do not depend on the probability form."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ddz_b200 as D
from oracle import ddz_oracle as O

assert D.native.lib.ddz_prob_form() == 1, "not the form-B build"
cnt = O.universe()[0]
packed = O.pack(cnt).astype(np.uint64)
assert np.array_equal(D.move_ids(packed).cpu().numpy(), np.arange(13551))
assert np.array_equal(D.moves_of_ids(torch.arange(13551, dtype=torch.int32)).cpu().numpy().view(np.uint64), packed)
env = D.BatchedEnvCooperation(512, seed=2)
env.prepare(*D.random_deals(512, seed=6))
for _ in range(20):
    env.step_random()
ids = env.legal_ids().to(torch.int64)
off = env.offsets.to(torch.int64)
owner = torch.repeat_interleave(torch.arange(512, device="cuda"), off[1:] - off[:-1], output_size=ids.numel())
want = torch.zeros((512, 13551), dtype=torch.bool, device="cuda")
want[owner, ids] = True
assert torch.equal(env.legal_mask("bool"), want)
bits = env.legal_mask("bits").to(torch.int64) & 0xFFFFFFFF
pad = torch.zeros((512, 424 * 32), dtype=torch.int64, device="cuda")
pad[:, :13551] = want.to(torch.int64)
assert torch.equal(bits, (pad.view(512, 424, 32) << torch.arange(32, device="cuda")).sum(-1))
print("form B ids ok")
