"""Runs the REFERENCE's own dataset readers on files written by this repository's generators, with
``acoustic_echo_cancellation_b200.h5lite`` standing in for ``h5py`` -- TEST INFRASTRUCTURE, executed in a subprocess by
tests/test_h5lite.py and only where AEC_REFERENCE_DIR names a checkout of the reference.

    python run_reference_readers.py <repo root> <reference Stage2_lhm/scripts> <tr_list.txt> <tt/test.ex> <out.npz>

Imports Stage2_lhm/scripts/test.py:19-33 (``ValidateDataset``) and scripts/train1.py:29-42 (``TrainDataset``) unmodified
from the reference; ``soundfile`` (used only by the tester's wav writer) is stubbed with an empty module.
Every array the readers return is saved to <out.npz> for the caller to compare with what went in.
"""
import sys
import types

import numpy as np

repo, ref_scripts, tr_list, test_ex, out = sys.argv[1:6]
sys.path.insert(0, repo)
from acoustic_echo_cancellation_b200 import h5lite  # noqa: E402

sys.modules["h5py"] = h5lite
sys.modules.setdefault("soundfile", types.ModuleType("soundfile"))
sys.path.insert(0, ref_scripts)
saved_argv, sys.argv = sys.argv, [sys.argv[0]]
from test import ValidateDataset  # noqa: E402  (Stage2_lhm/scripts/test.py)
from train1 import TrainDataset  # noqa: E402   (Stage2_lhm/scripts/train1.py)
sys.argv = saved_argv

res = {}
paths = [ln.strip() for ln in open(tr_list) if ln.strip()]
tr = TrainDataset(paths)
res["train_len"] = np.array(len(tr))
for i in range(len(tr)):
    for k, v in tr[i].items():
        res[f"train/{i}/{k}"] = v
va = ValidateDataset(test_ex)
res["val_len"] = np.array(len(va))
for i in range(len(va)):
    for k, v in va[i].items():
        res[f"val/{i}/{k}"] = np.asarray(v)
np.savez(out, **res)
print("reference readers ok:", len(tr), "train files,", len(va), "test groups")
