"""The window oracle against the reference's own AddBiomechanicsDataset, LIVE: where the original project's sources are
importable (IBM_REFERENCE_ROOT or the oracle/_ref snapshot; no stored copy of these cases exists, only the frozen
tests/golden/windows.npz of other cases) the real class runs over freshly drawn synthetic subjects
through oracle/fake_nimble.py and must agree with oracle/windows.py bit for bit — index (Dataset.py:131-139), every
__getitem__ dict (Dataset.py:161-285: strided frame gather, label re-order to the dataset's contact-body order, /mass except
CoP) — on seeds and shapes the frozen fixture never saw, including the degenerate ones: trials shorter than the window,
trials with every frame missing, a window as long as the trial allows, stride == window size, one subject."""
import tempfile

import numpy as np
import pytest

from oracle import windows as ow
from oracle.refimport import reference_available

pytestmark = pytest.mark.skipif(not reference_available(), reason="needs the original project's sources (IBM_REFERENCE_ROOT or oracle/_ref)")

CASES = [
    # seed, subjects, T, stride, format, hist_cols, max_len
    (101, 4, 50, 5, "all_frames", 15, 140),
    (102, 3, 50, 1, "last_frame", 30, 110),
    (103, 5, 12, 4, "all_frames", 12, 60),
    (104, 1, 30, 30, "last_frame", 90, 80),          # stride == window: one frame per window
    (105, 3, 9, 2, "all_frames", 6, 14),             # trials barely longer than the window (max_len = T + 5)
    (106, 2, 25, 7, "last_frame", 21, 70),           # T % stride != 0
]


def _degenerate(subjects, T):
    """Make the drawn subjects nastier: one trial entirely missing, one exactly T + 1 long (zero windows: range(max(L-T-1, 0)))
    and one T + 2 long (exactly one candidate window)."""
    tr = subjects[0]["trials"]
    tr[0]["missing"][:] = True
    for extra in (T + 1, T + 2):
        base = subjects[-1]["trials"][-1]
        short = {k: (v[:extra].copy() if isinstance(v, np.ndarray) and v.shape[0] >= extra else v) for k, v in base.items()}
        if short["missing"].shape[0] == extra:
            short["missing"] = np.zeros(extra, dtype=bool)
            subjects[-1]["trials"].append(short)
    return subjects


@pytest.mark.parametrize("seed,n_subj,T,s,fmt,hist,max_len", CASES)
def test_oracle_equals_live_reference_dataset(seed, n_subj, T, s, fmt, hist, max_len):
    from oracle.gen_golden import WINDOW_LABEL_KEYS, reference_dataset
    subjects = _degenerate(ow.make_synthetic_subjects(seed, n_subj, T, hist_cols=hist, max_len=max_len), T)
    with tempfile.TemporaryDirectory() as tmp:
        ds = reference_dataset(subjects, T, s, fmt, tmp)
        want = [tuple(int(v) for v in w) for w in ds.windows]
        got = ow.enumerate_windows(subjects, T, s)
        assert got == want
        assert len(want) > 0
        nb = ds.num_contact_bodies
        step = max(1, len(want) // 25)                 # ~25 windows per case, plus the first and last
        for i in sorted(set(list(range(0, len(want), step)) + [0, len(want) - 1])):
            inp, lab, si, ti = ds[i]
            assert (si, ti) == want[i][:2]
            o_in, o_lab = ow.get_window(subjects, want[i], T, s, fmt, nb)
            for k in ow.INPUT_ORDER:
                a = inp[k].numpy()
                assert o_in[k].dtype == np.float32 and o_in[k].shape == a.shape and np.array_equal(o_in[k], a), (i, k)
            for k in WINDOW_LABEL_KEYS:
                a = lab[k].numpy()
                assert o_lab[k].shape == a.shape and np.array_equal(o_lab[k], a), (i, k)
