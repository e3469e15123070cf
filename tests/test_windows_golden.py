"""The window batcher against the reference's OWN AddBiomechanicsDataset.

tests/golden/windows.npz was produced by oracle/gen_golden.py::gen_windows, which runs the real class
(/root/reference/src/data/AddBiomechanicsDataset.py:64-139 index, 161-285 __getitem__) over seeded synthetic
subjects through oracle/fake_nimble.py, and torch's DistributedSampler + DataLoader as wired at
/root/reference/src/cli/train.py:143-150.  Bar: bit-exact (integer index, fp32 copies, fp32 divide by mass).

CPU tests pin oracle/windows.py; the -m gpu tests pin the CUDA index/packer kernels and WindowStore.
"""
import os

import numpy as np
import pytest
import torch

from oracle import windows as ow
from oracle.gen_golden import WINDOW_CASES, WINDOW_LABEL_KEYS, window_digest

GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "windows.npz"))
CASES = sorted(WINDOW_CASES)


def _case(name):
    seed, n_subj, T, s, fmt, hist, max_len, _ = WINDOW_CASES[name]
    assert list(GOLD[f"{name}/meta"][:6]) == [seed, n_subj, T, s, hist, max_len] and str(GOLD[f"{name}/format"]) == fmt
    subjects = ow.make_synthetic_subjects(seed, n_subj, T, hist_cols=hist, max_len=max_len)
    return subjects, T, s, fmt, hist


@pytest.mark.parametrize("name", CASES)
def test_oracle_window_index_matches_reference_class(name):
    subjects, T, s, fmt, _ = _case(name)
    want = [tuple(int(v) for v in r) for r in GOLD[f"{name}/windows"]]
    assert len(want) > 20
    assert ow.enumerate_windows(subjects, T, s) == want


@pytest.mark.parametrize("name", CASES)
def test_oracle_getitem_matches_reference_class(name):
    subjects, T, s, fmt, _ = _case(name)
    windows = ow.enumerate_windows(subjects, T, s)
    nb = int(GOLD[f"{name}/meta"][7])
    for i in GOLD[f"{name}/sample_idx"]:
        inputs, labels = ow.get_window(subjects, windows[int(i)], T, s, fmt, nb)
        for k in ow.INPUT_ORDER:
            want = GOLD[f"{name}/w{int(i)}/in/{k}"]
            assert inputs[k].dtype == np.float32 and inputs[k].shape == want.shape and np.array_equal(inputs[k], want), k
        for k in WINDOW_LABEL_KEYS:
            want = GOLD[f"{name}/w{int(i)}/label/{k}"]
            assert labels[k].shape == want.shape and np.array_equal(labels[k], want), k
    # every window of the dataset, through one digest
    got = window_digest(ow.get_window(subjects, w, T, s, fmt, nb) for w in windows)
    assert got == str(GOLD[f"{name}/digest"])


@pytest.mark.parametrize("name", CASES)
def test_oracle_sampler_and_loader_match_torch(name):
    subjects, T, s, fmt, _ = _case(name)
    windows = ow.enumerate_windows(subjects, T, s)
    idx = ow.sampler_indices(len(windows), 3, 1)
    assert idx == GOLD[f"{name}/sampler_r1w3"].tolist()
    bt = ow.batches(idx, 5)
    assert [len(b) for b in bt] == GOLD[f"{name}/loader_bs5_sizes"].tolist()
    assert [windows[i][0] for i in idx] == GOLD[f"{name}/loader_bs5_subject"].tolist()
    assert [windows[i][1] for i in idx] == GOLD[f"{name}/loader_bs5_trial"].tolist()
    nb = int(GOLD[f"{name}/meta"][7])
    for b, want in zip(bt, GOLD[f"{name}/loader_bs5_pos_sum"]):
        pos = np.stack([ow.get_window(subjects, windows[i], T, s, fmt, nb)[0]["pos"] for i in b])
        assert np.float64(pos.astype(np.float64).sum()) == pytest.approx(float(want), rel=1e-12, abs=1e-9)


# ------------------------------------------------ CUDA path ---------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_window_store_and_pack_match_reference_class(name):
    from inferbiomechanics_b200.data.window_store import WindowStore
    subjects, T, s, fmt, _ = _case(name)
    nb = int(GOLD[f"{name}/meta"][7])
    store = WindowStore.from_subjects(subjects, T, s, fmt, device="cuda", num_contact_bodies=nb)
    want = [tuple(int(v) for v in r) for r in GOLD[f"{name}/windows"]]
    assert store.windows == want                                   # GPU index: same windows, same order
    assert store.shard(1, 3).cpu().tolist() == GOLD[f"{name}/sampler_r1w3"].tolist()
    assert [b.numel() for b in WindowStore.batches(store.shard(1, 3), 5)] == GOLD[f"{name}/loader_bs5_sizes"].tolist()
    pick = GOLD[f"{name}/sample_idx"]
    idx = torch.from_numpy(pick).cuda()
    x = store.pack_f32(idx).cpu().numpy()                          # (B, F, C) fp32 gather
    lab = store.labels(idx).cpu().numpy()                          # (B, Fo, 30) rows30
    F, C = store.F, store.C
    ld = (F * C + 7) // 8 * 8
    ff16 = torch.zeros(len(pick), ld, dtype=torch.bfloat16, device="cuda")
    store.pack(idx, (ff16, C, ld - F * C, 0))                      # FeedForward layout: one row per window
    for bi, i in enumerate(pick):
        g_in = np.concatenate([GOLD[f"{name}/w{int(i)}/in/{k}"] for k in ow.INPUT_ORDER], axis=-1)
        assert np.array_equal(x[bi], g_in)
        g16 = torch.from_numpy(g_in.reshape(-1)).to(torch.bfloat16)                    # RNE, like the kernel
        assert torch.equal(ff16[bi, :F * C].cpu(), g16) and not ff16[bi, F * C:].any()
        g_lab = np.concatenate([GOLD[f"{name}/w{int(i)}/label/{k}"] for k in
                                ("groundContactCenterOfPressureInRootFrame", "groundContactForceInRootFrame",
                                 "groundContactTorqueInRootFrame", "groundContactWrenchesInRootFrame")], axis=-1)
        assert np.array_equal(lab[bi], g_lab)
    # all windows through the digest: rebuild the dicts from the packed tensors (inputs + the 4 contact labels; the
    # last-pass labels tau/residual/comAcc are not on the packed path — the loss never reads them — so they are taken
    # from the oracle, which the CPU test above pins to the same digest)
    allidx = torch.arange(len(store), device="cuda")
    X = store.pack_f32(allidx).cpu().numpy()
    L = store.labels(allidx).cpu().numpy()
    widths = ow.input_widths(int(GOLD[f"{name}/meta"][6]), WINDOW_CASES[name][5])
    items = []
    for wi, w in enumerate(want):
        _, olab = ow.get_window(subjects, w, T, s, fmt, nb)
        inp, c0 = {}, 0
        for k in ow.INPUT_ORDER:
            inp[k] = X[wi][:, c0:c0 + widths[k]]
            c0 += widths[k]
        lab_d = dict(olab)
        lab_d["groundContactCenterOfPressureInRootFrame"] = L[wi][:, 0:3 * nb]
        lab_d["groundContactForceInRootFrame"] = L[wi][:, 3 * nb:6 * nb]
        lab_d["groundContactTorqueInRootFrame"] = L[wi][:, 6 * nb:9 * nb]
        lab_d["groundContactWrenchesInRootFrame"] = L[wi][:, 9 * nb:15 * nb]
        items.append((inp, lab_d))
    assert window_digest(items) == str(GOLD[f"{name}/digest"])
