"""HBM-resident window batcher.

The reference builds each window in Python, ~18 ``row_stack``s of per-frame tensors per window inside
DataLoader workers (/root/reference/src/data/AddBiomechanicsDataset.py:161-285), then concatenates and
copies to the device inside ``model.forward`` (FeedForwardRegressionBaseline.py:97-108).  Here the
frames of all trials sit once in HBM as fp32 rows (16-byte aligned leading dimension) and a batch is
one gather kernel (+ one label kernel); the window index is built on the GPU with the reference's
exact predicate and order (Dataset.py:131-139).  Reading ``.b3d`` files is nimblephysics' job and out
of scope: a store is filled from per-trial arrays (synthetic here; a one-off export elsewhere).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from .. import ops
from ..keys import MODEL_INPUT_ORDER


class WindowStore:
    def __init__(self, frames: torch.Tensor, raw_labels: torch.Tensor, missing: torch.Tensor, trial_len: Sequence[int],
                 trial_subject: Sequence[int], subject_mass: Sequence[float], subject_contact_idx: Sequence[Sequence[int]],
                 window_size: int, stride: int = 1, output_data_format: str = "last_frame", num_contact_bodies: int = 2,
                 frame_width: Optional[int] = None):
        """frames: fp32 CUDA [n_frames, ld] (first ``frame_width`` columns = per-frame model concat);
        raw_labels: fp32 CUDA [n_frames, >=15*nb] raw first-pass [cop|force|torque|wrench] in each subject's
        own body order; missing: uint8 CUDA [n_frames] (1 = GRF missing)."""
        self.device = frames.device
        self.frames, self.raw_labels, self.missing = frames, raw_labels, missing
        self.C = frame_width if frame_width is not None else frames.shape[1]
        self.window_size, self.stride, self.output_data_format = window_size, stride, output_data_format
        self.F = window_size // stride                      # frames read per window (Dataset.py:168)
        self.Fo = self.F if output_data_format == "all_frames" else 1
        self.nb = num_contact_bodies
        self.trial_len = np.asarray(trial_len, dtype=np.int64)
        self.trial_subject = np.asarray(trial_subject, dtype=np.int32)
        self.trial_base_np = np.concatenate([[0], np.cumsum(self.trial_len)[:-1]]).astype(np.int64) if len(trial_len) else np.zeros(0, np.int64)
        self.trial_base = torch.from_numpy(self.trial_base_np).to(self.device)
        self.subject_mass = torch.tensor(list(subject_mass), dtype=torch.float32, device=self.device)
        self.subject_contact_idx = torch.tensor([list(c) for c in subject_contact_idx], dtype=torch.int32, device=self.device).view(-1, self.nb)
        self._build_index()

    # ---- window index (Dataset.py:131-139), on the GPU -------------------------------------------
    def _build_index(self):
        n_cand = np.maximum(self.trial_len - self.window_size - 1, 0)            # range(max(L - T - 1, 0))
        total = int(n_cand.sum())
        if total == 0:
            self.win_trial = torch.zeros(0, dtype=torch.int32, device=self.device)
            self.win_start = torch.zeros(0, dtype=torch.int32, device=self.device)
        else:
            counts = torch.from_numpy(n_cand).to(self.device)
            cand_trial = torch.repeat_interleave(torch.arange(len(n_cand), device=self.device, dtype=torch.int32), counts)
            first = torch.cumsum(counts, 0) - counts
            cand_start = (torch.arange(total, device=self.device) - torch.repeat_interleave(first, counts)).to(torch.int32)
            valid = torch.empty(total, dtype=torch.uint8, device=self.device)
            ops.window_valid_mask(self.missing, self.trial_base, cand_trial, cand_start, self.window_size, self.stride, valid)
            keep = torch.nonzero(valid, as_tuple=False).view(-1)                   # stream compaction keeps order
            self.win_trial, self.win_start = cand_trial[keep], cand_start[keep]
        self.win_row0 = self.trial_base[self.win_trial.long()] + self.win_start.long()
        subj = torch.from_numpy(self.trial_subject).to(self.device)[self.win_trial.long()].long() if len(self.trial_subject) else torch.zeros(0, dtype=torch.long, device=self.device)
        self.win_subject = subj

    def __len__(self) -> int:
        return int(self.win_row0.numel())

    @property
    def windows(self) -> List[Tuple[int, int, int]]:
        """(subject, trial-within-subject, start) like the reference's ``dataset.windows``."""
        first_trial_of_subject = {}
        for ti, s in enumerate(self.trial_subject.tolist()):
            first_trial_of_subject.setdefault(s, ti)
        wt, ws = self.win_trial.cpu().tolist(), self.win_start.cpu().tolist()
        return [(int(self.trial_subject[t]), t - first_trial_of_subject[int(self.trial_subject[t])], s) for t, s in zip(wt, ws)]

    # ---- sharding (train.py:143: DistributedSampler(shuffle=False, drop_last=True)) ----------------
    def shard(self, rank: int, world_size: int) -> torch.Tensor:
        n = len(self)
        total = (n // world_size) * world_size
        return torch.arange(rank, total, world_size, device=self.device)

    @staticmethod
    def batches(indices: torch.Tensor, batch_size: int) -> List[torch.Tensor]:
        return [indices[i:i + batch_size] for i in range(0, indices.numel(), batch_size)]    # partial last batch kept

    # ---- packing -----------------------------------------------------------------------------------
    def pack(self, idx: torch.Tensor, layout) -> None:
        """Windows ``idx`` → bf16 rows in an engine's ``input_layout`` ``(buffer, frame_stride, win_extra, col0)``: frame t of
        window b starts at element (b * F + t) * frame_stride + b * win_extra + col0 of the buffer."""
        dst_bf16, frame_stride, win_extra, col0 = layout
        ops.pack_windows(self.frames, self.C, self.win_row0[idx], self.F, self.stride, out_bf16=dst_bf16, frame_stride=frame_stride,
                         win_extra=win_extra, col0=col0)

    def pack_f32(self, idx: torch.Tensor) -> torch.Tensor:
        out = torch.empty(idx.numel(), self.F, self.C, dtype=torch.float32, device=self.device)
        ops.pack_windows(self.frames, self.C, self.win_row0[idx], self.F, self.stride, out_f32=out)
        return out

    def labels(self, idx: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """rows30 labels fp32 [B, Fo, 30]: bodies re-ordered, force/torque/wrench divided by mass (Dataset.py:229-261)."""
        B = idx.numel()
        if out is None:
            out = torch.empty(B, self.Fo, 15 * self.nb, dtype=torch.float32, device=self.device)
        subj = self.win_subject[idx]
        ops.pack_labels(self.raw_labels, self.nb, self.win_row0[idx], self.subject_contact_idx[subj].contiguous(),
                        self.subject_mass[subj].contiguous(), self.F, self.stride, self.Fo == 1, out.view(B * self.Fo, -1))
        return out

    # ---- pre-packed store file (SURVEY §8f-1; replaces the pickled windows of src/cli/pickle_data.py:30-81 and
    #      src/data/PickledDataset.py:7-25 with the packer's own layout, so a training job maps the file and
    #      uploads three arrays instead of running Dataset.__getitem__ per window) -------------------------
    MAGIC = b"IBMSTORE1\0\0\0\0\0\0\0"          # 16 bytes

    def save(self, path: str) -> None:
        """[magic 16 B][header length u64][JSON header][64-byte-aligned sections: frames f32 [n, ld] | raw_labels f32
        [n, 15*nb] | missing u8 [n]].  Window size / stride / output format are NOT stored: they are indexing
        parameters chosen when the store is opened (Dataset.py:121-139)."""
        import json
        import struct
        arrays = [("frames", self.frames.cpu().numpy()), ("raw_labels", self.raw_labels.cpu().contiguous().numpy()),
                  ("missing", self.missing.cpu().numpy())]
        header = {"frame_width": int(self.C), "num_contact_bodies": int(self.nb), "trial_len": self.trial_len.tolist(),
                  "trial_subject": self.trial_subject.tolist(), "subject_mass": self.subject_mass.cpu().tolist(),
                  "subject_contact_idx": self.subject_contact_idx.cpu().tolist(), "sections": {}}
        off = 0
        for name, a in arrays:
            header["sections"][name] = {"offset": off, "shape": list(a.shape), "dtype": str(a.dtype)}
            off += (a.nbytes + 63) // 64 * 64
        blob = json.dumps(header).encode()
        pre = 16 + 8 + len(blob)
        pad = (-pre) % 64
        with open(path, "wb") as f:
            f.write(self.MAGIC)
            f.write(struct.pack("<Q", len(blob) + pad))
            f.write(blob + b" " * pad)
            for _, a in arrays:
                f.write(a.tobytes())
                f.write(b"\0" * ((-a.nbytes) % 64))

    @staticmethod
    def load(path: str, window_size: int, stride: int = 1, output_data_format: str = "last_frame", device="cuda") -> "WindowStore":
        import json
        import struct
        with open(path, "rb") as f:
            if f.read(16) != WindowStore.MAGIC:
                raise ValueError(f"{path} is not a window store file")
            (hlen,) = struct.unpack("<Q", f.read(8))
            header = json.loads(f.read(hlen).decode())
            base = 16 + 8 + hlen
        mm = np.memmap(path, dtype=np.uint8, mode="r")
        def section(name):
            sec = header["sections"][name]
            dt = np.dtype(sec["dtype"])
            n = int(np.prod(sec["shape"])) * dt.itemsize
            a = mm[base + sec["offset"]: base + sec["offset"] + n].view(dt).reshape(sec["shape"])
            return torch.from_numpy(np.array(a)).to(device)        # copy out of the read-only mapping, then upload
        return WindowStore(section("frames"), section("raw_labels"), section("missing"), header["trial_len"],
                           header["trial_subject"], header["subject_mass"], header["subject_contact_idx"], window_size, stride,
                           output_data_format, header["num_contact_bodies"], header["frame_width"])

    # ---- builders -------------------------------------------------------------------------------------
    @staticmethod
    def from_subjects(subjects: Sequence[dict], window_size: int, stride: int, output_data_format: str, device="cuda",
                      num_contact_bodies: int = 2, keys: Sequence[str] = MODEL_INPUT_ORDER) -> "WindowStore":
        """subjects: the synthetic-subject dicts of oracle/windows.py (any source with the same arrays works)."""
        fr, rw, ms, tl, ts, mass, cidx = [], [], [], [], [], [], []
        for si, s in enumerate(subjects):
            mass.append(s["mass"])
            cidx.append(s["contact_indices"])
            for tr in s["trials"]:
                fr.append(np.concatenate([tr[k] for k in keys], axis=1).astype(np.float32))
                rw.append(np.concatenate([tr["groundContactCenterOfPressureInRootFrame"], tr["groundContactForceInRootFrame"],
                                          tr["groundContactTorqueInRootFrame"], tr["groundContactWrenchesInRootFrame"]],
                                         axis=1).astype(np.float32))
                ms.append(np.asarray(tr["missing"]).astype(np.uint8))
                tl.append(len(tr["missing"]))
                ts.append(si)
        frames = np.concatenate(fr) if fr else np.zeros((0, 4), np.float32)
        C = frames.shape[1]
        ld = ops.round_up(C, 4)
        f = torch.zeros(frames.shape[0], ld, dtype=torch.float32, device=device)
        f[:, :C] = torch.from_numpy(frames).to(device)
        raw = torch.from_numpy(np.concatenate(rw) if rw else np.zeros((0, 15 * num_contact_bodies), np.float32)).to(device)
        missing = torch.from_numpy(np.concatenate(ms) if ms else np.zeros(0, np.uint8)).to(device)
        return WindowStore(f, raw, missing, tl, ts, mass, cidx, window_size, stride, output_data_format, num_contact_bodies, C)

    @staticmethod
    def synthetic(n_windows: int, window_size: int, stride: int, frame_width: int, output_data_format: str = "all_frames",
                  seed: int = 1234, device="cuda", trial_len: int = 2000) -> "WindowStore":
        """Synthetic AddBiomechanics-shaped store generated directly in HBM (SURVEY §8d): kinematics N(0,1); raw
        forces N(0,1)*700 N, torques *30, wrench *300, CoP N(0,1); masses U(45,110); no missing frames."""
        per_trial = trial_len - window_size - 1
        n_trials = (n_windows + per_trial - 1) // per_trial
        n_frames = n_trials * trial_len
        g = torch.Generator(device=device).manual_seed(seed)
        ld = ops.round_up(frame_width, 4)
        frames = torch.zeros(n_frames, ld, dtype=torch.float32, device=device)
        frames[:, :frame_width] = torch.randn(n_frames, frame_width, generator=g, device=device)
        raw = torch.randn(n_frames, 30, generator=g, device=device)
        raw[:, 6:12] *= 700.0
        raw[:, 12:18] *= 30.0
        raw[:, 18:30] *= 300.0
        missing = torch.zeros(n_frames, dtype=torch.uint8, device=device)
        n_subj = max(1, n_trials // 4)
        mass = (45.0 + 65.0 * torch.rand(n_subj, generator=g, device=device)).cpu().tolist()
        store = WindowStore(frames, raw, missing, [trial_len] * n_trials, [i % n_subj for i in range(n_trials)], mass,
                            [[0, 1] if i % 3 else [1, 0] for i in range(n_subj)], window_size, stride, output_data_format, 2,
                            frame_width)
        return store
