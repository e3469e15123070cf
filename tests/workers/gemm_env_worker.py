"""Worker of tests/test_gpu_gemm_matrix.py: runs GEMM case-table rows in a process whose environment carries one of the
library's process-wide switches (read once per process), and saves for each row the instantiations the profiler saw and
the outputs to <out_file>.

    python tests/workers/gemm_env_worker.py <out_file> <case id> [<case id> ...]
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))


def main(out_file, ids):
    import gemm_cases as gc
    results = {}
    for cid in ids:
        c = gc.find(cid)
        inp = gc.make_inputs(c)
        kerns, res = gc.profiled_launch(c, inp)
        results[cid] = {"kerns": sorted(kerns), **{k: v.cpu() for k, v in res.items()}}
    torch.save(results, out_file)


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2:])
