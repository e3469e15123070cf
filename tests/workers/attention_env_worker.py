"""Worker of tests/test_gpu_attention_matrix.py: runs attention case-table rows in a process whose environment carries
one of the library's process-wide switches (read once per process), and saves for each row the instantiations the
profiler saw and the output buffers to <out_file> (only the instantiations with --kerns-only).  The matrix's dispatch
check runs here too, without a switch, so that its hundreds of profiler sessions stay out of the test process.

    python tests/workers/attention_env_worker.py [--kerns-only] <out_file> <case id> [<case id> ...]
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))


def main(out_file, ids, kerns_only=False):
    import attention_cases as ac
    results = {}
    for cid in ids:
        c = ac.find(cid)
        kerns, res = ac.profiled_launch(c, ac.make_inputs(c))
        results[cid] = {"kerns": sorted(kerns)}
        if not kerns_only:
            results[cid].update({k: v.cpu() for k, v in res.items() if torch.is_tensor(v)})
    torch.save(results, out_file)


if __name__ == "__main__":
    args = sys.argv[1:]
    only = args[0] == "--kerns-only"
    main(args[only], args[only + 1:], kerns_only=only)
