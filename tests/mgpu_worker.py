"""Worker for tests/test_multigpu_gpu.py (launched under torchrun, one process per rank).

Runs Step 1 twice on the same synthetic fileset - sharded over the ranks (level-0 blocks by the reference's
--split-l0 rule, level 1 by phenotype, W tiles stored into the owner's HBM through CUDA IPC) and unsharded on
this rank alone - and requires bit-identical CV sums, tau* and LOCO predictions: the invariant the reference
checks for its own multi-process mode (test/test_bash.sh:127-137, sharded == unsharded byte for byte).
With fewer GPUs than ranks the ranks share cuda:0 and torch.distributed runs on gloo; the IPC path is the same.
"""
import os
import sys
import tempfile

import numpy as np
import torch
import torch.distributed as dist
from torch.distributed.elastic.multiprocessing.errors import record

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import helpers  # noqa: E402
from oracle import prep  # noqa: E402
from regenie_b200 import sharding  # noqa: E402


def run(pb, dev, distributed):
    st = pb.gpu_step1(device=dev)
    nb = len(pb.blocks)
    B = nb * 5
    h1 = prep.set_ridge_params(5)
    tau = np.tile(B * (1 - h1) / h1, (pb.prep.Y.shape[1], 1))
    chr_of_block = [c for c, _, _ in pb.blocks]
    if distributed:
        out = sharding.step1_distributed(st, nb, lambda b: pb.gpu_l0_block(st, b), tau, chr_of_block,
                                         torch.device("cuda", dev))
    else:
        for b in range(nb):
            pb.gpu_l0_block(st, b)
        assert st.status() == 0
        cs, best = st.l1_fit(tau)
        out = (cs, best, st.loco(chr_of_block))
    st.close()
    return out


@record                                 # a failing rank's traceback goes into torchrun's error report
def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    ngpu = torch.cuda.device_count()
    dev = int(os.environ.get("LOCAL_RANK", rank)) % ngpu
    torch.cuda.set_device(dev)
    backend = "nccl" if ngpu >= world else "gloo"
    dist.init_process_group(backend=backend)
    for loocv in (False, True):
        with tempfile.TemporaryDirectory() as tmp:
            pb = helpers.synthetic_problem(tmp, N=900, M=700, P=3, C=3, bsize=100, K=5, seed=5, loocv=loocv)
            a = run(pb, dev, True)
            b = run(pb, dev, False)
        for x, y, name in zip(a, b, ("cumsums", "best_idx", "loco")):
            assert np.array_equal(x, y), (name, loocv, float(np.abs(np.asarray(x, float) - np.asarray(y, float)).max()))
    dist.barrier()
    print("MGPU_OK rank %d/%d backend=%s device=%d" % (rank, world, backend, dev), flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
