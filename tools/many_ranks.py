"""synthesize_many under the launcher's world size (1 process, or `torch.distributed.run --nproc-per-node N`, one GPU per
rank, NCCL) -> a JSON summary of the per-target Results on rank 0.  tests/test_gpu_multi_target.py runs it with 1 and 2
ranks and checks that sharding the target x sample items over GPUs changes nothing.

    python tools/many_ranks.py OUT.json
"""
import contextlib
import io
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


def main():
    out = sys.argv[1]
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        saved = os.dup(1)           # NCCL prints its version on stdout at communicator creation
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.all_reduce(torch.zeros(1, device="cuda"))
        finally:
            os.dup2(saved, 1)
    import cpflow_b200 as cp
    from cpflow_b200.gates import u_toff3
    from cpflow_b200.topology import chain_layer
    from scipy.stats import unitary_group
    ccz = np.diag([1, 1, 1, 1, 1, 1, 1, -1]).astype(complex)
    targets = np.stack([ccz, u_toff3, unitary_group.rvs(8, random_state=17)])
    opts = cp.StaticOptions(num_cp_gates=12, accepted_num_cz_gates=14, num_samples=41)
    with contextlib.redirect_stdout(io.StringIO()):
        res = cp.synthesize_many(chain_layer(3), targets, opts, labels=["ccz", "toffoli", "haar"])
    summary = [[[d.cz_count, repr(d.loss), np.asarray(d._cp_data[2]).astype(np.float64).tolist()]
                for d in r.decompositions] for r in res]
    if rank == 0:
        with open(out, "w") as f:
            json.dump({"world": world, "results": summary}, f)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
