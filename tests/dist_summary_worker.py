"""One rank of the multi-GPU histogram check (launched by tests/test_summaries.py through torch.distributed.run): every rank
sets the same seeded variables on an engine with row-sharded tables, the ranks bin them together (Engine.histograms: shards
binned per rank and summed, everything else binned by rank 0), and every rank compares the result with the float64
restatement of TensorFlow's histogram over the whole variables."""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from pamrec_b200.engine import Engine  # noqa: E402
from test_summaries import assert_same_histogram  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    eng = Engine(301, 3001, 53, 20, 10 * world, world_size=world, rank=rank, tables="sharded").allocate(f"cuda:{local}").init_comm()
    rng = np.random.default_rng(5)
    variables = {n: (rng.standard_normal(s) * 10.0 ** rng.integers(-4, 2)).astype(np.float32) for n, s in eng.variable_shapes().items()}
    eng.set_variables(variables)
    got = eng.histograms(list(variables)).result()
    again = eng.histograms(list(variables)).result()
    for name, val in variables.items():
        assert_same_histogram(got[name], val, name)
        assert all(np.array_equal(got[name][k], again[name][k]) for k in got[name]), name
    dist.barrier()
    if rank == 0:
        print(f"SUMMARY_DIST_OK world={world} variables={len(variables)}", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
