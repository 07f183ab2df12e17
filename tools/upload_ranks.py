"""Upload of this rank's share of C3 (12.5M x 16 doubles, 1.6 GB) from pageable numpy memory through the pinned bounce
buffers (context.cu, staged_h2d) with every rank of the job uploading at once, twice.  Run under torchrun; one JSON line."""
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ml_b200 import cabi  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
box = [cabi.nccl_unique_id() if rank == 0 else None]
dist.broadcast_object_list(box, src=0)
ctx = cabi.Context.for_rank(local, rank, world, box[0])
n_total, d = 12_500_000 * world, 16
begin, end = cabi.shard_range(n_total, world, rank)
n = end - begin
points = np.random.default_rng(rank).normal(size=(n, d))
gb = points.nbytes / 1e9
out = {"world": world, "gb_per_rank": gb, "host_cores": os.cpu_count()}
for _ in range(2):
    dist.barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    dev = cabi.Data.upload(ctx, points, n_total=n_total)
    ctx.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    check = bool(np.array_equal(dev.download(begin, 1000), points[:1000]) and np.array_equal(dev.download(end - 1000, 1000), points[-1000:]))
    dev.close()
    out.setdefault("staged", []).append({"max_seconds": float(t.item()), "gb_per_s_per_rank": gb / float(t.item()), "round_trip_ok": check})
if rank == 0:
    print(json.dumps(out), flush=True)
dist.barrier()
dist.destroy_process_group()
