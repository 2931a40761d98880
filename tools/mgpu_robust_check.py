"""Sharded robust Grassmann averages (run under torchrun by tests/test_gpu_robust_select.py): every rank solves its row
shard of X with mu = entrywise_trimmed_mean / entrywise_median and compares it with the 1-GPU solve stored in the npz
file given as the only argument."""
import os, sys, warnings
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import torch.distributed as dist
import tlsq_b200 as T

rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dev = torch.device("cuda", lr)
dist.init_process_group("nccl", device_id=dev)
T.init_distributed(lr)
ref = np.load(sys.argv[1])
A, q0 = ref["A"], ref["q0"]
a0, a1 = T.synth.shard_rows(A.shape[0], world, rank)
Al = torch.from_numpy(np.ascontiguousarray(A[a0:a1].T)).to(dev).t()
ql = torch.from_numpy(np.ascontiguousarray(q0[a0:a1].T)).to(dev).t()
ok = True
for name, tag in (("trimmed", T.entrywise_trimmed_mean), ("median", T.entrywise_median)):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        Q, info = T.rpca_ga(Al, q0.shape[1], mu=tag, q0=ql, iters=30, return_info=True)
    Qn, Qr = Q.cpu().numpy(), ref[f"Q_{name}"][a0:a1]
    diff = np.abs(Qn - Qr).max()
    good = bool(diff < 1e-8 and list(info["iters"]) == list(ref[f"its_{name}"]))
    ok &= good
    print(f"[rank {rank}] {name} rows[{a0},{a1}) iters {info['iters']}/{list(ref[f'its_{name}'])} maxdiff {diff:.1e} "
          f"ok={good}", flush=True)
t = torch.tensor([1 if ok else 0], device=dev)
dist.all_reduce(t, op=dist.ReduceOp.MIN)
if rank == 0:
    print("MGPU_ROBUST", "PASS" if t.item() == 1 else "FAIL", flush=True)
dist.destroy_process_group()
