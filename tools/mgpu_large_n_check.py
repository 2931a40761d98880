"""Multi-GPU parity above 2048 columns (run under torchrun): every rank solves its row shard of a 9000 x n matrix,
n = 2304 and n = 4096, and compares it with the CPU oracle run on the full matrix.  The n x n Gram all-reduce is
128 MB at n = 4096."""
import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import torch
import torch.distributed as dist

import tls_oracle as O
import tlsq_b200 as T

rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dev = torch.device("cuda", lr)
dist.init_process_group("nccl", device_id=dev)
T.init_distributed(lr)
relF = lambda a, b: float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))
ok = True
for (M, N, its) in [(9000, 2304, 4), (9000, 4096, 3)]:
    D = T.synth.lowrank_sparse_np(M, N, 10, 0.05, seed=M + N)
    r0, r1 = T.synth.shard_rows(M, world, rank, align=2)
    Dl = torch.from_numpy(np.ascontiguousarray(D[r0:r1].T)).to(dev).t()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        A, E, s, sv, info = T.rpca(Dl, iters=its, tol=0.0, return_info=True)
        ref = O.rpca(D, iters=its, tol=0.0)
    ea, ee = relF(A.cpu().numpy(), ref.A[r0:r1]), relF(E.cpu().numpy(), ref.E[r0:r1])
    S = s.S.cpu().numpy()
    es = float(np.abs(S - ref.s.S).max() / ref.s.S[0])
    Vt = s.Vt.cpu().numpy()
    eo = float(np.abs(Vt @ Vt.T - np.eye(Vt.shape[0])).max())
    good = ea < 1e-9 and ee < 1e-9 and es <= 1e-12 and eo < 1e-11 and sv == ref.sv and \
        np.array_equal(info["hist"][:, 1], ref.hist[:, 1])
    ok &= good
    print(f"[rank {rank}] rpca {M}x{N} rows[{r0},{r1}) relF A={ea:.1e} E={ee:.1e} S={es:.1e} Vt_orth={eo:.1e} "
          f"sv={sv}/{ref.sv} ok={good}", flush=True)
flag = torch.tensor([1.0 if ok else 0.0], device=dev)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
if rank == 0:
    print("MGPU_LARGE_N_CHECK PASS" if flag.item() > 0.5 else "MGPU_LARGE_N_CHECK FAIL", flush=True)
dist.destroy_process_group()
sys.exit(0 if flag.item() > 0.5 else 1)
