"""Multi-GPU check of lowrankfilter with lag > 1 on the factored route (run under torch.distributed.run with 2 ranks):
n = 256 on replicated signals of 6 sinusoids, lag 2 and 3.  The Hankel row counts are odd, so the last shard has an odd
row count and every rank takes the one-pass kernel.  Each rank first solves the whole problem on its own GPU (before the
communicator is attached), then the sharded one, and compares the sharded filtered signal with its single-GPU result
(1e-12) and with the CPU oracle (1e-9, same iteration count and rank history)."""
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
relF = lambda a, b: float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))
n, k, K = 256, 6, 20_001


def unhankel_lag(A, lag, Ns):
    Kr, L = A.shape
    s, cnt = np.zeros(Ns), np.zeros(Ns)
    for l in range(L):
        s[l:l + (Kr - 1) * lag + 1:lag] += A[:, l]
        cnt[l:l + (Kr - 1) * lag + 1:lag] += 1
    return s / np.maximum(cnt, 1)


cases = []
for lag in (2, 3):
    Ns = (K - 1) * lag + n
    _, y = T.synth.sinusoids_np(Ns, k, seed=5)
    yd = torch.from_numpy(y).to(dev)
    yf1, info1 = T.lowrankfilter(yd, n, lag=lag, return_info=True)          # single GPU: no communicator yet
    cases.append((lag, Ns, y, yd, yf1.cpu().numpy(), info1))

dist.init_process_group("nccl", device_id=dev)
T.init_distributed(lr)
per = ((K + world - 1) // world + 31) // 32 * 32                           # solver.cu shard_hankel_rows
last = K - per * (world - 1)
ok = True
for lag, Ns, y, yd, yf1, info1 in cases:
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = O.rpca(O.hankel(y, n, lag), tol=1e-3)
    yo = unhankel_lag(ref.A, lag, Ns)
    T.set_profiling(True, lr)
    yf, info = T.lowrankfilter(yd, n, lag=lag, return_info=True)
    prof = T.get_profile(lr)
    T.set_profiling(False, lr)
    yf = yf.cpu().numpy()
    e_single, e_oracle = relF(yf, yf1), relF(yf, yo)
    good = (e_single < 1e-12 and e_oracle < 1e-9 and info["iters"] == ref.iters == info1["iters"]
            and np.array_equal(info["hist"][:, 1], ref.hist[:, 1]) and prof["fused"][1] > 0
            and prof["epilogue"][1] == 0)
    ok &= bool(good)
    print(f"[rank {rank}] lowrankfilter lag={lag} Ns={Ns}: shards {per} x {world - 1} + {last}, iters "
          f"{info['iters']}/{ref.iters}, vs single GPU {e_single:.1e}, vs oracle {e_oracle:.1e}, fused spans "
          f"{prof['fused'][1]} ok={good}", flush=True)
t = torch.tensor([1 if ok else 0], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MIN)
if rank == 0:
    print("MGPU_LAG", "PASS" if t.item() == 1 else "FAIL", flush=True)
dist.destroy_process_group()
