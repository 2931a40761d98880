"""Multi-GPU check of the one-pass kernel above rank 16 (run under torch.distributed.run with 2 ranks): lowrankfilter at
n = 256 on a replicated 20 256-sample signal of 13 sinusoids (rank estimate up to 26).  The 20 001 Hankel rows are split
10 016 + 9 985: the last shard has an odd row count, so every rank takes the one-pass kernel.  Each rank compares the
filtered signal, iteration count and rank history with the CPU oracle."""
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
Ns, k, n = 20_256, 13, 256
_, y = T.synth.sinusoids_np(Ns, k, seed=5)
with warnings.catch_warnings():
    warnings.simplefilter("ignore")
    ref = O.rpca(O.hankel(y, n), tol=1e-3)
yo = O.unhankel_fast(ref.A)
K = Ns - n + 1
per = ((K + world - 1) // world + 31) // 32 * 32                 # solver.cu shard_hankel_rows
last = K - per * (world - 1)
T.set_profiling(True, lr)
yf, info = T.lowrankfilter(torch.from_numpy(y).to(dev), n, return_info=True)
prof = T.get_profile(lr)
err = relF(yf.cpu().numpy(), yo)
good = (err < 1e-9 and info["iters"] == ref.iters and np.array_equal(info["hist"][:, 1], ref.hist[:, 1])
        and ref.hist[:, 1].max() > 16 and prof["fused"][1] > 0 and prof["epilogue"][1] == 0)
ok &= bool(good)
print(f"[rank {rank}] lowrankfilter Ns={Ns} k={k}: shards {per} x {world - 1} + {last}, iters {info['iters']}/{ref.iters}, "
      f"peak rank {int(info['hist'][:, 1].max())}/{int(ref.hist[:, 1].max())}, fused spans {prof['fused'][1]}, "
      f"rel {err:.1e} ok={good}", flush=True)
t = torch.tensor([1 if ok else 0], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MIN)
if rank == 0:
    print("MGPU_FUSED_RANK", "PASS" if t.item() == 1 else "FAIL", flush=True)
dist.destroy_process_group()
