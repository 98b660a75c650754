"""Per-role cycle accounting of the tensor-core top-k kernel (retrieval_tc.cuh): where the tensor-core issue thread,
the operand producers and the epilogue warps of CTA (0, 0) spend their time, per database tile.

Needs a library built with the counters compiled in:
  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -diag-suppress 128 -DDSPX_TC_PROFILE \
       -Xcompiler -fPIC -shared -o gpurun_scratch/libdspx_prof.so dsp_final_b200/csrc/dspx.cu
  DSPX_LIBRARY=$PWD/gpurun_scratch/libdspx_prof.so python benchmarks/retr_tc_roles.py
"""
import ctypes, os, sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch
from dsp_final_b200 import retrieval as R
g = torch.Generator(device="cuda"); g.manual_seed(0)
names = ["mma wait acc_empty", "mma wait full_b", "mma issue+commit", "prod wait empty", "prod store", "epi wait acc_full", "epi masks", "epi enqueue+drain", "tiles", "mma total"]
for nq, ndb in ((8192, 262144), (20000, 1000000)):
    q = torch.randn((nq, 26), generator=g, device="cuda"); db = torch.randn((ndb, 26), generator=g, device="cuda")
    R.cosine_topk(q, db, 20); torch.cuda.synchronize()
    out = (ctypes.c_longlong * 16)()
    h = ctypes.CDLL(os.environ["DSPX_LIBRARY"])
    rc = h.dspx_debug_tc_prof(out)
    tiles = out[8]
    print(nq, ndb, "rc", rc, "tiles", tiles)
    for i, n in enumerate(names):
        if i != 8: print(f"   {n:22s} {out[i]/max(tiles,1):9.0f} cycles/tile")
