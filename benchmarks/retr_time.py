import sys, os
sys.path.insert(0, str(__import__('pathlib').Path(__file__).resolve().parents[1]))
import torch
from dsp_final_b200 import retrieval as R
dev=torch.device('cuda'); g=torch.Generator(device=dev); g.manual_seed(5)
q=torch.randn((20000,26),generator=g,device=dev); db=torch.randn((1000000,26),generator=g,device=dev)
for _ in range(2): R.cosine_topk(q,db,20)
torch.cuda.synchronize()
e0,e1=torch.cuda.Event(enable_timing=True),torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(5): R.cosine_topk(q,db,20)
e1.record(); torch.cuda.synchronize()
print(os.environ.get('DSPX_LIBRARY','default'), 'ms per call', e0.elapsed_time(e1)/5)
