import sys, time
sys.path.insert(0, str(__import__('pathlib').Path(__file__).resolve().parents[1]))
import torch
from dsp_final_b200 import retrieval as R
dev=torch.device('cuda'); g=torch.Generator(device=dev); g.manual_seed(5)
qa=torch.randn((20000,26),generator=g,device=dev); dba=torch.randn((1000000,26),generator=g,device=dev)
R.cosine_topk(qa,dba,20); torch.cuda.synchronize()
q=torch.randn((8192,26),generator=g,device=dev); db=torch.randn((262144,26),generator=g,device=dev)
ev=[]; wall=[]
for i in range(20):
    e0,e1=torch.cuda.Event(enable_timing=True),torch.cuda.Event(enable_timing=True)
    t0=time.perf_counter(); e0.record(); R.cosine_topk(q,db,20); e1.record(); torch.cuda.synchronize(); wall.append((time.perf_counter()-t0)*1e3); ev.append(e0.elapsed_time(e1))
print('event ms:', ' '.join(f'{x:.2f}' for x in ev))
print('wall  ms:', ' '.join(f'{x:.2f}' for x in wall))
