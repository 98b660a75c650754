import sys; sys.path.insert(0, str(__import__('pathlib').Path(__file__).resolve().parents[1]))
import torch, json
from dsp_final_b200 import synth
from dsp_final_b200.batch import features_batch
from dsp_final_b200.dsp.mfcc import MfccConfig
from dsp_final_b200.plan import get_plan
clips = synth.device_clips(500, seed=1, device=torch.device('cuda'))
for fl,hop,nfft in ((4096,256,None),(4096,1024,None),(400,160,512),(1000,300,None),(1024,511,None),(256,128,None)):
    cfg = MfccConfig(44100, fl, hop, n_fft=nfft)
    for _ in range(2): out = features_batch(clips, cfg, ("mfcc",))
    torch.cuda.synchronize()
    e0,e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3): out = features_batch(clips, cfg, ("mfcc",))
    e1.record(); torch.cuda.synchronize()
    dt = e0.elapsed_time(e1)/3*1e-3
    print(json.dumps({"cfg":[fl,hop,nfft],"kernel":get_plan(cfg).kernel,"audio_s_per_s":round(500*5/dt),"ms":round(dt*1e3,2)}))
