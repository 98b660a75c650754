import sys; sys.path.insert(0, str(__import__('pathlib').Path(__file__).resolve().parents[1]))
import torch, json
from dsp_final_b200 import synth
from dsp_final_b200.batch import stft_batch
clips = synth.device_clips(500, seed=1, device=torch.device('cuda'))
for fl,hop in ((1024,512),(512,256),(2048,1024)):
    for _ in range(3): out = stft_batch(clips, fl, hop)
    torch.cuda.synchronize()
    e0,e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5): out = stft_batch(clips, fl, hop)
    e1.record(); torch.cuda.synchronize()
    dt = e0.elapsed_time(e1)/5*1e-3
    nb = 500*(220500*4 + out.shape[1]*out.shape[2]*8)
    print(json.dumps({"stft":[fl,hop],"audio_s_per_s":500*5/dt,"ms":dt*1e3,"GBps":nb/dt/1e9}))
