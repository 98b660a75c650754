import sys; sys.path.insert(0, str(__import__('pathlib').Path(__file__).resolve().parents[1]))
import torch, json
from dsp_final_b200 import synth
from dsp_final_b200.batch import features_batch, log_mel_nchw
from dsp_final_b200.dsp.mfcc import MfccConfig
clips = synth.device_clips(1000, seed=4, device=torch.device('cuda'))
for nm in (40, 128):
    cfg = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512, n_mels=nm)
    for name, fn in (("time_major", lambda: features_batch(clips, cfg, ("log_mel",))), ("nchw", lambda: log_mel_nchw(clips, cfg))):
        for _ in range(3): fn()
        torch.cuda.synchronize()
        e0,e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10): fn()
        e1.record(); torch.cuda.synchronize()
        dt = e0.elapsed_time(e1)/10*1e-3
        print(json.dumps({"n_mels": nm, "layout": name, "audio_s_per_s": round(1000*5/dt), "ms": round(dt*1e3,3)}), flush=True)
