import os, sys
sys.path.insert(0, '/root/repo'); sys.path.insert(0, '/root/repo/tests')
import torch, ntm_b200
from ntm_b200 import lib, signals
from conftest import load_ckpt
dev="cuda:0"; L=lib.load()
e0,e1=torch.cuda.Event(enable_timing=True),torch.cuda.Event(enable_timing=True)
with torch.inference_mode():
    m=ntm_b200.RNN(1,64,1,False).to(dev); m.load_state_dict(load_ckpt("cfg2")); m.mode="f16"
    m.initialize_hidden(); m.warm_start(); hw=m.hidden.clone()
    for B,T in ((2048,24000),(4096,12000),(4736,12000),(8192,12000),(9472,12000),(12000,6000),(16000,6000)):
        x=signals.stream_batch_device(B,T,dev,dur=10.0).reshape(B,1,T)
        row=[]
        for tune in ((8,3),(1,4),(0,0)):
            L.ntm_set_tuning(*tune)
            m.hidden=hw.expand(1,B,64).contiguous(); m(x[:,:,:1000])
            best=1e9
            for _ in range(2):
                m.hidden=hw.expand(1,B,64).contiguous()
                e0.record(); y=m(x); e1.record(); torch.cuda.synchronize(); best=min(best,e0.elapsed_time(e1))
            row.append(f"{tune} {best*1e6/T:7.1f} ns/step {B*T/best/1e6:6.2f} Gs/s")
        print(f"B={B}: "+" | ".join(row),flush=True)
L.ntm_set_tuning(0,0)
