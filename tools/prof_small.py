import os, sys, json, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import drecpy_b200 as drb
from drecpy_b200 import _lib
lib=_lib.load()
def prof(m, fn, n=50):
    for _ in range(10): fn()
    torch.cuda.synchronize()
    e0,e1=torch.cuda.Event(enable_timing=True),torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    ms=e0.elapsed_time(e1)/n
    _lib.check(lib.drb_ctx_profile_enable(m._ctx,1))
    for _ in range(20): fn()
    p=_lib.profile_read(m._ctx); _lib.check(lib.drb_ctx_profile_enable(m._ctx,0))
    return ms, {k:(round(v[0]/20*1000,1), v[1]//20) for k,v in p.items()}
# C1 CDAE
u,i,v=drb.synthetic_interactions(943,1682,100000,seed=10)
ds=drb.InteractionData(u,i,v)
for gemm in ('tcgen05','ffma'):
    m=drb.CDAE(hidden_factors=50,seed=10,verbose=False,rng_mode='philox',gemm=gemm); m.fit(ds,epochs=0,batch_size=64)
    uu=m._sampler.sample_arrays(64)[0]; off=np.zeros(65,np.int32); _lib.check(lib.drb_batch_offsets(_lib.np_ptr(uu),64,_lib.np_ptr(m._h_indptr),_lib.np_ptr(off)))
    du,do=torch.as_tensor(uu,device='cuda'),torch.as_tensor(off,device='cuda'); loss=torch.zeros(2,device='cuda')
    ms,k=prof(m, lambda: m.step_device(du,do,None,1e-3,loss))
    print('C1',gemm,'ms/step',ms,'samples/s',64/ms*1e3,'kernels us',k)
    t=time.perf_counter()
    for s in range(200):
        m._step+=1; m._train_step(64,1e-3,want_loss=True,prefetch=True)
    print('  e2e philox samples/s', 64*200/(time.perf_counter()-t))
m=drb.CDAE(hidden_factors=50,seed=10,verbose=False); m.fit(ds,epochs=0,batch_size=64)
t=time.perf_counter()
for s in range(200):
    m._step+=1; m._train_step(64,1e-3,want_loss=True,prefetch=True)
print('C1 e2e mt19937 (reference-faithful) samples/s', 64*200/(time.perf_counter()-t))
# C2 DMF
u,i,v=drb.synthetic_interactions(6040,3706,1000000,seed=10)
ds=drb.InteractionData(u,i,v)
m=drb.DMF(seed=10,verbose=False); m.fit(ds,epochs=0,batch_size=256,reg_rate=1e-4)
uu,ii,vv=m._sampler.sample_arrays(256)
du,di,dl=torch.as_tensor(uu,device='cuda'),torch.as_tensor(ii,device='cuda'),torch.as_tensor(m.labels_from_values(vv),device='cuda'); loss=torch.zeros(2,device='cuda')
ms,k=prof(m, lambda: m.step_device(du,di,dl,1e-4,loss))
print('C2 DMF ms/step',ms,'samples/s',256/ms*1e3,'kernels us',k)
