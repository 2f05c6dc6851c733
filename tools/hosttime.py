import time, numpy as np, torch, sys, os
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import sameold_b200 as sb
from sameold_b200 import synth
RATE=22050; ns=4096; secs=60.0
n=int(secs*RATE); stride=(n+7)//8*8
buf=torch.empty((ns,stride),dtype=torch.int16,device="cuda")
plans=synth.plan_corpus(ns,RATE,secs,first_stream=0)
synth.generate_on_device(plans,buf.data_ptr(),stride,n,RATE,device=0)
offsets=np.arange(ns,dtype=np.uint64)*np.uint64(stride); lengths=np.full(ns,n,np.uint32)
rx=sb.SameReceiverBuilder.samedec(RATE).build_batch(ns)
def step():
    t=[time.perf_counter()]
    rx.reset(); t.append(time.perf_counter())
    rx.submit_device(buf.data_ptr(), ns*stride, offsets, lengths); t.append(time.perf_counter())
    rx.sync(); t.append(time.perf_counter())
    evs,pay=rx.drain_raw(reuse=REUSE); t.append(time.perf_counter())
    return [ (b-a)*1e3 for a,b in zip(t,t[1:])], evs.size
for REUSE in (False, True, False, True):
  for i in range(3):
      d,nev=step(); print(REUSE, "reset %.2f submit %.2f sync(kernel+collect) %.2f drain %.2f ms; events %d; kernel %.2f" % (*d, nev, rx.last_timing()[1]))
