import sys, time, numpy as np, torch
sys.path.insert(0,'/root/repo')
from bench import make_shard, grid_hops, sigma_at
from dbgsom_b200.engine import DeviceEngine
dev=torch.device('cuda',0); n,d,side=10_000_000,256,64; m=side*side
X=make_shard(torch,dev,n,d,64,0)
host=torch.empty((n,d),dtype=torch.float32,pin_memory=True); host.copy_(X); torch.cuda.synchronize()
def t(f,k=3):
    torch.cuda.synchronize(); t0=time.perf_counter()
    for _ in range(k): f()
    torch.cuda.synchronize(); return (time.perf_counter()-t0)/k*1e3
print('plain copy ms', t(lambda: X.copy_(host,non_blocking=True)))
cs=torch.cuda.Stream()
def chunked():
    with torch.cuda.stream(cs):
        for c0 in range(0,n,1<<20):
            X[c0:c0+(1<<20)].copy_(host[c0:c0+(1<<20)],non_blocking=True)
    torch.cuda.current_stream().wait_stream(cs)
print('chunked copy on side stream ms', t(chunked))
eng=DeviceEngine(bmu_backend='tensor'); eng.load_device_data(X)
eng.init_map_from_rows(np.random.default_rng(0).choice(n,m,replace=False),capacity=m); eng.set_hops(grid_hops(side))
for e in range(3): eng.epoch(sigma_at(e,m),True,False)
print('resident epoch ms', t(lambda: eng.epoch(sigma_at(5,m),True,False)))
print('epoch_from_host ms', t(lambda: eng.epoch_from_host(host,sigma_at(5,m),True,False)))
print('epoch_from_host 4M chunks ms', t(lambda: eng.epoch_from_host(host,sigma_at(5,m),True,False,chunk_rows=1<<22)))
def serial():
    X.copy_(host,non_blocking=True); eng.samples.X16_hi=eng.samples.row_perm=None; eng.epoch(sigma_at(5,m),True,False)
print('serial copy+epoch ms', t(serial))
