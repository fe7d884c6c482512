import os, sys, time; sys.path[:0]=[os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", d) for d in (".", "dnn-mppi-mpc_b200", "tests")]
import os, numpy as np, torch
NH = int(os.environ.get("NH", "2")); NIN = int(os.environ.get("NIN", "3"))    # hidden tanh layers (2 | 3), inputs (3 | 5)
from golden_util import Golden
from gpu_util import engine_from_spec
from oracle import mppi_oracle as orc
g = Golden("diffdrive_pe0.05")
K,T = 65536,30
mlp = orc.make_mlp(seed=0, out_scale=0.01, n_hidden=NH, n_in=NIN)
sp = orc.diffdrive_spec(K=K, T=T, param_exploration=0.05, cost_mode="sum", waypoint_mode="frozen", model="diffdrive_mlp", mlp=mlp)
sp.temperature = 2.0
eng = engine_from_spec(sp, g.path)
eng.set_mlp([mlp["W%d"%i] for i in range(NH + 2)],[mlp["b%d"%i] for i in range(NH + 2)])
st = torch.cuda.Stream(); eng.set_stream(st.cuda_stream)
x0=np.array([0.4,0.3,0.5])
for i in range(3): eng.step_async(x0, None, 7, i)
torch.cuda.synchronize()
a,b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
n=10
a.record(st)
for i in range(n): eng.step_async(x0, None, 7, 10+i)
b.record(st); torch.cuda.synchronize()
ms=a.elapsed_time(b)/n
print(f"MLP NH={NH} NIN={NIN} K={K} T={T}: {ms:.3f} ms/tick  {K*T/ms/1e6:.3f} G sample-steps/s  executed-GEMM {K*T*2*512*512*(NH-1)/ms/1e9/1e3:.3f} PFLOP/s")
# accuracy on a subset
Ks=2048
sp2 = orc.diffdrive_spec(K=Ks, T=T, param_exploration=0.05, cost_mode="sum", waypoint_mode="frozen", model="diffdrive_mlp", mlp=mlp); sp2.temperature=2.0
e2 = engine_from_spec(sp2, g.path); e2.set_mlp([mlp["W%d"%i] for i in range(NH + 2)],[mlp["b%d"%i] for i in range(NH + 2)])
eps = torch.zeros(Ks,T,2,device="cuda"); e2.generate_noise(eps, seed=3, tick=1)
S = torch.zeros(Ks,device="cuda"); e2.rollout_costs(x0,S,None,seed=3,tick=1)
So,_,_ = orc.costs_vec(sp2, g.path, np.zeros((T,2)), 0, x0, eps.cpu().numpy().astype(np.float64))
rel=np.abs(S.cpu().numpy()-So)/So
print("rel err max %.2e median %.2e"%(rel.max(), np.median(rel)))
