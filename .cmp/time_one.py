import sys, json, torch
sys.path.insert(0, ".")
from poseestimationkf_b200 import batched as B
from poseestimationkf_b200.synth import make_imu
dev = torch.device("cuda:0")
Ns, G, T = 256, 256, 2000
imu = make_imu(Ns, T, seed=3, sigma=0.01, device=dev)
N = Ns * G
q = torch.logspace(-2, 0, G, device=dev).repeat_interleave(Ns).contiguous(); r = torch.full((N,), 0.1, device=dev)
dt = torch.full((T, Ns), imu.dt, device=dev)
def run():
    st = B.ReplayState.initial(N, dev, r=r)
    B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=dt, q=q, r=r, n_filters=N, state=st, staging="tma_packed",
             share_measurements=False, precise_state=False, innovation=True, innovation_model="tangent")
    return st
st = run(); torch.cuda.synchronize()
ms = []
for _ in range(9):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); run(); e1.record(); torch.cuda.synchronize(); ms.append(e0.elapsed_time(e1))
print(json.dumps({"lib": sys.argv[1], "ms_median": sorted(ms)[4], "innov_sum": float(st.innov.double().sum())}))
