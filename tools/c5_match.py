"""Development aid: the C5-sized matching request (10 008 keyframes x 1000 ORB descriptors resident, one query keyframe),
timed on the device path of the map database."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, covins_b200
from covins_b200 import matching as M, synth
ctx = covins_b200.Context(0); dev = torch.device("cuda", 0)
n_kf, nf = int(sys.argv[1]) if len(sys.argv) > 1 else 10008, 1000
db = M.DescriptorDatabase(ctx, reserve_rows=n_kf * nf)
for c in range(0, n_kf, 1112):
    d, _ = synth.orb_keyframes(seed=100 + c, n_kf=min(1112, n_kf - c), n_feat=nf)
    db.append(d.reshape(-1, 32), [nf] * d.shape[0])
    if c == 0: q = torch.from_numpy(np.ascontiguousarray(d[7])).to(dev)
for _ in range(3): out = db.match_hamming_dev(q)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(10): out = db.match_hamming_dev(q)
e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / 10
print(f"{n_kf} KF: {ms:.3f} ms per request = {n_kf * nf * nf / ms / 1e6:.0f} Gpairs/s, accepted {int(out[2].sum())}", flush=True)
