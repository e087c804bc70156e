"""Device-resident decode timing of one configuration: python scripts/decode_probe.py CHANSTR RESOLUTION [reps].
Prints ms per decode of all leaves (CUDA events), points and an order-sensitive checksum."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench

chanstr, res = sys.argv[1], int(sys.argv[2])
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
torch.cuda.set_device(0)
pts, origins = bench.make_cloud(res)
thh = 0.65
dw = bench.DecodeWorkload(chanstr, 0, 1, pts, origins, thh)
for i in range(2):
    r = dw.step(i, False)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for i in range(reps):
    r = dw.step(i, False)
e1.record()
torch.cuda.synchronize()
c = r["coords"].cpu().long()
w = torch.arange(1, c.shape[0] + 1, dtype=torch.int64) % 1000003
chk = int(((c * torch.tensor([1, 1 << 11, 1 << 22])).sum(1) * w).sum() % (1 << 61))
print("%s res %d: %d leaves, %.3f ms per decode, %d points, checksum %d" % (
    chanstr, res, dw.n_all, e0.elapsed_time(e1) / reps, c.shape[0], chk))
