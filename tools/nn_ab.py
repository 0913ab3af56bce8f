"""Quick timing of one batched GetClosestNeighbor configuration (used for same-box A/B of library builds via KB_LIB)."""
import ctypes as C, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import kiss_icp_b200 as K
from kiss_icp_b200 import _native as N, synthetic
dev = torch.device("cuda", 0)
stream = torch.cuda.Stream(device=dev)
torch.cuda.set_stream(stream)
N.check(N.lib().kb_set_stream(C.c_void_p(stream.cuda_stream)))
m = K.VoxelHashMap(1.0, 1e9, 20)
m.add_points(synthetic.surface_cloud(1_000_000, seed=5))
stored = torch.from_numpy(m.point_cloud())
g = torch.Generator(device="cpu"); g.manual_seed(5)
n_q = 1 << 20
sel = stored[torch.randint(0, stored.shape[0], (n_q,), generator=g)]
q = (sel + torch.randn(n_q, 3, generator=g, dtype=torch.float64) * 0.3).to(dev).contiguous()
outp = torch.empty_like(q); outd = torch.empty(n_q, dtype=torch.float64, device=dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
ts = []
for it in range(8):
    flush.fill_(it)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    N.check(N.lib().kb_map_closest_neighbors_dev(m._h, C.c_void_p(q.data_ptr()), n_q, C.c_void_p(outp.data_ptr()), C.c_void_p(outd.data_ptr())))
    e1.record(stream)
    torch.cuda.synchronize()
    if it >= 3: ts.append(e0.elapsed_time(e1))
import hashlib
digest = hashlib.sha1(outp.cpu().numpy().tobytes() + outd.cpu().numpy().tobytes()).hexdigest()[:16]  # equal across library builds = bit-identical answers
print(os.environ.get("KB_LIB", "default"), "nn ms", round(float(np.median(ts)), 4), "checksum", float(outd[outd < 1e300].sum()),
      "sha1(points, distances)", digest, flush=True)
