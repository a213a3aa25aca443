"""Per-GEMM cycle summary of CTA 0 of mlp_bwd (debug trace): epilogue, hand-over, copy-out, MMA phase.
usage: trace_bwd.py   (env TRACE_VERBOSE=1: per-layer stamps of the first iterations)"""
import os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import nerf_sh_oracle as O
from plenoctree_b200 import ops
from plenoctree_b200._lib import check, lib, ptr
flat = O.init_flat_params(3, 1, bias_scale=0.05)
blob = ops.pack_weights(torch.from_numpy(flat).cuda(), 3)
m = 148 * 256 * 6
tiles = (m + 511) // 512 * 4
G = torch.randn((m, 4), device="cuda") * 1e-3
vd = torch.nn.functional.normalize(torch.randn((m, 3), device="cuda"), dim=-1).contiguous()
mask = torch.randint(-2**31, 2**31 - 1, (8 * tiles * 128 * 8,), dtype=torch.int32, device="cuda")
dz = torch.empty(tiles * 8 * 65536, dtype=torch.uint8, device="cuda")
do = torch.empty(tiles * 32768, dtype=torch.uint8, device="cuda")
tr = torch.zeros((2, 256), dtype=torch.int64, device="cuda")
ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
for i in range(3):
    tr.zero_()
    if i == 2: ev[0].record()
    check(lib.pob_debug_trace_bwd(ptr(blob), 3, m, ptr(G), ptr(vd), ptr(mask), ptr(dz), ptr(do), ptr(tr), None))
ev[1].record()
torch.cuda.synchronize()
t = tr.cpu().numpy()
t0 = t[t > 0].min()
mma = t[0][t[0] > 0] - t0
e = t[1][t[1] > 0] - t0
mm = mma[: (len(mma) // 2) * 2].reshape(-1, 2)     # per GEMM: [operand X observed, all issued]
ee = e[: (len(e) // 4) * 4].reshape(-1, 4)         # per dZ layer: [d_ready, drained, handed over, (unused)]
n = min(len(ee), 24)
epi = (ee[:n, 1] - ee[:n, 0]); sig = (ee[:n, 2] - ee[:n, 1]); cp = (ee[:n, 3] - ee[:n, 2])
ph = (mm[:, 1] - mm[:, 0])
per = [int(mm[8 * (k + 1)][0] - mm[8 * k][0]) for k in range((len(mm) - 1) // 8)]
print(f"kernel {ev[0].elapsed_time(ev[1])*1e3:.0f} us | epilogue {epi.mean():.0f} "
      f"hand-over {sig.mean():.0f} copy-out {cp.mean():.0f} | MMA phase {np.median(ph):.0f} | iteration {np.mean(per):.0f} cycles")
if os.environ.get("TRACE_VERBOSE"):
    for k in range(min(10, len(ee))):
        print("  dZ", k, "d_ready", ee[k][0], "epi", epi[k], "sig", sig[k], "copy", cp[k], "| MMA a_rdy", mm[k][0], "issued", mm[k][1])
