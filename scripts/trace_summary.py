"""Per-layer-step cycle summary of CTA 0 of mlp_fwd (debug trace): epilogue, MMA phase, iteration period.
usage: trace_summary.py [save]   (save: with the training-mode stores)"""
import os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import nerf_sh_oracle as O
from plenoctree_b200 import ops
from plenoctree_b200._lib import check, lib, ptr
flat = O.init_flat_params(3, 1, bias_scale=0.05)
blob = ops.pack_weights(torch.from_numpy(flat).cuda(), 3)
m = 148 * 256 * 6
pts = (torch.rand((m, 3), device="cuda") * 3 - 1.5).contiguous()
sig = torch.empty(m, device="cuda")
tr = torch.zeros((5, 256), dtype=torch.int64, device="cuda")
saving = len(sys.argv) > 1 and sys.argv[1] == "save"
tiles = (m + 511) // 512 * 4
sh = torch.empty(tiles * 8 * 65536, dtype=torch.uint8, device="cuda") if saving else None
se = torch.empty(tiles * 16384, dtype=torch.uint8, device="cuda") if saving else None
sm = torch.empty(8 * tiles * 128 * 8, dtype=torch.int32, device="cuda") if saving else None
ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
for i in range(3):
    tr.zero_()
    if i == 2: ev[0].record()
    check(lib.pob_debug_trace_fwd(ptr(blob), 3, ptr(pts), m, ptr(sig), ptr(tr), ptr(sh), ptr(se), ptr(sm), None))
ev[1].record()
torch.cuda.synchronize()
t = tr.cpu().numpy()
t0 = t[t > 0].min()
mma = t[0][t[0] > 0] - t0
e0 = t[1][t[1] > 0] - t0
ee = e0[: (len(e0) // 4) * 4].reshape(-1, 4)
mm = mma[: (len(mma) // 2) * 2].reshape(-1, 2)
epi = (ee[:, 2] - ee[:, 0])[1:17]
sigt = (ee[:, 3] - ee[:, 2])[1:17]
ph = np.array([mm[k + k // 8][1] - mm[k + k // 8][0] for k in range(1, 17)])
per = [int(mm[9 * (k + 1)][0] - mm[9 * k][0]) for k in range((len(mm) - 1) // 9)]
print(f"save={saving}: kernel {ev[0].elapsed_time(ev[1])*1e3:.0f} us | "
      f"epilogue {epi.mean():.0f} signal {sigt.mean():.0f} MMA-phase {ph.mean():.0f} (min {ph.min()} max {ph.max()}) | iteration {np.mean(per):.0f} cycles")
