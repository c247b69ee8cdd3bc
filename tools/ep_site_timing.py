"""clock64() stamps of the EP site kernel (ep_sites_block_w) on one synthetic 64-site block: where the ~2100 cycles per
site go.  python tools/ep_site_timing.py  ->  profiles/r02_ep_site_timing.log"""
import ctypes as C, sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from gp_algos_b200 import _lib
h = _lib.default_handle()
st = (C.c_longlong * 897)()
for chain in (1, 10):     # 1 = reference kernel (ep_sites_block_w); 10 = warp-specialised kernel (ep_sites_block_p, branch-free scalar update): loop-top stamps only
    h.check(h.lib.gpk_debug_ep_site_timing(h.h, chain, C.addressof(st)))
    v = np.array(list(st)[:320], dtype=np.int64).reshape(64, 5)
    top, sc, dn, pub, bar = v.T
    per_site = np.diff(top)
    print(f"chain {chain}: cycles per site  median {np.median(per_site):.0f}  (k=1..8 {per_site[:8].tolist()}, k=56..63 {per_site[-8:].tolist()})")
    if chain >= 10:       # scalar warp: [top, scalar update done, results stored / barrier reached, barrier passed, next inputs formed]
        print(f"   scalar update        median {np.median(sc - top):.0f}")
        print(f"   store results        median {np.median(dn - sc):.0f}")
        print(f"   barrier              median {np.median(pub - dn):.0f}   per site k=1..8 {(pub - dn)[1:9].tolist()}  k=56..63 {(pub - dn)[56:].tolist()}")
        print(f"   next site's inputs   median {np.median(bar - pub):.0f}")
        print(f"   loop back            median {np.median(top[1:] - bar[:-1]):.0f}")
        arr = np.array(list(st)[321:577], dtype=np.int64).reshape(64, 4)      # barrier arrival: tile warps 0 / 3, helper warps 0 / 7
        lead = dn[:, None] - arr                                               # cycles before the scalar warp's arrival
        tw = np.array(list(st)[577:897], dtype=np.int64).reshape(64, 5)       # tile warp 0: [barrier k passed, post phase of k-1 done (top of k), downdate done]
        print(f"   tile warp 0: post phase (mu / diagonal / row of A) median {np.median(tw[1:, 1] - tw[:-1, 0]):.0f}, loads + downdate {np.median(tw[1:, 2] - tw[1:, 1]):.0f}, publish -> barrier {np.median(arr[1:, 0] - tw[1:, 2]):.0f}, barrier {np.median(tw[1:, 0] - arr[1:, 0]):.0f}")
        for name, col_ in (("tile warp 0", 0), ("tile warp 3 (finishes the site's outputs)", 1), ("helper warp 0", 2), ("helper warp 7", 3)):
            print(f"   {name:45s} arrives {np.median(lead[2:, col_]):.0f} cycles before the scalar warp (k=2..9 {lead[2:10, col_].tolist()}, k=56..63 {lead[56:, col_].tolist()})")
        continue
    print(f"   scalar update        median {np.median(sc - top):.0f}")
    print(f"   rank-1 tile downdate median {np.median(dn - sc):.0f}")
    print(f"   mu / A row / publish median {np.median(pub - dn):.0f}")
    print(f"   barrier              median {np.median(bar - pub):.0f}   (late sites, helper-bound? k=60: {int((bar - pub)[60])})")
    print(f"   barrier -> next top  median {np.median(top[1:] - bar[:-1]):.0f}")
print(f"unstamped default kernel (ep_sites_block_p), one 64-site block, CUDA events: {st[320] / 1e3:.1f} us")
