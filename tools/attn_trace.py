"""Timeline of ONE attention CTA from the instrumented build (python -m tpdm_b200.build --variant trace TPDM_ATTN_TRACE):
clock64() stamps of softmax warp 4 (keys [0,64) of every tile) and of the two MMA-issuing warps, per 128-key tile, plus CTA-level
stamps of an early and a late CTA.  Run on the GPU box:
    TPDM_B200_LIB=tpdm_b200/_build/libtpdm_trace.so python tools/attn_trace.py"""
import ctypes as C
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tpdm_b200 import _lib as L  # noqa: E402

lib = L.load()
Bt, S, H, d = 2, 4429, 24, 64
qkv = torch.randn(Bt, S, 3, H, d, device="cuda").bfloat16().contiguous()
out = torch.zeros(Bt, S, H, d, device="cuda", dtype=torch.bfloat16)
for _ in range(3):
    L.check(lib.tpdm_joint_attention(L.ptr(qkv), L.ptr(out), Bt, S, H, 64, d, 0, None))
torch.cuda.synchronize()
buf = (C.c_longlong * (3 * 2048))()
lib.tpdm_attn_trace_read.argtypes = [C.POINTER(C.c_longlong), C.c_int]
assert lib.tpdm_attn_trace_read(buf, 3 * 2048) == 0
sm, qk, pv = ([buf[r * 2048 + i] for i in range(2048)] for r in range(3))
n_kv = (S + 127) // 128
names = ["wait s_full", "checkpoint + ld chunks 0-1", "chunk 0 (pv_done wait, st)", "chunk 1 + s_free", "chunks 2-3 + p_full"]
print("softmax warp 4 of one CTA, cycles per phase of a 128-key tile (period = top(j+1) - top(j))")
tot = [0.0] * 6
cnt = 0
for j in range(4, n_kv - 2):
    e = sm[8 * j: 8 * j + 6]
    nxt = sm[8 * (j + 1)]
    if 0 in e or nxt == 0:
        continue
    ph = [e[k + 1] - e[k] for k in range(5)] + [nxt - e[0]]
    for k in range(6):
        tot[k] += ph[k]
    cnt += 1
    if 10 <= j < 16:
        print(f"  j={j:3d}: " + "  ".join(f"{names[k]}={ph[k]:4d}" for k in range(5)) + f"  | period={ph[5]}")
print("mean over", cnt, "tiles: " + "  ".join(f"{names[k]}={tot[k] / cnt:6.1f}" for k in range(5)) + f"  | period={tot[5] / cnt:.1f}")
for role, name, arr in ((1, "QK issuer", qk), (2, "PV issuer", pv)):
    w = s_ = c = 0.0
    for j in range(4, n_kv - 2):
        a = arr[4 * j: 4 * j + 3]
        if 0 in a:
            continue
        w += a[1] - a[0]
        s_ += a[2] - a[1]
        c += 1
    print(f"{name}: mean wait {w / c:.1f} cycles, issue+commit {s_ / c:.1f} cycles per 128-key tile")
lag_s = [sm[8 * j + 1] - qk[4 * j + 2] for j in range(4, n_kv - 2) if sm[8 * j + 1] and qk[4 * j + 2]]
print(f"S(j) issued -> softmax(j) past its wait: mean {sum(lag_s) / len(lag_s):.0f} cycles (min {min(lag_s)}, max {max(lag_s)})")

cbuf = (C.c_longlong * 32)()
if hasattr(lib, "tpdm_attn_cta_trace_read") and lib.tpdm_attn_cta_trace_read(cbuf) == 0:
    for c, name in ((0, "CTA (qt 5, head 3, batch 0) -- first wave"), (1, "CTA (qt 7, head 20, batch 1) -- late wave")):
        t = [cbuf[16 * c + i] for i in range(9)]
        if not t[6]:
            continue
        cyc, ns = t[6] - t[0], t[8] - t[7]
        print(f"{name}: {cyc} cycles = {ns} ns ({cyc / max(ns, 1):.3f} GHz): entry->pdl_wait {t[1] - t[0]}, TMEM alloc + sync {t[2] - t[1]}, "
              f"first score tile + its maximum {t[3] - t[2]}, {n_kv} key tiles {t[4] - t[3]} ({(t[4] - t[3]) / n_kv:.0f} each), "
              f"last P V + O store {t[5] - t[4]}, exit {t[6] - t[5]}")
