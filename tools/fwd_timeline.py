"""Protocol timeline of CTA 0 of dense_fwd_tma_kernel (SM clocks), Gowalla-sized layer.  python tools/fwd_timeline.py [mess_p]"""
import ctypes as C, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from seoul_tourism_recommendation_ngcf_b200 import _lib

lib = _lib.load()
raw = C.CDLL(_lib.LIB_PATH)
raw.ngcf_debug_bwd_timeline.argtypes = [C.c_int, C.c_void_p]
dev = torch.device("cuda:0")
MESS_P = float(sys.argv[1]) if len(sys.argv) > 1 else 0.1
N, d = 70839, 64
st = torch.cuda.current_stream().cuda_stream
X = torch.randn(N, d, device=dev); S = torch.randn(N, d, device=dev); Y = torch.empty(N, d, device=dev)
W1 = torch.randn(d, d, device=dev) * 0.1; W2 = torch.randn(d, d, device=dev) * 0.1
b1 = torch.randn(d, device=dev); b2 = torch.randn(d, device=dev)
wcat = torch.empty(2 * d * d, device=dev); bias = torch.empty(d, device=dev)
lib.ngcf_pack_weights(W1.data_ptr(), b1.data_ptr(), W2.data_ptr(), b2.data_ptr(), d, d, wcat.data_ptr(), bias.data_ptr(), st)
flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
run = lambda: lib.ngcf_dense_fwd(S.data_ptr(), X.data_ptr(), N, d, d, wcat.data_ptr(), bias.data_ptr(), 0.2, None, None, MESS_P, 1, None, 0, 0, Y.data_ptr(), st)
for _ in range(3): run()
torch.cuda.synchronize()
raw.ngcf_debug_bwd_timeline(1, None)
flush.zero_(); run(); torch.cuda.synchronize()
out = np.zeros(4 * 8 * 8, dtype=np.int64)
raw.ngcf_debug_bwd_timeline(0, out.ctypes.data)
t = out.reshape(4, 8, 8); t0 = t[0, 7, 7]
print("dense_fwd_tma_kernel, CTA 0, SM cycles after the set-up barrier; kernel end =", t[1, 7, 7] - t0)
print(f"pdl_wait returned {t[0, 7, 6] - t0}; weights staged {t[0, 7, 5] - t0}")
for it in range(4):
    print(f"tile {it}: producer got raw_empty " + " ".join(str(int(t[3, it, k] - t0)) for k in range(2)) +
          " | converter " + " ".join(f"{n}={int(t[2, it, k] - t0)}" for k, n in enumerate(
              ["q0 raw_full", "q0 a_empty", "q0 done", "q1 raw_full", "q1 a_empty", "q1 done"])) +
          " | mma tmem_empty=" + str(int(t[1, it, 0] - t0)) + " a_full " + " ".join(str(int(t[1, it, 1 + k] - t0)) for k in range(4)) +
          " | epilogue " + " ".join(f"{n}={int(t[0, it, k] - t0)}" for k, n in enumerate(["wait", "tmem_full", "stored", "tmem read", "transposed"])))
