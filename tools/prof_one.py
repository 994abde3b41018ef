import sys, os
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ggllm_cpp_b200.binding as b
b.init(0); L = b.lib()
K, M, mode = int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3])
Ws = [b.Weight(12, K, M, seed=i + 1) for i in range(4)]
x = b.DevBuf(src=np.random.default_rng(0).standard_normal(K).astype(np.float32))
yd = b.DevBuf(M * 4)
A = b.ActQ(12, K, 1); A.quantize(x.ptr)
for r in range(3):
    for w in Ws:
        if mode == 0: L.b200_mul_mat_vec_q(w.h, A.h, yd.ptr, M, 0, None, None)
        else: L.b200_mul_mat_vec_fused(w.h, x.ptr, None, None, None, None, None, yd.ptr, 0)
L.b200_synchronize()
