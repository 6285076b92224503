import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mujoco_reinforcement_learning_b200 import _lib
lib = _lib.load()
for (M, N, K) in [(65536, 128, 17)]:
    print("shape", M, N, K, file=sys.stderr, flush=True)
    A = torch.randn(M, K, device="cuda"); B = torch.randn(N, K, device="cuda"); C = torch.zeros(M, N, device="cuda")
    for i in range(2):
        _lib.check(lib.b200ppo_debug_tc_gemm(_lib.ptr(A), _lib.ptr(B), _lib.ptr(C), M, N, K, 0, 0, -2, 1, _lib.stream_ptr()))
