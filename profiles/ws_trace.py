import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mujoco_reinforcement_learning_b200 import _lib
lib = _lib.load()
for (M, N, K) in [(32768, 256, 376), (32768, 256, 256)]:
    A = torch.randn(M, K, device="cuda"); B = torch.randn(N, K, device="cuda"); C = torch.zeros(M, N, device="cuda")
    for i in range(2):
        _lib.check(lib.b200ppo_debug_tc_gemm(_lib.ptr(A), _lib.ptr(B), _lib.ptr(C), M, N, K, 0, 0, -2, 1, _lib.stream_ptr()))
