"""clock64 timeline of CTA 0 of the weights-stationary kernels on the bench shapes (debug entry point, bn = -2).

B200PPO_DEBUG_DGRAD=1 traces the dgrad epilogue instead of the forward one, B200PPO_DEBUG_RELU=1 drops the MUFU work,
B200PPO_DEBUG_TWICE=1 launches the problem twice in one group (actor + critic)."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mujoco_reinforcement_learning_b200 import _lib
lib = _lib.load()
shapes = [(32768, 256, 256), (32768, 256, 376)]
for (M, N, K) in shapes:
    print("shape", M, N, K, file=sys.stderr, flush=True)
    A = torch.randn(M, K, device="cuda"); B = torch.randn(N, K, device="cuda"); C = torch.zeros(M, N, device="cuda")
    for i in range(2):
        _lib.check(lib.b200ppo_debug_tc_gemm(_lib.ptr(A), _lib.ptr(B), _lib.ptr(C), M, N, K, 0, 0, -2, 1, _lib.stream_ptr()))
