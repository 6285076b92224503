"""Gather kernel variants on the bench shape (4096 envs x 128 steps, 376-float rows): B200PPO_GATHER=tma|ldg.

Round-1 measurement (fraction of the 6547 GB/s copy peak; random permutation / identity index):
  tma (default, one bulk copy per row per lane)   0.672 / 0.761
  ldg (warp per row, float4 loads/stores)          0.658 / 0.665
  two rows per warp (removed)                      0.597 / 0.628
  two bulk copies in flight per lane (removed)     0.536 / 0.703   (halves the resident warps)
"""
import sys, torch, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
import mujoco_reinforcement_learning_b200 as pkg
m=4096*128; dev="cuda"
obs=torch.randn(m,376,device=dev); act=torch.randn(m,17,device=dev); s=torch.randn(m,device=dev)
idx=torch.randperm(m,device=dev); ident=torch.arange(m,device=dev)
by=(2*(4*376+4*17+12)+8)*m
for name,ix in (("random",idx),("identity",ident)):
    med,best=bench.cuda_time(lambda: pkg.gather_minibatch(ix,obs,act,s,s,s,check=False),20)
    print(os.environ.get("B200PPO_GATHER","tma"), name, round(med*1e3,1),"us", round(by/1e9/(med*1e-3)), "GB/s", round(by/1e9/(med*1e-3)/6547.2,3))
o=pkg.gather_minibatch(idx,obs,act,s,s,s)
assert torch.equal(o[0],obs[idx]) and torch.equal(o[1],act[idx]) and torch.equal(o[2],s[idx])
