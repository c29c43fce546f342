import os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from f110_gymnasium_ros2_jazzy_b200 import ShapedReward
from tests import helpers as H
g = H.reward_recording()
N = 8192
obs = torch.from_numpy(g['obs'][np.arange(N) % len(g['obs'])]).cuda().contiguous()
rw = ShapedReward(N, g['centerline'], w_prog=5.0, alive_bonus=0.5, grace_steps_wall=25, grace_steps_opp=175, wall_quantile=0.10)
for _ in range(30): rw(obs)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(20): rw(obs)
e1.record(); torch.cuda.synchronize()
print("reward kernel %d envs: %.4f ms" % (N, e0.elapsed_time(e1) / 20))
