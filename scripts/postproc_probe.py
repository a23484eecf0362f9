"""Runs every kernel outside the per-iterate path once at B = 4096 (config 2 / config 4 recipes) so that an ncu launch list
(--metrics gpu__time_duration.sum) shows their durations: TrajectoryKernel, InitialGuessKernel, FootstepPlanKernel, NearestPlaneKernel,
GoalInstanceKernel, CostKernel, LinearEqualityKernel, SoftConstraintKernel, LmStepKernel.
    ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file out.csv python scripts/postproc_probe.py"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import towr_b200 as tb
from towr_b200 import capi
from towr_b200.configs import synthetic_iterates_fast
from towr_b200.solver import BatchedLevenbergMarquardt

B = 4096
for name in ("anymal_trot_block", "hyq_gallop_gap"):
    f = tb.make_formulation(name)
    f.params_.costs_ = [(capi.COST_FORCES, 1.0)]
    p = tb.Problem(f.to_spec())
    X = synthetic_iterates_fast(p, B, seed=3)
    bt = p.batch(B)
    bt.eval_host(X, flags=capi.EVAL_ALL)                       # CostKernel
    bt.sample_trajectory(X, 0.01)                              # TrajectoryKernel (201 samples)
    bt.initial_guesses(X, np.linspace(0.0, 2.0, 41))           # InitialGuessKernel
    plan = bt.footstep_plans(X, 2.0)                           # FootstepPlanKernel
    polys = [np.array([[-1.0, -1.0], [4.0, -1.0], [4.0, 1.0], [-1.0, 1.0], [-1.0, -1.0]]), np.array([[0.5, -0.5], [1.5, -0.5], [1.5, 0.5], [0.5, 0.5], [0.5, -0.5]])]
    bt.footstep_contact_sets(X, 2.0, polys)                    # NearestPlaneKernel
    goals = np.column_stack([np.full(B, 1.5), np.zeros(B), np.full(B, 0.5), np.zeros(B), np.zeros(B), np.zeros(B)])
    bt.goal_instances_device(torch.from_numpy(goals).cuda())   # GoalInstanceKernel
    bt.soft_constraint("dynamic")                              # SoftConstraintKernel
    if name == "anymal_trot_block":
        lm = BatchedLevenbergMarquardt(bt)
        lm.run(torch.from_numpy(X).cuda(), 2)                  # LmStepKernel
    torch.cuda.synchronize()
print("done")
