"""towr_b200 — B200-native batched evaluation of towr's NLP (constraints, cost,
sparse Jacobian values) behind a C ABI.  See DESIGN.md / INTEGRATION.md."""
from . import _capi as capi
from ._capi import (ANYMAL, BIPED, BLOCK, CHIMNEY, CHIMNEY_LR, EVAL_ALL, EVAL_COST, EVAL_G, EVAL_JAC, FLAT, GAP,
                    GO1, GRID_CSV, GRID_MAP, HYQ, MONOPED, SLOPE, STAIRS, TowrB200Error)
from .formulation import (BaseState, Batch, GaitGenerator, NlpFormulation, Parameters, Problem, robot_info,
                          pack_polygons, terrain_height)
from .configs import make_formulation, CONFIGS
from .sharding import shard_range, gather_cost_status
