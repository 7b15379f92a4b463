"""The fp64 linear residual of one Newton step's update, with and without the multigrid's single-precision companion
planes (pnp_tune "mg_f32_min_rows": -1 the default rule, 1e30 none).  bench.py's workload: pore refined `levels` times
(default 7, 141 M dofs), the state of its nested iteration, one step (BiCGSTAB + V(2,2)).  For each rule it prints the
linear iterations, the line-search trials and ||J(u_s) d - F(u_s)|| / ||F(u_s)|| for the update d = u_s - u, J the exact
fp64 Jacobian: the step's stopping criterion asks for at most min_linear_reduction.
  python scripts/f32_step_residual.py [levels]
"""
import json
import os
import sys

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from test_gpu_f32_smoother import OFF, newton_step_both_rules  # noqa: E402

levels = int(sys.argv[1]) if len(sys.argv) > 1 else 7
out, mlr = newton_step_both_rules(levels, (-1, OFF))
for rule, r in out.items():
    print(json.dumps({"levels": levels, "mg_f32_min_rows": rule, "linear_iterations": r["its"], "line_search_trials": r["trials"],
                      "spmv_fine_gb": round(r["fine"] / 1e9, 2), "linear_residual": r["lin_res"], "min_linear_reduction": mlr,
                      "meets_criterion": bool(r["lin_res"] <= mlr)}), flush=True)
