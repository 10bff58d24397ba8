"""juqbox_b200: B200-native objective + adjoint-gradient path of Juqbox (see DESIGN.md)."""
from .params import (objparams, lsolver_object, wmatsetup, orig_wmatsetup, setup_rotmatrices, initial_cond,
                     calculate_timestep, estimate_Neumann, assign_thresholds, assign_thresholds_freq,
                     change_target, tikhonov_pen, tikhonov_grad, NEUMANN_SOLVER, JACOBI_SOLVER, Stormer_Verlet)
from . import configs
from .api import (Working_Arrays, traceobjgrad, traceobjgrad_batch, forward_sensitivity, final_state, state_history, eval_forward, evalctrl, eval_f_g_grad, eval_f_par, eval_grad_f_par,
                  eval_g_par, eval_jac_g_par)
from .optimize import setup_ipopt_problem, run_optimizer, run_optimizer_multistart
