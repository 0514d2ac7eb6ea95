"""sdp-b200: finite-horizon SDP backward induction on B200 behind the reference's recursion API.

Everything that computes lives in libsdpb200.so (hand-written sm_100a CUDA, csrc/); this package
is the host-side mirror of the reference's Java classes plus the descriptor builders.
"""
from . import _abi as abi
from ._abi import (ALLOW_CAPPED_ACTIONS, ALLOW_CLIPPED_SUCCESSORS, COST_STAFF, COST_CASH_TWO_PRODUCT, KERNEL_LEAD_COL, KERNEL_LEAD_Q2, KERNEL_LEAD_Q2M, KERNEL_COLLAPSED, KERNEL_TWO_PRODUCT_ROW, KERNEL_FUSED, KERNEL_CASH_ROW, KERNEL_CASH_TAIL, KERNEL_CASH_DIAG, COST_CASH_LOAN, COST_CASH_OD_LIMIT, COST_CASH_OD_TESTING, Q_TRUNC, KERNEL_CASH_INT, KERNEL_TILED2, KERNEL_LEAD_SLAB, COST_BACKORDER, COST_CASH_DEPOSIT, COST_CASH_OVERDRAFT, COST_CASH_XR, KERNEL_AUTO,
                   KERNEL_GENERIC, KERNEL_STAGED, KERNEL_TILED, MAX, MIN, Q_DIV, Q_LONGDIV, REC_EXPECT, REC_SURVIVAL,
                   SdpbError)
from .getpmf import (GetPmfMulti, DiscreteDistribution, GammaDist, GetPmf, NormalDist, PoissonDist, UniformIntDist,
                     clsp_inline_pmf, poisson_pmf)
from .models import (workforce_model, two_product_cash_model, ModelSpec, cash_loan_model, cash_overdraft_limit_model, cash_overdraft_testing_model,
                     cash_constraint_model, cash_leadtime_model, cash_overdraft_model,
                     cash_survival_model, cash_xr_model, inventory_model, leadtime_model)
from .recursion import (CashRecursionMultiLead, CashRecursionMultiXR, CashRecursionRounded, CashRecursionV, CashStateMultiLead, CashStateMultiXR, StaffRecursion, StaffState, Actions, CashRecursionMulti, CashStateMulti, CashLeadtimeRecursion, CashLeadtimeState, CashRecursion, CashRecursionXR,
                        CashState, CashStateXR, LeadtimeRecursion, LeadtimeRecursion2, LeadtimeState,
                        OptDirection, Recursion, RiskRecursion, RiskState, State)
from .solver import Group, Reached, Solver, TopDown, reachable_hull, solve_batch
from .simulation import CashSimulation, Simulation, generate_lh_samples
from .sampling import MRG32k3a, Sampling
from .write import WriteToCsv, WriteToExcelTxt, java_double
from . import configs
from . import parallel
