/*
 * sdpb200.h — C-ABI of libsdpb200.so: finite-horizon stochastic dynamic programming
 * (backward induction) for the inventory models of RobinChen121/Stochastic-Inventory,
 * solved on NVIDIA B200 (sm_100a) with hand-written CUDA kernels, one launch per period.
 *
 *     V_t(s) = opt_{a in A(s)}  sum_j [ p_j * c(s,a,d_j)  (+)  (p_j * gamma) * V_{t+1}( f(s,a,d_j) ) ]
 *
 * This header is the drop-in boundary.  The reference has no FFI layer: its "operator API"
 * is the Java class surface of the recursion engines, which take Java lambdas.  A GPU cannot
 * call lambdas, so the lambdas of every in-scope reference driver are lowered to ONE
 * parameterised descriptor (`sdpb_model`); each entry point below names the Java member it
 * replaces (paths relative to the reference repository root).
 *
 *   reference (Java)                                               this library
 *   -------------------------------------------------------------  ----------------------------
 *   new Recursion(dir, pmf, A, f, c)   src/sdp/inventory/Recursion.java:49-63      sdpb_create
 *   new LeadtimeRecursion(pmf,A,f,c)   src/sdp/inventory/LeadtimeRecursion.java:28-45  sdpb_create
 *   new CashRecursion(dir,pmf,A,f,c,g) src/sdp/cash/CashRecursion.java:39-57       sdpb_create
 *   new CashLeadtimeRecursion(...)     src/sdp/cash/CashLeadtimeRecursion.java:28-46   sdpb_create
 *   new RiskRecursion(pmf,A,f,c)       src/sdp/cash/RiskRecursion.java:31-45       sdpb_create
 *   new CashRecursionXR(...)           src/sdp/cash/CashRecursionXR.java:39-57     sdpb_create
 *   getExpectedValue(state)            Recursion.java:89-163, CashRecursion.java:79-140,
 *                                      LeadtimeRecursion.java:47-75, CashLeadtimeRecursion.java:48-79,
 *                                      CashRecursionXR.java:79-125                 sdpb_solve + sdpb_value
 *   getSurvProb(state)                 CashRecursion.java:143-194, RiskRecursion.java:64-108
 *                                                                                  sdpb_solve + sdpb_value
 *   getAction(state)                   Recursion.java:165-167 (and siblings)       sdpb_value (q out)
 *   getOptTable()/getCacheActions()    Recursion.java:169-186 (and siblings)       sdpb_reach + sdpb_opt_table
 *   the same at off-grid states, steps that are not powers of two, unclamped models without a hull
 *                                      (the memo maps of Recursion.java:89-163)     sdpb_topdown_solve +
 *                                                                                  sdpb_topdown_value / _opt_table
 *   getExpectedValue(state) of any period on those memo maps                      sdpb_topdown_extend
 *   Simulation over them, solving the states a path meets (Simulation.java:62)    sdpb_topdown_simulate
 *   the lambdas A, f, c                src/capacitated/CLSPTesting.java:78-106, src/leadtime/Leadtime.java:50-81,
 *                                      src/cash/singleItem/CashConstraint.java:95-133,
 *                                      src/cash/overdraft/CashOverdraft.java:72-118,
 *                                      src/cash/overdraft/SingleProductLeadtime.java:72-119,
 *                                      src/cash/risk/cashSurvival.java:102-147,
 *                                      src/cash/singleItem/CashConstraintXR.java:71-110   sdpb_model fields
 *
 * Conventions: every function returns 0 (SDPB_OK) or a negative sdpb_status; no exceptions
 * cross the boundary; all result buffers are caller-allocated host memory unless a function
 * says "device"; a handle is not thread-safe, distinct handles are independent; calls block
 * until the result is on the host (except sdpb_solve_period_async).  There is NO CPU fallback:
 * without a CUDA device sdpb_create fails with SDPB_ERR_NO_DEVICE.
 */
#ifndef SDPB200_H
#define SDPB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDPB_ABI_VERSION 4

typedef enum sdpb_status {
    SDPB_OK = 0,
    SDPB_ERR_ARG = -1,        /* null pointer, bad enum, bad size                     */
    SDPB_ERR_OFFGRID = -2,    /* grid/pmf/step not exactly representable on the grid  */
    SDPB_ERR_NO_DEVICE = -3,  /* no CUDA device / wrong architecture                  */
    SDPB_ERR_CUDA = -4,       /* a CUDA runtime call failed (see sdpb_last_error)     */
    SDPB_ERR_STATE = -5,      /* call out of order (e.g. value before solve)          */
    SDPB_ERR_NOMEM = -6,
    SDPB_ERR_UNSOLVED = -7,   /* query of a state outside the grid (Java: NullPointerException,
                                 Recursion.java:165-167)                               */
    SDPB_ERR_PEER = -8        /* multi-GPU exchange: a peer's tables cannot be mapped, or a peer did not
                                 deliver its rows of V_t in time                         */
} sdpb_status;

/* Which immediate-value / transition lambdas the descriptor stands for. */
typedef enum sdpb_cost_kind {
    /* (a>0?K:0) + v*a + h*max(l,0) + pi*max(-l,0),  l = x + a - d   (lead_time 0)
     *                                               l = x + q1 - d  (lead_time >= 1)
     * CLSPTesting.java:89-106, CLSP.java:251-272, Leadtime.java:61-81                 */
    SDPB_COST_BACKORDER = 0,
    /* cash increment with deposit interest: CashConstraint.java:103-133,
     * cashSurvival.java:116-147                                                       */
    SDPB_COST_CASH_DEPOSIT = 1,
    /* cash increment with four-branch overdraft interest: CashOverdraft.java:80-118,
     * SingleProductLeadtime.java:82-119 (lead_time 1)                                 */
    SDPB_COST_CASH_OVERDRAFT = 2,
    /* (x, R = w + v*x) re-parameterisation, action = order-up-to level y:
     * CashConstraintXR.java:71-110 with CashRecursionXR.java:79-125                   */
    SDPB_COST_CASH_XR = 3,
    /* overdraft with one loan rate (r2) and one deposit rate on the balance after ordering, holding and
     * overhead costs: src/cash/overdraft/CashOverdraftLimit.java:70-86 */
    SDPB_COST_CASH_OD_LIMIT = 4,
    /* loan interest on the balance after revenue; the transition recomputes the cash balance itself
     * instead of adding the immediate value: src/cash/overdraft/CashOverdraftTesting.java:85-118 */
    SDPB_COST_CASH_OD_TESTING = 5,
    /* deposit interest on max(w - v a, 0), loan interest (r2) on max(v a - w, 0), no holding cost in
     * the last period: src/cash/overdraft/TestPaper.java:82-93 */
    SDPB_COST_CASH_LOAN = 6,
    /* two products sharing one cash account, state (inv1, inv2, cash), action pairs (Q1, Q2) limited
     * by cash, revenue on what is sold, salvage in the last period:
     * src/cash/multiItem/MultiItemCash.java:69-117 with src/sdp/cash/multiItem/CashRecursionMulti.java:81-116
     * (MAX only, an action replaces the incumbent only if better by more than `tie_tolerance`). */
    SDPB_COST_CASH_TWO_PRODUCT = 7,
    /* workforce planning: state = staff on hand, action = hires, random turnover whose pmf depends on the
     * hire-up-to level y = x + a (SURVEY.md §8(f) rank 4):
     * src/workforce/WorkforcePlanning.java:71-104 with src/workforce/StaffRecursion.java:81-121 (MIN).
     * c = (a>0?K:0) + v*a + salary*(y-j) + (y-j > minStaff_t ? 0 : penalty*(minStaff_t - (y-j))). */
    SDPB_COST_STAFF = 8
} sdpb_cost_kind;

typedef enum sdpb_recursion {
    SDPB_REC_EXPECT = 0,   /* getExpectedValue: s += p*c; s += (p*gamma)*V'            */
    SDPB_REC_SURVIVAL = 1  /* getSurvProb: terminal 1[w + c >= 0]; continuation 0 if w' < 0,
                              RiskRecursion.java:73-104, CashRecursion.java:152-185   */
} sdpb_recursion;

typedef enum sdpb_direction { SDPB_MIN = 0, SDPB_MAX = 1 } sdpb_direction;

/* Cash quantiser applied after the cash clamp (SURVEY Appendix B).
 *   kk = Math.round(w * q_mul)                 (Java round-half-up to long)
 *   SDPB_Q_DIV      w' = (double)kk / q_div            e.g. round(w*10)/10.0
 *   SDPB_Q_LONGDIV  w' = (double)(kk / (long)q_div)    e.g. round(w*10)/10  (long division)
 *   SDPB_Q_TRUNC    w' = (double)(int) w, preceded from period q_from_period on (t >= q_from_period > 0) by
 *                   w = Math.round(w * q_mul) / q_div     (TestPaper.java:107-109: t > 2, 1e-4) */
typedef enum sdpb_quantiser { SDPB_Q_DIV = 0, SDPB_Q_LONGDIV = 1, SDPB_Q_TRUNC = 2 } sdpb_quantiser;

enum sdpb_flags {
    SDPB_F_CLAMP_INV = 1u << 0,        /* x' = clamp(x', inv_min, inv_max), upper clamp first
                                          (CLSPTesting.java:91-92); off for Leadtime.java:65-66 */
    SDPB_F_LOST_SALES = 1u << 1,       /* x' = max(0, .) before the clamp (CashConstraint.java:124) */
    SDPB_F_GY_MODE = 1u << 2,          /* period 1 is the "no order" G(y) pass, CLSPforDraw.java:147-170 */
    SDPB_F_NO_ORDER_LAST = 1u << 3,    /* A(s) = {0} when t == T (SingleProductLeadtime.java:74-75) */
    SDPB_F_CASH_LIMITED_ACTIONS = 1u << 4 /* |A(s)|-1 = (int)min(maxQ, max(0,(w - reserve_t)/v_t))
                                          (CashConstraint.java:96-99, cashSurvival.java:103-110) */
};

/*
 * The model descriptor.  All pointers are caller-owned and are copied by sdpb_create.
 * Arithmetic is IEEE-754 double, evaluated in the order written in the cited Java lines,
 * never contracted into FMA (Java has no fused multiply-add).
 */
typedef struct sdpb_model {
    uint32_t struct_size;   /* = sizeof(sdpb_model); ABI guard */
    int32_t  cost_kind;     /* sdpb_cost_kind */
    int32_t  recursion;     /* sdpb_recursion */
    int32_t  direction;     /* sdpb_direction */
    int32_t  T;             /* horizon = pmf.length */
    int32_t  lead_time;     /* 0, 1 (LeadtimeState, CashLeadtimeState) or 2 (synthetic C4) */
    uint32_t flags;         /* sdpb_flags */
    int32_t  max_order_idx; /* actions are a_i = i*step, i = 0..max_order_idx (order-up-to offset for XR) */
    double   gamma;         /* discount factor; classes without one use 1.0 (p*1.0 == p exactly) */

    /* demand pmf, GetPmf.getpmf() layout flattened: period t (0-based) owns
     * entries [off_t, off_t + pmf_len[t]), off_t = sum of earlier lengths. */
    const int32_t* pmf_len; /* [T] */
    const double*  pmf_d;   /* demand values  pmf[t][j][0] */
    const double*  pmf_p;   /* probabilities  pmf[t][j][1] */

    /* inventory axis: x_i = inv_min + i*step, i = 0..(inv_max-inv_min)/step */
    double inv_min, inv_max, step;

    /* cash axis (cash kinds only): clamp to [cash_min, cash_max], then quantise */
    double  cash_min, cash_max;
    int32_t quantiser;      /* sdpb_quantiser */
    int32_t q_from_period;  /* SDPB_Q_TRUNC only; 0 = never round */
    double  q_mul, q_div;

    /* cost parameters (unused ones are ignored) */
    double fixed_cost;      /* K */
    double vari_cost;       /* v   (per-period override: vari_cost_t) */
    double hold_cost;       /* h */
    double penalty_cost;    /* backorder pi; CASH_DEPOSIT: penalty on negative end cash */
    double price;           /* per-period override: price_t */
    double salvage;         /* applied to max(l,0) when t == T */
    double deposit_rate;    /* CASH_DEPOSIT: (w - K - v a) * (1 + deposit_rate) */
    double overhead_rate;   /* CASH_DEPOSIT: (1 - overhead_rate) * revenue */
    double overhead;        /* per-period override: overhead_t */
    double r0, r2, r3, od_limit, interest_free; /* CASH_OVERDRAFT, CashOverdraft.java:88-95 */
    const double* price_t;      /* [T] or NULL */
    const double* vari_cost_t;  /* [T] or NULL */
    const double* overhead_t;   /* [T] or NULL */
    const double* reserve_t;    /* [T] or NULL (= 0): cash kept back in the action bound,
                                   (int)min(maxQ, max(0, ((w - reserve_t) - reserve2) / v_t));
                                   overhead then K in CashConstraint.java:98, 0 in cashSurvival.java:105 */
    double reserve2;

    /* second product (SDPB_COST_CASH_TWO_PRODUCT only).  Product 1 uses price / vari_cost / salvage and
     * pmf_d; both inventories live on the inventory axis; actions are pairs (i, j), 0 <= i, j <=
     * max_order_idx, scanned i-major (MultiItemCash.java:69-79) and feasible while
     * v1*i + v2*j < cash + 0.1.  sdpb_value / sdpb_period_tables report the pair as i*(max_order_idx+1)+j. */
    double price2, vari_cost2, salvage2;
    const double* pmf_d2;   /* second product's demand of every pmf row (same layout as pmf_d) */
    double tie_tolerance;   /* 0.1 in CashRecursionMulti.java:108; 0 = plain strict compare */

    /* action-dependent demand (SDPB_COST_STAFF only): for period t and hire-up-to level y (grid index
     * 0..n_inv-1; levels beyond the grid use the last row, StaffRecursion.java:95-96) the turnover j has
     * probability apmf_p[off(t,y) + j], j = 0..apmf_len[t*n_inv + y]-1, rows concatenated in (t, y) order.
     * hold_cost is the salary, penalty_cost the unit penalty, min_level_t the required staff per period.
     * pmf_len / pmf_d / pmf_p are ignored (pass one dummy row per period). */
    const int32_t* apmf_len;
    const double*  apmf_p;
    const double*  min_level_t;

    /* Terminal boundary function (FinalCash.BoundaryFuncton, src/sdp/inventory/FinalCash.java:16-18, consumed
     * at src/sdp/cash/multiItem/CashRecursionV.java:125-128: a state of period T+1 is worth b(s)).  NULL =
     * the engines without one: no continuation in period T (Recursion.java:140 `if (n < T)`).  Otherwise
     * n_states doubles in the library's state order (sdpb_state_of_index gives the coordinates of entry i),
     * V_{T+1}(s) = terminal_value[index of s]: period T then accumulates (p*gamma) * V_{T+1}(f(s,a,d)) like every
     * other period.  Copied by sdpb_create.  Not available with SDPB_REC_SURVIVAL (its terminal rule is the
     * indicator of RiskRecursion.java:80-84). */
    const double* terminal_value;
} sdpb_model;

typedef enum sdpb_kernel_choice {
    SDPB_KERNEL_AUTO = 0,     /* fastest bit-exact kernel available for the model */
    SDPB_KERNEL_GENERIC = 1,  /* always the generic per-(s,a,d) kernel */
    SDPB_KERNEL_TILED = 2,    /* shared-memory kernel: tiled for lead_time 0; for backorder lead-time models the
                                 column kernel (else slab, else staged); for integer-exact cash models the
                                 integer cash kernels; error if the model has none */
    SDPB_KERNEL_STAGED = 3,   /* warp-per-state staged kernel for backorder lead-time models (as a request:
                                 skip the all-actions-in-thread, column and slab kernels) */
    SDPB_KERNEL_CASH_INT = 4, /* integer-exact cash kernel (as a request: skip the diagonal-window variant) */
    SDPB_KERNEL_CASH_DIAG = 8,/* reported only: integer-exact cash kernel with a register window along the
                                 (1, -price) diagonal; the last period runs on SDPB_KERNEL_CASH_INT */
    SDPB_KERNEL_LEAD_SLAB = 6,/* shared-memory slab kernel for backorder lead-time models (as a request: skip
                                 the column kernel) */
    SDPB_KERNEL_LEAD_COL = 7, /* thread-per-successor-column kernel for backorder lead-time models (as a request:
                                 skip the all-actions-in-thread kernel) */
    SDPB_KERNEL_LEAD_Q2 = 9,  /* lead time 2: a thread owns 8 preQ1 levels of one (x, preQ2), walks every action
                                 itself and reads V_{t+1} through a transposed copy; AUTO picks it when the
                                 model is not folded */
    SDPB_KERNEL_LEAD_Q2M = 14,/* reported only: SDPB_KERNEL_LEAD_Q2 with the products p*(fixed + variable + level cost) formed once
                                 per CTA and action in shared memory and two preQ2 columns per thread; chosen on large grids
                                 (no action slices); request SDPB_KERNEL_LEAD_Q2 to get either */
    SDPB_KERNEL_COLLAPSED = 15,/* REQUEST ONLY, never chosen by AUTO, NOT bit-identical to the reference: the 1-D inventory family
                                 solved as G(y) = sum_j p_j L(y-d_j) + p_j gamma V(y-d_j) per order-up-to level and
                                 V(x) = opt_a ordering cost(a) + G(x+a) per state -- D operations per level and A per
                                 state instead of A*D per state.  Values agree with the exact kernels to ~1e-13 relative
                                 (the rounding of the demand sum and 1 - sum_j p_j); the optimal action can move between
                                 actions whose values are that close.  Unsharded handles, no G(y) pass, no
                                 SDPB_F_NO_ORDER_LAST; sdpb_create fails with SDPB_ERR_ARG otherwise */
    SDPB_KERNEL_TWO_PRODUCT_ROW = 10, /* reported only: two-product kernel that shares the cash-independent terms
                                         of an (action, demand) pair across a row of cash levels (integer prices) */
    SDPB_KERNEL_CASH_ROW = 12,/* cash-constraint kind on any cash grid; a CTA is one inventory level x 128 cash levels and
                                 shares the cash-independent terms of each (action, demand).  As a request: skip
                                 SDPB_KERNEL_CASH_TAIL (integer-exact models still run the integer cash kernels) */
    SDPB_KERNEL_CASH_TAIL = 13,/* reported only: cash-constraint and overdraft kinds on any rounding cash grid; row-shared terms as
                                 SDPB_KERNEL_CASH_ROW, with the cash clamp applied to the rounded integer (as a request,
                                 SDPB_KERNEL_CASH_ROW skips it) */
    SDPB_KERNEL_FUSED = 11,   /* the whole horizon of a small 1-D inventory model in one cooperative launch (one CTA
                                 per SM, grid-wide barrier between periods); sdpb_solve / sdpb_solve_async only;
                                 AUTO picks it when the grid has at most 64 states per SM */
    SDPB_KERNEL_TILED2 = 5    /* 2-D register-tile variant of the tiled kernel: chosen automatically for
                                 large grids; as a request it forces the variant wherever it applies */
} sdpb_kernel_choice;

typedef struct sdpb_options {
    uint32_t struct_size;  /* = sizeof(sdpb_options) */
    int32_t  device;       /* CUDA ordinal; -1 = current device */
    int32_t  shard_rank;   /* this handle computes states [lo,hi) of rank r of n contiguous blocks */
    int32_t  shard_count;  /* 1 = whole grid */
    int32_t  kernel;       /* sdpb_kernel_choice */
    int32_t  dedup;        /* 1 = states that provably share (c,f) for every (a,d) are solved once
                              and broadcast (exact; lead-time kinds). 0 = brute force per state. */
    void*    stream;       /* cudaStream_t to launch on; NULL = a stream owned by the handle */
    uint32_t allow;        /* sdpb_allow bits: dense-grid artefacts sdpb_reach reports as SDPB_ERR_OFFGRID unless allowed */
    int32_t  strict_cash_bounds; /* 1: sdpb_reach also fails when a state the reference would visit has its successor cash
                              clamped at cash_min / cash_max (the clamp is part of the reference lambdas,
                              CashConstraint.java:128-129, so this is off by default) */
    int32_t  profile;      /* 1: a sharded solve records CUDA events around every period's kernels, pushes and
                              waits (sdpb_period_profile) */
    int32_t  reserved;
} sdpb_options;

/* A dense grid solves EVERY grid state, the reference only the states it reaches from the initial state.
 * Two artefacts of the dense grid are therefore harmless as long as no reached state is touched by them, and
 * wrong answers otherwise; sdpb_reach checks exactly that and fails with SDPB_ERR_OFFGRID unless allowed here:
 *   SDPB_ALLOW_CLIPPED_SUCCESSORS  a reached (state, action, demand) whose successor inventory lies outside
 *                                  [inv_min, inv_max] although the model does not clamp (SDPB_F_CLAMP_INV off,
 *                                  Leadtime.java:65-66): the kernels fold it onto the boundary row
 *   SDPB_ALLOW_CAPPED_ACTIONS      a reached state of the XR kind whose order-up-to range
 *                                  (CashConstraintXR.java:71-75, uncapped) is longer than max_order_idx + 1 */
enum sdpb_allow { SDPB_ALLOW_CLIPPED_SUCCESSORS = 1u << 0, SDPB_ALLOW_CAPPED_ACTIONS = 1u << 1 };

typedef struct sdpb_grid {
    int32_t ndim;          /* API state vector length: 1 + has_cash + lead_time */
    int32_t n_inv, n_cash, n_q; /* axis sizes (n_cash = 1 / n_q = 1 when absent) */
    int64_t n_states;      /* dense states per period */
    int64_t shard_lo, shard_hi; /* flattened range owned by this handle */
    int32_t n_actions;     /* max_order_idx + 1 */
    int32_t T;
    int64_t cash_k_min;    /* integer cash index of the lowest cash point */
    int64_t window_lo, window_hi; /* flattened range of V_t this handle holds in device memory: the whole grid when
                              unsharded, else the rows its kernels can read (sdpb_shard_reads) plus a guard margin */
    int64_t device_bytes;  /* bytes of device memory the handle allocated */
} sdpb_grid;

typedef struct sdpb_stats {
    double  evals;          /* sum_t sum_{s in shard} |A_t(s)| * D_t  (feasible actions only) */
    double  solve_ms;       /* device time of the last sdpb_solve (CUDA events) */
    double  kernel_ms;      /* of which inside backward-induction kernels */
    int32_t launches;       /* backward-induction kernel launches in the last solve */
    int32_t kernel_used;    /* sdpb_kernel_choice actually run */
    double  fp64_ops;       /* fp64 add/mul/min/max instructions the kernels executed, by construction */
    double  evals_executed; /* = evals unless dedup folded identical states together */
    /* what the last sdpb_reach saw at states the reference would visit (see sdpb_allow) */
    double  clipped_successors; /* (s,a,d) triples whose successor inventory left the grid of an unclamped model */
    double  capped_action_sets; /* XR states whose order-up-to range was cut at max_order_idx */
    double  cash_bound_hits;    /* (s,a,d) triples whose successor cash was clamped at cash_min / cash_max */
    double  exchange_ms;        /* sharded solve with sdpb_peer_attach: device time between the end of a period's
                                   kernels and the arrival of every peer's rows, summed over periods (profile = 1) */
} sdpb_stats;

typedef struct sdpb_handle sdpb_handle;

int sdpb_abi_version(void);
/* sizeof(sdpb_model) / sizeof(sdpb_options) as compiled into the library: lets a foreign-function
 * binding (Panama FFM StructLayout, ctypes.Structure) verify its layout before the first call. */
size_t sdpb_sizeof_model(void);
size_t sdpb_sizeof_options(void);
size_t sdpb_sizeof_grid(void);
size_t sdpb_sizeof_stats(void);

/* Build a solver for `m` on one GPU (opt may be NULL).  Validates that the grid is exact. */
int sdpb_create(const sdpb_model* m, const sdpb_options* opt, sdpb_handle** out);
void sdpb_destroy(sdpb_handle* h);
const char* sdpb_last_error(const sdpb_handle* h); /* h may be NULL: last create error */

int sdpb_grid_info(const sdpb_handle* h, sdpb_grid* g);
/* Multi-GPU: the contiguous range [lo, hi) of flattened V_{t+1} indices the kernels of this shard may read in
 * any period (its own band of inventory rows widened by the largest order and the largest demand, plus the
 * zero row for lost-sales clamps).  Ranks exchange only these rows instead of all-gathering V_t. */
int sdpb_shard_reads(const sdpb_handle* h, int64_t* lo, int64_t* hi);

/* Backward induction over periods T..1 for this handle's shard (whole grid when unsharded). */
int sdpb_solve(sdpb_handle* h);
/* sdpb_solve without the final synchronisation: every period is enqueued on the handle's stream and the
 * call returns.  From the second solve of a handle on, the T launches are replayed as one CUDA graph
 * (the per-period launch latency dominates small grids such as C1/C2). */
int sdpb_solve_async(sdpb_handle* h);
/* One period (1-based), asynchronous on the handle's stream.  For a sharded grid the caller
 * all-gathers the V_t device buffer (sdpb_device_tables) across ranks before period t-1. */
int sdpb_solve_period_async(sdpb_handle* h, int period);
int sdpb_sync(sdpb_handle* h);

/* getExpectedValue + getAction for `n` states of one period.  `states` is n*ndim doubles in the
 * reference constructor order: (inv) | (inv, preQ[, preQ2]) | (inv, cash) | (inv, cash, preQ).
 * v and q may be NULL.  q is the order quantity (order-up-to level for XR), as a double. */
int sdpb_value(sdpb_handle* h, int period, const double* states, int n, double* v, double* q);

/* Whole-grid tables of one period in the library's state order (inv outermost, then preQ.., cash
 * innermost); V and Q are n_states doubles each, either may be NULL.  Plain host pointers; if they
 * point into page-locked memory (cudaHostAlloc / cudaHostRegister) the copies run at PCIe speed
 * (160 MB in 3 ms instead of 40-70 ms from pageable memory, profiles/r01_bench_n1.json). */
int sdpb_period_tables(sdpb_handle* h, int period, double* V, double* Q);
/* Device pointers: V_t as double[n_states], action index as int32[n_states]. */
int sdpb_device_tables(sdpb_handle* h, int period, void** dV, void** dQidx);
/* Grid coordinates of flattened state `idx` as API-order doubles (ndim of them). */
int sdpb_state_of_index(const sdpb_handle* h, int64_t idx, double* state);

/* Forward reachability from `n` period-1 states through every feasible action and demand (what
 * the reference's top-down memoisation visits), then the getOptTable() rows
 * [t, state dims..., Q*] sorted by (t, state dims).  Call sdpb_opt_table with rows == NULL to get the count. */
int sdpb_reach(sdpb_handle* h, const double* init_states, int n);
int sdpb_opt_table(sdpb_handle* h, double* rows, size_t* nrows);

int sdpb_stats_get(const sdpb_handle* h, sdpb_stats* s);

/* Policy roll-out over caller-supplied demand sample paths — the loop of
 * Simulation.simulateSDPGivenSamplNum (src/sdp/inventory/Simulation.java:53-74) and
 * CashSimulation.simulateSDPGivenSamplNum (src/sdp/cash/CashSimulation.java:85-118):
 *     for each path i:  state = init;  sum = 0
 *         for t = 1..T:  Q = getAction(state);  d = Math.round(samples[i][t-1])
 *                        sum += Math.pow(discount, t-1) * immediateValue(state, Q, d)
 *                        state = stateTransition(state, Q, d)
 *     values[i] = sum
 * `samples` is n*T doubles, row-major (what Sampling.generateLHSamples returns; the host keeps drawing
 * them — the reference draws with Math.random(), so its own numbers are not reproducible).  One thread
 * per path, same device lambdas as the solve.  `values` receives the n sums; averaging (and adding
 * iniCash, CashSimulation.java:115) is left to the caller.  Needs a solved, unsharded handle. */
int sdpb_simulate(sdpb_handle* h, const double* init_state, const double* samples, int n, double discount,
                  double* values);

/* Evaluate the descriptor's lambdas on the device for `n` (state, action, demand) triples of one
 * period, with the same device code the solve uses: c = immediateValue(s,a,d), next = stateTransition
 * (API-order state of period+1; clipped to the grid when the model does not clamp), n_actions =
 * |getFeasibleAction(s)|.  Lets a host facade spot-check a descriptor against the user's lambdas
 * before trusting it (a mismatch would otherwise be silent).  action_idx[i] is the action's index. */
int sdpb_eval_triples(sdpb_handle* h, int period, const double* states, const int32_t* action_idx,
                      const double* demand, int n, double* c, double* next_states, int32_t* n_actions);

/* Roofline denominators of this path, measured on `device` with CUDA events (best of 5):
 *   nofma_tops  non-fused fp64 instruction rate, DADD/DMUL mix, in 1e12 instructions/s
 *   fma_tflops  fused fp64 rate in TFLOP/s (2 flops per DFMA) — for context, the kernels cannot use it
 *   lds_gbs     shared-memory LDS.128 bandwidth, GB/s
 * Any pointer may be NULL. */
int sdpb_microbench(int device, double* nofma_tops, double* fma_tflops, double* lds_gbs);

/* ---- grid bounds for models that do not clamp ------------------------------------------------------------------
 * Inventory interval that contains every state the reference's top-down recursion can visit from the `n`
 * period-1 states `init_states` (n * ndim doubles, API order) -- the bounds a caller must give the dense grid
 * of an unclamped model (Leadtime.java:63-67 has none: its memo map simply grows).  Interval propagation
 * through x' = x + (order or pipeline quantity in [0, max_order]) - d, d in [dmin_t, dmax_t], with the
 * lost-sales lift and the model's own clamps applied; exact for the lead-time model, a superset otherwise.
 * Pure host arithmetic: needs no device and no handle; m->inv_min / inv_max are ignored.
 * Replaces nothing in the reference (its maps are unbounded); sdpb_reach reports a grid that is too small. */
int sdpb_reachable_hull(const sdpb_model* m, const double* init_states, int n, double* inv_lo, double* inv_hi);

/* ---- multi-GPU inside the library -------------------------------------------------------------------------------
 * The state grid is cut into shard_count contiguous blocks of the flattened index (inventory outermost).  Each
 * handle holds, for every period, only the window of V_t its kernels can read and the policy of its own block.
 * After the kernels of period t every shard copies the rows of its block that a peer's window contains straight
 * into that peer's table through peer-mapped device memory (NVLink), raises a flag in the peer's memory, and waits
 * on the device for the flags of the peers it reads from before period t-1 starts: no host round trip, no
 * collective library.  Two ways to connect the shards:
 *
 *   one process, several GPUs (what a JVM host does):   sdpb_group_create / sdpb_group_solve / ...
 *   one process per GPU (torchrun, MPI):                sdpb_create with shard_rank / shard_count in every
 *       process, sdpb_peer_export -> exchange the blobs by any means (they are plain bytes) ->
 *       sdpb_peer_attach with all of them in rank order (CUDA IPC), then sdpb_solve in every process.
 *
 * Replaces: nothing in the reference (single-threaded Java); SURVEY.md section 8(e). */
#define SDPB_PEER_BLOB_BYTES 256
int sdpb_peer_export(sdpb_handle* h, void* blob /* SDPB_PEER_BLOB_BYTES */);
int sdpb_peer_attach(sdpb_handle* h, const void* blobs /* shard_count * SDPB_PEER_BLOB_BYTES, rank order */,
                     int n_blobs);
/* bytes this shard sends to / receives from its peers per period (after sdpb_peer_attach) */
int sdpb_peer_traffic(const sdpb_handle* h, int64_t* bytes_out, int64_t* bytes_in);
/* profile = 1: device milliseconds of the last sharded solve per period, three doubles each
 * (kernels, pushes to peers + flags, wait for the peers' flags), period 1 first. */
int sdpb_period_profile(const sdpb_handle* h, double* ms /* 3 * T */);
/* This shard's block of a period's tables: V and Q are (shard_hi - shard_lo) doubles each, either may be NULL. */
int sdpb_shard_tables(sdpb_handle* h, int period, double* V, double* Q);

typedef struct sdpb_group sdpb_group;
/* n shards of one model on the CUDA devices `devices[0..n-1]` of this process (an ordinal may repeat).  opt may be
 * NULL; its device / shard_rank / shard_count / stream are ignored. */
int sdpb_group_create(const sdpb_model* m, const sdpb_options* opt, const int* devices, int n, sdpb_group** out);
void sdpb_group_destroy(sdpb_group* g);
const char* sdpb_group_last_error(const sdpb_group* g);
int sdpb_group_solve(sdpb_group* g);            /* whole horizon on every shard; blocks */
sdpb_handle* sdpb_group_shard(sdpb_group* g, int rank);
/* getExpectedValue + getAction, each state answered by the shard that owns it */
int sdpb_group_value(sdpb_group* g, int period, const double* states, int n, double* v, double* q);
/* whole-grid tables of a period assembled from the shards' blocks (n_states doubles each) */
int sdpb_group_period_tables(sdpb_group* g, int period, double* V, double* Q);
/* evals / fp64_ops / launches summed over the shards, solve_ms = the slowest shard */
int sdpb_group_stats(const sdpb_group* g, sdpb_stats* s);

/* ---- many small instances at once ---------------------------------------------------------------------------------
 * The reference's drivers sweep hundreds of small instances (810 in src/capacitated/CLSPTesting.java:57-61), one
 * Recursion object each.  sdpb_solve_batch solves n independent unsharded handles of one device together: every
 * handle's periods are enqueued on its own stream, the whole batch is replayed as ONE CUDA graph from the second
 * call with the same handle list on, and the call returns when all are solved. */
int sdpb_solve_batch(sdpb_handle* const* handles, int n);

/* ---- the two-product recursions: solved over the states they REACH ---------------------------------------------------
 * The reference's own scaling wall (src/cash/overdraft/MultiProductLeadtime.java:28, "3 hour no solution").  Its
 * two-product engines keep states that a dense grid cannot hold -- a cash balance that is not rounded at all
 * (MultiProductLeadtime.java:219 is commented out), or a 201 x 201 x 10001 grid of which a run touches a sliver --
 * so sdpb_reached_solve builds, period by period, the set of states the reference's memoised recursion visits from
 * `init_state` (expand every (state, action, demand), sort, unique), then runs the backward induction over those sets
 * on the GPU; successors are found by binary search.  Same arithmetic and the same order-dependent acceptance rule
 * `value > best + tie_tolerance` as the reference.  Three engines + driver lambdas:
 *   SDPB_REACHED_MULTILEAD  new CashRecursionMultiLead(...).getExpectedValue / getAction
 *                           (src/sdp/cash/multiItem/CashRecursionMultiLead.java:54-95) with the lambdas of
 *                           src/cash/overdraft/MultiProductLeadtime.java:150-224; state (x1, x2, preQ1, preQ2, cash),
 *                           actions (i, j) in [0, q_bound)^2, tie 0.1
 *   SDPB_REACHED_MULTI_XR   new CashRecursionMultiXR(...).getExpectedValue / getAction
 *                           (src/sdp/cash/multiItem/CashRecursionMultiXR.java:61-95) with the lambdas of
 *                           src/cash/multiItem/MultiItemCashXR.java:73-126; state (x1, x2, R), actions = order-up-to
 *                           pairs (x1 + i, x2 + j), tie 0.1
 *   SDPB_REACHED_MULTI_YR   new CashRecursionV(...).getExpectedValueV / getAction
 *                           (src/sdp/cash/multiItem/CashRecursionV.java:83-131: V(x1,x2,w) = max_y Pi(y1,y2,R),
 *                           Pi = E V_{t+1}, V_{T+1} = boundFinalCash(s) = w + salvage . x) with the lambdas of
 *                           src/cash/multiItem/MultiItemYR.java:89-146; actions = affordable order-up-to pairs
 *                           (v . y < R + 0.1), tie 0.01
 *   SDPB_REACHED_CASH_ROUNDED  new CashRecursion(MAX, pmf, A, f, c, gamma).getExpectedValue / getAction
 *                           (src/sdp/cash/CashRecursion.java:79-140) with the lambdas of
 *                           src/cash/singleItem/CashConstraintTest.java:76-116: ONE product, state (x, w) with both
 *                           components rounded as Math.round(v * q) / q (q = 0.1: values such as 30.000000000000004, so
 *                           neither axis is a grid with an exact step) and an initial state that need not be rounded
 *                           (iniCash = 33); actions 0..(int) min(maxQ, max(0, (w - minCashRequired - K) / v)), strict
 *                           compare.  q_bound = maxOrderQuantity + 1; d2 / price[1] / vari_cost[1] / salvage[1] unused */
typedef enum sdpb_reached_kind { SDPB_REACHED_MULTILEAD = 0, SDPB_REACHED_MULTI_XR = 1, SDPB_REACHED_MULTI_YR = 2,
                                 SDPB_REACHED_CASH_ROUNDED = 3 } sdpb_reached_kind;

typedef struct sdpb_reached_model {
    uint32_t struct_size;      /* = sizeof(sdpb_reached_model) */
    int32_t  kind;             /* sdpb_reached_kind */
    int32_t  T;                /* horizon */
    int32_t  q_bound;          /* the action list has q_bound^2 entries, scanned first component outermost */
    int32_t  n_demands;        /* demand pairs per period */
    int32_t  reserved;
    const double* d1;          /* [T * n_demands] demand of product 1 (GetPmfMulti.getPmf(t)[j][0]) */
    const double* d2;          /* [T * n_demands] demand of product 2 */
    const double* p;           /* [T * n_demands] probabilities (GetPmfMulti.getPmf(t)[j][2]) */
    const double* overhead_t;  /* [T] (MULTILEAD; may be NULL otherwise) */
    double price[2], vari_cost[2], salvage[2];
    double r0, r1, r2, limit, interest_free;   /* MULTILEAD: deposit rate, overdraft rate, penalty rate, limit, free amount */
    double deposit_rate;                       /* MULTI_XR, MULTI_YR: depositeRate */
    double min_inv, max_inv, min_cash, max_cash;
    double gamma, tie_tolerance;               /* discount factor; 0.1 / 0.1 / 0.01 / 0 in the reference */
    double fixed_cost, hold_cost, min_cash_required, state_q;  /* CASH_ROUNDED: K, h, minCashRequired, q; deposit_rate = interestRate */
    const int32_t* n_demands_t; /* [T] demand points of each period when they differ (rows of d1 / d2 / p stay n_demands
                                   apart, the tail of a shorter period is ignored); NULL = n_demands everywhere */
} sdpb_reached_model;

/* init_state = (x1, x2, preQ1, preQ2, cash) | (x1, x2, R) | (x1, x2, cash) | (x, cash).  value = getExpectedValue(iniState);
 * action1 / action2 = getAction(iniState) (order quantities, or order-up-to levels); n_states[t-1] = states of period t
 * (may be NULL, T entries); solve_ms = device time.  Blocks.  No CPU fallback. */
int sdpb_reached_solve(const sdpb_reached_model* m, int device, const double* init_state, double* value,
                       double* action1, double* action2, int64_t* n_states, double* solve_ms);
/* The message of the last failed sdpb_reached_* call of this thread. */
const char* sdpb_reached_last_error(void);

/* A reached-state solve kept as a handle: the memo of getExpectedValue calls, every reached state queryable.
 *   States      API order, as sdpb_reached_solve takes them: kind 0 (x1, x2, preQ1, preQ2, cash), kind 1 (x1, x2, R),
 *               kind 2 (x1, x2, cash), kind 3 (x, cash).  A root (of open, extend, simulate) must have integer
 *               inventories and pipeline quantities in [0, 65535] (kind 3: x = k / state_q with such a k), otherwise
 *               SDPB_ERR_OFFGRID; a queried state that has no such form is simply not reached (SDPB_ERR_UNSOLVED).
 *               A coordinate that is not finite is SDPB_ERR_ARG.
 *   Actions     a1 / a2 as sdpb_reached_solve reports them, for every state: order quantities for kinds 0 and 3 (a2 = 0
 *               for kind 3), order-up-to levels for kinds 1 and 2.  A state without any accepted action keeps the
 *               reference's default: {0, 0} for kind 1, (x1, x2) for kind 2.
 *   Order       memo-map order (t, x1, x2, preQ1, preQ2, cash) with cash compared numerically
 *               (CashRecursionMultiLead.java:45-51); -0.0 is stored as +0.0.
 *   Extension   only the states no earlier call reached are expanded and solved, each against the merged tables of the
 *               next period, so a state's value never depends on the order of the calls.  The candidate successors of
 *               the new states of one period are expanded at once: when candidates * 16 B * 2.2 exceed the budget --
 *               the free device memory, or scratch_bytes when > 0 -- the call fails with SDPB_ERR_NOMEM naming the
 *               period.  A failed call leaves states, tables and stats exactly as they were.
 *   Stats       evals = sum_t sum_{s reached} |listed actions of s| * D_t over the life of the handle, evals_executed =
 *               evals; solve_ms (device time between events at the start and end of the call), kernel_ms (its backward
 *               pass) and launches (its backward launches) describe the latest call.  For simulate see there.
 * The handle keeps, per period, the sorted keys (16 B), V (8 B) and action index (4 B) of the reached states; the
 * candidate buffers of an extension are freed when it returns. */
typedef struct sdpb_reached sdpb_reached;
/* getExpectedValue on n >= 0 period-1 roots, one memo (the union of their visit sets); n == 0: an empty handle. */
int  sdpb_reached_open(const sdpb_reached_model* m, int device, int64_t scratch_bytes, const double* init_states, int n,
                       sdpb_reached** out);
void sdpb_reached_destroy(sdpb_reached* h);
/* value + action of n reached states of one period (v, a1, a2 may be NULL); SDPB_ERR_UNSOLVED for a state not reached */
int  sdpb_reached_value(sdpb_reached* h, int period, const double* states, int n, double* v, double* a1, double* a2);
/* getExpectedValue(state) on n states of one period 1..T; n == 0 does nothing */
int  sdpb_reached_extend(sdpb_reached* h, int period, const double* states, int n);
/* rows [t, state dims (API order)..., a1, a2] of every reached state in memo-map order; rows == NULL: *nrows = the count */
int  sdpb_reached_opt_table(sdpb_reached* h, double* rows, size_t* nrows);
int  sdpb_reached_states(const sdpb_reached* h, int64_t* n_states /* T: reached states of each period */);
int  sdpb_reached_stats(const sdpb_reached* h, sdpb_stats* s);
/* The policy rolled out over n demand sample paths, with a lazy getExpectedValue at every step (CashSimulation's loop,
 * CashSimulation.java:85-118, over this engine's lambdas):
 *     for each path i:  state = init;  sum = 0
 *         for t = 1..T:  getExpectedValue(state);  (a1, a2) = getAction(state);  d = Math.round(samples[i][t-1][.])
 *                        c = immediateValue(state, a, d)  (with the salvage term when t == T)
 *                        sum += Math.pow(discount, t-1) * c;  state = stateTransition(state, a, d, c)
 *     values[i] = sum
 * `samples` is n * T * nd doubles, row-major: nd = 2 (one demand per product) for kinds 0-2, 1 for kind 3.  Kind 2, the
 * V / Pi form, has no immediate value: a path is worth boundFinalCash (w + salvage . x) of the state reached after
 * period T, and a discount other than 1 is SDPB_ERR_ARG.  A path that meets a state the handle has not reached stops
 * there with its partial sum kept in fp64; the stalled states become the roots of one extension over several periods
 * and the stalled paths go on, at least one period further each round: at most T rounds.  SDPB_ERR_ARG: n < 1, a null
 * pointer, a sample or initial coordinate that is not finite.  stats: solve_ms = host wall time of the call, kernel_ms
 * = the roll-out kernels' device time, launches = rounds; evals grows by the evaluations of the added states. */
int  sdpb_reached_simulate(sdpb_reached* h, const double* init_state, const double* samples, int n, double discount,
                           double* values);

/* ---- any single-product model, solved over the states its top-down recursion reaches ---------------------------------
 * The reference answers getExpectedValue(state) for ANY state: it recurses top-down over real-valued states and memoises
 * what it visits (Recursion.java:89-163).  sdpb_create needs a grid (every level, action and demand a multiple of a
 * power-of-two step, initial states on it, an unclamped model sized with sdpb_reachable_hull); this engine needs none.
 * From the period-1 states it builds, period by period, exactly the states the reference visits -- successors through
 * feasible actions only, while t < T, and in the survival recursion not a successor whose cash is negative
 * (RiskRecursion.java:87-95) -- then runs the backward induction over them on the GPU with the dense engine's
 * arithmetic.  Two states are one iff their coordinates are == as doubles.
 *   inv_min / inv_max, cash_min / cash_max  only the clamp bounds the lambdas apply (no grid is built)
 *   step                                    only defines the actions a_i = i * step (exactness is not required)
 * An XR state whose order-up-to range is longer than max_order_idx + 1 is counted in sdpb_stats.capped_action_sets; the
 * solve fails with SDPB_ERR_OFFGRID unless SDPB_ALLOW_CAPPED_ACTIONS is set (the rule sdpb_reach applies).
 * Refused with SDPB_ERR_ARG: SDPB_COST_CASH_TWO_PRODUCT and SDPB_COST_STAFF (their action pairs / pmf rows are tied to
 * the grid), and a non-NULL terminal_value (tabulated on the grid: it has no value at an off-grid state).
 * stats: evals = sum_t sum_{s reached} |A_t(s)| * D_t, evals_executed = evals and capped_action_sets accumulate over
 * the life of the handle (a solve, then every extension).  solve_ms, kernel_ms and launches describe the most recent
 * call only: for a solve or an extension, solve_ms = time between CUDA events recorded on the engine's stream at its
 * start and end -- the forward pass synchronises with the host after every chunk and allocates as it goes, so this is
 * close to the wall time of the call, not kernel time alone; kernel_ms = the backward pass (its kernels and the merges
 * of new states into the tables); launches = backward launches.  For sdpb_topdown_simulate see there. */
typedef struct sdpb_topdown_options {
    uint32_t struct_size;     /* = sizeof(sdpb_topdown_options) */
    int32_t  device;          /* CUDA ordinal; -1 = current device */
    uint32_t allow;           /* sdpb_allow bits (SDPB_ALLOW_CAPPED_ACTIONS) */
    int32_t  reserved;
    int64_t  scratch_bytes;   /* forward-expansion budget, a hard bound on the scratch the expansion allocates (three
                                 buffers of 32-byte keys and the radix sort's temporary storage); 0 = half of the free
                                 device memory.  A period whose candidate successors do not fit is expanded in chunks,
                                 each holding at least as many candidates as the period has reached so far; a period
                                 whose reached states pass half a buffer fails with SDPB_ERR_NOMEM naming the period.
                                 The reached states and value tables of every period are kept outside the budget */
} sdpb_topdown_options;
typedef struct sdpb_topdown sdpb_topdown;
/* new Recursion(...) / CashRecursion / LeadtimeRecursion / RiskRecursion / CashRecursionXR + getExpectedValue on each of
 * the n period-1 states `init_states` (n * ndim API-order doubles, as sdpb_value): the memo maps the calls fill.
 * opt may be NULL. */
int  sdpb_topdown_solve(const sdpb_model* m, const sdpb_topdown_options* opt, const double* init_states, int n,
                        sdpb_topdown** out);
void sdpb_topdown_destroy(sdpb_topdown* h);
const char* sdpb_topdown_last_error(const sdpb_topdown* h);   /* h may be NULL: last sdpb_topdown_solve error, or the
                                                                 error of a call given a NULL handle */
/* getExpectedValue / getAction (Recursion.java:89-90,165-167): cacheValues / cacheActions of n reached states of one
 * period; SDPB_ERR_UNSOLVED for a state that was not reached (Java: NullPointerException).  v, q may be NULL. */
int  sdpb_topdown_value(sdpb_topdown* h, int period, const double* states, int n, double* v, double* q);
/* getOptTable() / getCacheActions() (Recursion.java:169-186): rows [t, state dims (API order)..., Q*] of every reached
 * state, sorted in memo-map order (t, x, preQ1, preQ2, cash), as sdpb_opt_table.  rows == NULL: *nrows = the count. */
int  sdpb_topdown_opt_table(sdpb_topdown* h, double* rows, size_t* nrows);
int  sdpb_topdown_states(const sdpb_topdown* h, int64_t* n_states /* T: reached states of each period */);
int  sdpb_topdown_stats(const sdpb_topdown* h, sdpb_stats* s);
/* getExpectedValue(state) on n states of one period (1..T) of a solved handle: the memo maps grow by exactly the states
 * the reference's recursion reaches from them (Recursion.java:89-163).  States already reached cost nothing, and each
 * state is evaluated once over the life of the handle, so extending with roots r2 after a solve from r1 leaves the
 * same states, values and evals as a solve from {r1, r2}.  Only the new states are expanded and solved; their values
 * do not change those already held.  Fails with SDPB_ERR_ARG (period outside 1..T, n < 0, a coordinate that is not
 * finite), SDPB_ERR_NOMEM (the scratch rule of sdpb_topdown_options, applied to the states new in a period) or
 * SDPB_ERR_OFFGRID (a new XR state with a capped action set, unless SDPB_ALLOW_CAPPED_ACTIONS); a failed call leaves
 * the reached states, tables and stats as they were.  n == 0 does nothing. */
int  sdpb_topdown_extend(sdpb_topdown* h, int period, const double* states, int n);
/* Simulation.simulateSDPGivenSamplNum / CashSimulation over the memo maps, with the reference's lazy
 * getExpectedValue(state) at every step (Simulation.java:62-63): the loop and arguments of sdpb_simulate,
 *     for each path i:  state = init;  sum = 0
 *         for t = 1..T:  getExpectedValue(state);  Q = getAction(state);  d = Math.round(samples[i][t-1])
 *                        sum += Math.pow(discount, t-1) * immediateValue(state, Q, d)
 *                        state = stateTransition(state, Q, d)
 *     values[i] = sum
 * over real-valued states: no grid, and any rounded demand.  A path that meets a state the handle has not reached
 * stops there; the stalled states become the roots of one extension (sdpb_topdown_extend, over several periods at
 * once) and the stalled paths go on from where they stopped, at least one period further each round, so there are at
 * most T rounds.  Partial sums stay in fp64 between rounds: each path's sum is the reference's bit for bit, and
 * the handle ends up with the memo the reference's roll-out leaves.  The transition is applied whatever the cash (a
 * survival model's path goes on after a bankrupt period).  SDPB_ERR_ARG: n < 1, a null pointer, a sample or initial
 * coordinate that is not finite.  An extension that fails returns its error and leaves the handle as that extension
 * found it (states added by earlier rounds stay).  stats: solve_ms = host wall time of the call, kernel_ms = the
 * roll-out kernels' device time, launches = roll-out rounds; evals grows by the evaluations of the added states. */
int  sdpb_topdown_simulate(sdpb_topdown* h, const double* init_state, const double* samples, int n, double discount,
                           double* values);

/* Return the memory cached by the library's private stream-ordered pool on `device` to the driver (-1 = current). */
int sdpb_trim_pool(int device);

#ifdef __cplusplus
}
#endif
#endif /* SDPB200_H */
