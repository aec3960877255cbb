// sqp_outer.cu -- the per-instance steps of the Sl1QP outer loop (src/Algorithm.cpp) as device kernels, one thread per NLP
// instance (SURVEY.md 8f-1): the iterate, the trust-region radius, the penalty parameter and all flags stay in HBM in SoA
// layout between the QP/LP solves and the NLP evaluations, which also run on the device; the host only sequences the
// launches and reads back a handful of counters per iteration (how many instances are still active, which Update_* flags are
// raised, how many need the penalty update).
//
// Every phase restates the corresponding reference routine with its sums in the reference's index order:
//   PH_FLAGS      loop condition of Algorithm::Optimize (:59-61) + the flag bookkeeping of setupQP (:645-697)
//   PH_AFTER_QP   QP status / KKT acceptance (QPhandler::solveQP :470-499, Algorithm :64-72), get_search_direction (:609),
//                 infea_measure_model (:592-594) and the entry test of update_penalty_parameter (:886-900)
//   PH_LP_AFTER   results of the feasibility LP (:900-912)
//   PH_PEN_CHECK  loop conditions of the two penalty while-loops (:914-972), rho_trial *= increase_parm
//   PH_PEN_AFTER  after a QP re-solve with rho_trial
//   PH_PEN_FINAL  accept / reject rho_trial (:975-1010)
//   PH_TRIAL      x_trial = x_k + p_k (:414-429)
//   PH_RATIO      cal_infea of the trial point (:577-602), ratio_test (:722-801), get_multipliers for accepted steps (:618-630)
//   PH_FINISH     new derivatives for accepted steps, iter++, check_optimality (:170-411), update_radius (:820-849)
//   PH_FINAL      EXCEED_MAX_ITER (:160-168)
//   PH_SOC_*      second_order_correction (:1140-1211, opt-in): corrected QP data, step p_k + s_k, second ratio test
//   PH_INIT       initialization (:438-472) after the evaluation at the start
// and, for streamed solves (sqpb200_sqp_optimize_stream), three phases that exchange the instance a slot holds:
//   PH_RETIRE     stopped instances: PH_FINAL's label, results to out[instance], slot freed
//   PH_REFILL     free slots take the next starting points of the queue
//   PH_INIT_REFILLED  PH_INIT for the refilled slots, from the derivatives the refill evaluation left in the scratch buffers
#include "../../include/sqpb200.h"

#include <cuda_runtime.h>

#include <vector>

int sqpb200_solve_prepare(sqpb200_handle h);  // capi.cu: a handle's first-solve allocations, made before a solve is recorded

namespace {

enum { EX_OPTIMAL = 0, EX_EXCEED_MAX_ITER = 2, EX_TRUST_REGION_TOO_SMALL = 4, EX_UNKNOWN = -99,
       EX_QP_UNCHANGED = SQPB200_EXIT_QP_UNCHANGED };
enum { CT_BOUNDED = 5, CT_EQUAL = -5, CT_BOUNDED_ABOVE = 9, CT_BOUNDED_BELOW = 1, CT_UNBOUNDED = 0 };
enum { UP_A = 1, UP_H = 2, UP_BOUNDS = 4, UP_DELTA = 8, UP_PENALTY = 16, UP_G = 32 };
// phases only the streamed loop runs (not callable through sqpb200_sqp_phase: they need the stream descriptor)
enum { PH_RETIRE = 14, PH_REFILL = 15, PH_INIT_REFILLED = 16 };
// counters[6]: occupied slots that have stopped (PH_FLAGS of a streamed solve)
enum { CNT_STOPPED = 6 };

// what the streamed phases read besides the state: the caller's descriptor and the scratch buffers of the refill evaluation.
// Zero (slot_id == nullptr) outside a streamed solve.
struct StreamArgs {
    sqpb200_sqp_stream d;
    double *f_tmp, *c_tmp;
};

// the branch points of the loop: the host decides them from the counters it reads back (synchronous solves), a CUDA graph of the loop
// from the device counters (sqp_branch_kernel)
enum { BR_ACTIVE, BR_PENALTY, BR_PEN_GO, BR_SOC, BR_STREAM_LOOP, BR_REFILL };
__host__ __device__ __forceinline__ bool branch_taken(int br, const int* cnt, unsigned long long head, long long N, int refill_min) {
    const bool queued = head < (unsigned long long)N;
    switch (br) {
    case BR_ACTIVE: return cnt[0] > 0;                 // instances active in PH_FLAGS: the outer loop goes on
    case BR_PENALTY: return cnt[2] > 0;                // PH_AFTER_QP: instances that need the penalty update
    case BR_PEN_GO: return cnt[3] > 0;                 // PH_PEN_CHECK: the penalty loop goes on
    case BR_SOC: return cnt[5] > 0;                    // PH_SOC_PREP: rejected steps enter the second-order correction
    case BR_STREAM_LOOP: return cnt[0] > 0 || queued;  // streamed: active slots or starting points left
    default: return queued && (cnt[CNT_STOPPED] >= refill_min || cnt[0] == 0);  // BR_REFILL: a refill round is due
    }
}

__device__ __forceinline__ double cal_infea(const sqpb200_sqp_state& S, const double* c, int b) {
    double s = 0.0;
    for (int i = 0; i < S.m; i++) {
        const double ci = c[(size_t)b * S.m + i], cl = S.c_l[(size_t)b * S.m + i], cu = S.c_u[(size_t)b * S.m + i];
        const double below = (ci < cl) ? cl - ci : 0.0;
        const double above = (ci >= cl && ci > cu) ? ci - cu : 0.0;
        s = s + below + above;
    }
    return s;
}

__device__ __forceinline__ void get_multipliers(const sqpb200_sqp_state& S, int b) {
    const int nV = S.n + 2 * S.m;
    const double* y = S.qp_y + (size_t)b * (nV + S.m);
    for (int i = 0; i < S.m; i++) S.lam_c[(size_t)b * S.m + i] = y[nV + i];
    for (int i = 0; i < S.n; i++) S.lam_x[(size_t)b * S.n + i] = y[i];
}

// Algorithm::check_optimality for instance b (multipliers already refreshed); writes KKT_error, may set OPTIMAL
__device__ __forceinline__ void check_optimality(const sqpb200_sqp_state& S, int b, double* diff) {
    const int n = S.n, m = S.m;
    const double *mv = S.lam_x + (size_t)b * n, *mc = S.lam_c + (size_t)b * m;
    const double primal = S.infea[b];
    double dual = 0.0, compl_ = 0.0;
    for (int i = 0; i < n; i++) {
        const int t = S.bound_type[(size_t)b * n + i];
        dual = dual + (t == CT_BOUNDED_ABOVE ? fmax(mv[i], 0.0) : 0.0) + (t == CT_BOUNDED_BELOW ? -fmin(mv[i], 0.0) : 0.0);
    }
    for (int i = 0; i < m; i++) {
        const int t = S.cons_type[(size_t)b * m + i];
        dual = dual + (t == CT_BOUNDED_ABOVE ? fmax(mc[i], 0.0) : 0.0) + (t == CT_BOUNDED_BELOW ? -fmin(mc[i], 0.0) : 0.0);
    }
    for (int i = 0; i < m; i++) {
        const int t = S.cons_type[(size_t)b * m + i];
        const double ck = S.c_k[(size_t)b * m + i];
        compl_ = compl_ + (t == CT_BOUNDED_ABOVE ? fabs(mc[i] * (S.c_u[(size_t)b * m + i] - ck)) : 0.0)
                        + (t == CT_BOUNDED_BELOW ? fabs(mc[i] * (ck - S.c_l[(size_t)b * m + i])) : 0.0)
                        + (t == CT_UNBOUNDED ? fabs(mc[i]) : 0.0);
    }
    for (int i = 0; i < n; i++) {
        const int t = S.bound_type[(size_t)b * n + i];
        const double xk = S.x_k[(size_t)b * n + i];
        compl_ = compl_ + (t == CT_BOUNDED_ABOVE ? fabs(mv[i] * (S.x_u[(size_t)b * n + i] - xk)) : 0.0)
                        + (t == CT_BOUNDED_BELOW ? fabs(mv[i] * (xk - S.x_l[(size_t)b * n + i])) : 0.0)
                        + (t == CT_UNBOUNDED ? fabs(mv[i]) : 0.0);
    }
    // stationarity: || J'y_c + y_b - grad f ||_1, triplet SpMTV in storage order (src/SpTripletMat.cpp:311-323)
    for (int i = 0; i < n; i++) diff[i] = 0.0;
    const double* jv = S.jac + (size_t)b * S.zJ;
    for (int k = 0; k < S.zJ; k++) diff[S.J_col1[k] - 1] += jv[k] * mc[S.J_row1[k] - 1];
    double stat = 0.0;
    for (int i = 0; i < n; i++) {
        const double d = diff[i] + mv[i] - S.grad[(size_t)b * n + i];
        stat = stat + fabs(d);
    }
    S.kkt_err[b] = dual + primal + compl_ + stat;
    if (primal < S.opt_prim_fea_tol && dual < S.opt_dual_fea_tol && compl_ < S.opt_compl_tol && stat < S.opt_stat_tol) S.exitflag[b] = EX_OPTIMAL;
}

// Algorithm::initialization (src/Algorithm.cpp:438-472) per instance, after f, c and the derivatives have been evaluated at the
// (shifted) start: infeasibility measure of the start, algorithm state back to the option values, backend state machines back to
// "no QP solved yet".
__device__ void init_instance(const sqpb200_sqp_state& S, int b) {
    const int n = S.n, m = S.m;
    S.infea[b] = cal_infea(S, S.c_k, b);
    S.delta[b] = S.delta0; S.rho[b] = S.rho0; S.eps1[b] = S.eps10;
    S.kkt_err[b] = __longlong_as_double(0x7ff0000000000000LL);
    S.exitflag[b] = EX_UNKNOWN; S.iter[b] = 0; S.pen_trial[b] = 0; S.qp_iter[b] = 0;
    S.active[b] = 0; S.need[b] = 0; S.go[b] = 0; S.acc[b] = 0; S.upd[b] = 0; S.feasible_lp[b] = 0; S.rej[b] = 0;
    for (int i = 0; i < n; i++) S.lam_x[(size_t)b * n + i] = 0.0;
    for (int i = 0; i < m; i++) S.neg_lam[(size_t)b * m + i] = -S.lam_c[(size_t)b * m + i];
    // st[0] = 0 ("no QP solved yet") makes the next solve of this instance an init whatever its hot-start image holds: the solve
    // kernels choose MODE_COLD from it (qp_instance_mode), the warp kernel then never reads the image and the one-QP-per-cluster
    // kernel's cold_start_state() rewrites every part of its global slice the solve reads.  So a slot that takes a new instance
    // needs no per-slot form of sqpb200_reset's image invalidation.
    for (int k = 0; k < 2; k++) {
        signed char* st = k ? S.lp_inst : S.qp_inst;
        if (st) { st += 8 * (size_t)b; st[0] = 0; st[1] = 0; st[2] = -1; st[3] = -1; st[4] = 0; st[5] = 0; st[6] = 0; st[7] = 0; }
    }
}

// PH_FINAL's labelling (src/Algorithm.cpp:160-168)
__device__ __forceinline__ void label_final(const sqpb200_sqp_state& S, int b) {
    if (S.iter[b] == S.iter_max && S.exitflag[b] == EX_UNKNOWN) S.exitflag[b] = EX_EXCEED_MAX_ITER;
}

__global__ void sqp_phase_kernel(const __grid_constant__ sqpb200_sqp_state S, int phase, const __grid_constant__ StreamArgs X) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= S.B) return;
    const int n = S.n, m = S.m, nV = n + 2 * m;
    switch (phase) {
    case SQPB200_PH_FLAGS: {
        const bool occupied = !X.d.slot_id || X.d.slot_id[b] >= 0;  // a free slot of a streamed solve is never active
        bool a = occupied && S.iter[b] < S.iter_max && S.exitflag[b] == EX_UNKNOWN;
        // no Update_* flag raised since the instance's last solve: the reference throws QP_UNCHANGED (src/Algorithm.cpp:651-670),
        // which nothing catches; here the instance ends with its own exit flag instead of re-solving the same QP until iter_max
        if (a && S.iter[b] > 0 && S.upd[b] == 0) { S.exitflag[b] = EX_QP_UNCHANGED; a = false; }
        S.active[b] = a ? 1 : 0;
        if (X.d.slot_id && occupied && !a) atomicAdd(&S.counters[CNT_STOPPED], 1);
        if (a) {
            atomicAdd(&S.counters[0], 1);
            if (S.upd[b]) atomicOr(&S.counters[1], (int)S.upd[b]);
            // this instance's matrices change (it accepted a step): its backend sees Update_A / Update_H (:361-496)
            if (S.qp_inst && (S.upd[b] & (UP_A | UP_H)) && S.clear_flags) S.qp_inst[8 * (size_t)b + 1] = 1;
            if (S.clear_flags) S.upd[b] = 0;
        }
        break;
    }
    case SQPB200_PH_AFTER_QP: {
        S.rho_trial[b] = S.rho[b];
        if (!S.active[b]) { S.need[b] = 0; break; }
        S.qp_iter[b] += S.qp_iters[b];
        const int st = S.qp_status[b];
        const bool ok = (S.qp_kkt[(size_t)b * 5 + 4] <= 1.0e-6) && st == SQPB200_QP_OPTIMAL;
        if (!ok) {
            S.exitflag[b] = (st == SQPB200_QP_OPTIMAL) ? SQPB200_QPERROR_INTERNAL_ERROR : st;
            S.active[b] = 0; S.need[b] = 0;
            break;
        }
        const double* x = S.qp_x + (size_t)b * nV;
        for (int i = 0; i < n; i++) S.p_k[(size_t)b * n + i] = x[i];
        unsigned char need = 0;
        if (S.penalty_update) {
            double s = 0.0;
            for (int i = n; i < nV; i++) s = s + fabs(x[i]);
            S.infea_model[b] = s;
            need = s > S.penalty_update_tol;
            if (need) {
                atomicAdd(&S.counters[2], 1); S.infea_model_tmp[b] = s;
                if (S.lp_inst) S.lp_inst[8 * (size_t)b + 1] = 1;  // setupLP hands this instance's Jacobian to the LP backend (:700-704)
            }
        }
        S.need[b] = need;
        break;
    }
    case SQPB200_PH_LP_AFTER: {
        if (!S.need[b]) break;
        S.qp_iter[b] += S.lp_iters[b];
        const int st = S.lp_status[b];
        if (st != SQPB200_QP_OPTIMAL) { S.exitflag[b] = st; S.need[b] = 0; break; }  // LP_NOT_OPTIMAL leaves Optimize (:900-906)
        const double* x = S.lp_x + (size_t)b * nV;
        double s = 0.0;
        for (int i = n; i < nV; i++) s = s + fabs(x[i]);
        S.infea_infty[b] = s;
        S.feasible_lp[b] = s <= S.penalty_update_tol;
        break;
    }
    case SQPB200_PH_PEN_CHECK: {
        unsigned char go = 0;
        if (S.need[b] && S.exitflag[b] == EX_UNKNOWN) {
            const double rt = S.rho_trial[b];
            const bool cont_a = S.feasible_lp[b] && S.infea_model[b] > S.penalty_update_tol && rt < S.rho_max;
            const bool cont_b = !S.feasible_lp[b] && ((S.infea[b] - S.infea_model[b]) < S.eps1[b] * (S.infea[b] - S.infea_infty[b])) &&
                                S.pen_trial[b] < S.penalty_iter_max && rt < S.rho_max;
            if (cont_a || cont_b) {
                go = 1;
                S.rho_trial[b] = fmin(S.rho_max, rt * S.increase_parm);
                S.pen_trial[b] += 1;
                atomicAdd(&S.counters[3], 1);
            }
        }
        S.go[b] = go;
        break;
    }
    case SQPB200_PH_PEN_AFTER: {
        if (!S.go[b]) break;
        S.qp_iter[b] += S.qp_iters[b];
        const int st = S.qp_status[b];
        const bool ok = (S.qp_kkt[(size_t)b * 5 + 4] <= 1.0e-6) && st == SQPB200_QP_OPTIMAL;
        if (!ok) {
            // QP_NOT_OPTIMAL inside the penalty loop only leaves the loop (:932-935, :958-961): the acceptance test of
            // PH_PEN_FINAL then sees the objective of an unsolved QP (INFTY) and takes its failure branch, and the instance runs
            // the rest of the iteration (trial point, ratio test, iter++, check_optimality) before PH_FLAGS ends its solve
            S.exitflag[b] = (st == SQPB200_QP_OPTIMAL) ? SQPB200_QPERROR_INTERNAL_ERROR : st;
            S.need[b] = 2;
            break;
        }
        const double* x = S.qp_x + (size_t)b * nV;
        double s = 0.0;
        for (int i = n; i < nV; i++) s = s + fabs(x[i]);
        S.infea_model[b] = s;
        break;
    }
    case SQPB200_PH_PEN_FINAL: {
        if (!(S.need[b] && S.rho_trial[b] > S.rho[b] && (S.exitflag[b] == EX_UNKNOWN || S.need[b] == 2))) break;
        const double rt = S.rho_trial[b], qp_obj = S.qp_obj[b];
        const bool succ = rt * S.infea[b] - qp_obj >= S.eps2 * rt * (S.infea[b] - S.infea_model[b]);
        if (succ) {
            S.eps1[b] += (1 - S.eps1[b]) * S.eps1_change_parm;
            const double* x = S.qp_x + (size_t)b * nV;
            for (int i = 0; i < n; i++) S.p_k[(size_t)b * n + i] = x[i];
            S.rho[b] = rt;
        } else {
            S.infea_model[b] = S.infea_model_tmp[b];
            S.upd[b] |= UP_PENALTY;  // the backend still holds rho_trial in g: setupQP restores rho next iteration (:1003-1006)
        }
        break;
    }
    case SQPB200_PH_TRIAL: {
        if (S.active[b] && S.exitflag[b] != EX_UNKNOWN && S.need[b] != 2) S.active[b] = 0;
        if (!S.active[b]) break;
        double np_ = 0.0;  // ||p_k||_inf for update_radius (:822); an accepted second-order correction replaces it (SOC_RATIO)
        for (int i = 0; i < n; i++) {
            S.x_trial[(size_t)b * n + i] = S.x_k[(size_t)b * n + i] + S.p_k[(size_t)b * n + i];
            np_ = fmax(np_, fabs(S.p_k[(size_t)b * n + i]));
        }
        S.norm_p[b] = np_;
        break;
    }
    case SQPB200_PH_RATIO: {
        S.acc[b] = 0;
        if (!S.active[b]) break;
        const double infea_t = cal_infea(S, S.c_trial, b);
        S.infea_trial[b] = infea_t;
        const double P1_x = S.f_k[b] + S.rho[b] * S.infea[b];
        const double P1_t = S.f_trial[b] + S.rho[b] * infea_t;
        const double ared = P1_x - P1_t, pred = S.rho[b] * S.infea[b] - S.qp_obj[b];
        S.actual_red[b] = ared; S.pred_red[b] = pred;
        if (ared >= S.eta_s * pred && ared >= -S.tol) {
            S.acc[b] = 1;
            S.infea[b] = infea_t;
            S.f_k[b] = S.f_trial[b];
            for (int i = 0; i < n; i++) S.x_k[(size_t)b * n + i] = S.x_trial[(size_t)b * n + i];
            for (int i = 0; i < m; i++) S.c_k[(size_t)b * m + i] = S.c_trial[(size_t)b * m + i];
            get_multipliers(S, b);
            S.upd[b] |= UP_A | UP_H | UP_BOUNDS | UP_G;
            atomicAdd(&S.counters[4], 1);
        }
        // multipliers handed to the Hessian evaluation: -lambda (src/SQPTNLP.cpp:124-126)
        for (int i = 0; i < m; i++) S.neg_lam[(size_t)b * m + i] = -S.lam_c[(size_t)b * m + i];
        break;
    }
    case SQPB200_PH_FINISH: {
        if (!S.active[b]) break;
        if (S.acc[b]) {
            for (int i = 0; i < n; i++) S.grad[(size_t)b * n + i] = S.g_new[(size_t)b * n + i];
            for (int i = 0; i < S.zJ; i++) S.jac[(size_t)b * S.zJ + i] = S.j_new[(size_t)b * S.zJ + i];
            for (int i = 0; i < S.zH; i++) S.hess[(size_t)b * S.zH + i] = S.h_new[(size_t)b * S.zH + i];
        }
        S.iter[b] += 1;
        double* diff = S.scratch + (size_t)b * n;
        get_multipliers(S, b);
        check_optimality(S, b, diff);
        if (S.exitflag[b] != EX_UNKNOWN) break;
        // update_radius
        const double ared = S.actual_red[b], pred = S.pred_red[b];
        const bool shrink = ared < S.eta_c * pred;
        const double norm_p = S.norm_p[b];
        const bool grow = !shrink && ared > S.eta_e * pred && S.tol > fabs(S.delta[b] - norm_p);
        if (shrink) S.delta[b] = S.gamma_c * S.delta[b];
        if (grow) S.delta[b] = fmin(S.gamma_e * S.delta[b], S.delta_max);
        if (shrink || grow) S.upd[b] |= UP_DELTA;
        if (S.delta[b] < S.delta_min) {
            S.exitflag[b] = EX_TRUST_REGION_TOO_SMALL;
            check_optimality(S, b, diff);  // :149-152
        }
        break;
    }
    case SQPB200_PH_SOC_PREP: {
        // rejected steps: QP data of the corrected subproblem (gradient H_k p_k + g_k, bounds around the trial point); every
        // other instance keeps its current data in the mixed arrays
        const bool rj = S.active[b] && !S.acc[b] && S.exitflag[b] == EX_UNKNOWN;
        S.rej[b] = rj ? 1 : 0;
        double* sg = S.soc_g + (size_t)b * n;
        if (rj) {
            atomicAdd(&S.counters[5], 1);
            const double *hv = S.hess + (size_t)b * S.zH, *p = S.p_k + (size_t)b * n;
            for (int i = 0; i < n; i++) sg[i] = 0.0;
            for (int k = 0; k < S.zH; k++) {  // symmetric-half triplet product in storage order (src/SpTripletMat.cpp:237-258)
                const int i = S.H_row1[k] - 1, j = S.H_col1[k] - 1;
                sg[i] += hv[k] * p[j];
                if (i != j) sg[j] += hv[k] * p[i];
            }
            for (int i = 0; i < n; i++) { sg[i] = sg[i] + S.grad[(size_t)b * n + i]; S.p_tmp[(size_t)b * n + i] = p[i]; }
            S.qp_obj_tmp[b] = S.qp_obj[b];
        } else {
            for (int i = 0; i < n; i++) sg[i] = S.grad[(size_t)b * n + i];
        }
        for (int i = 0; i < n; i++) S.soc_x[(size_t)b * n + i] = rj ? S.x_trial[(size_t)b * n + i] : S.x_k[(size_t)b * n + i];
        for (int i = 0; i < m; i++) S.soc_c[(size_t)b * m + i] = rj ? S.c_trial[(size_t)b * m + i] : S.c_k[(size_t)b * m + i];
        break;
    }
    case SQPB200_PH_SOC_AFTER: {
        if (!S.rej[b]) break;
        S.qp_iter[b] += S.qp_iters[b];
        const int st = S.qp_status[b];
        const bool ok = (S.qp_kkt[(size_t)b * 5 + 4] <= 1.0e-6) && st == SQPB200_QP_OPTIMAL;
        if (!ok) {
            S.exitflag[b] = (st == SQPB200_QP_OPTIMAL) ? SQPB200_QPERROR_INTERNAL_ERROR : st;
            S.rej[b] = 2;  // left the correction with a solver failure: the saved step is restored in SOC_RATIO
            break;
        }
        const double* x = S.qp_x + (size_t)b * nV;
        S.qp_obj_soc[b] = S.qp_obj[b] + (S.qp_obj_tmp[b] - S.rho[b] * S.infea_model[b]);
        for (int i = 0; i < n; i++) {
            const double pk = S.p_k[(size_t)b * n + i] + x[i];
            S.p_k[(size_t)b * n + i] = pk;
            S.x_trial[(size_t)b * n + i] = S.x_k[(size_t)b * n + i] + pk;
        }
        break;
    }
    case SQPB200_PH_SOC_RATIO: {
        if (S.rej[b] == 1) {
            const double infea_t = cal_infea(S, S.c_trial, b);
            S.infea_trial[b] = infea_t;
            const double P1_x = S.f_k[b] + S.rho[b] * S.infea[b];
            const double P1_t = S.f_trial[b] + S.rho[b] * infea_t;
            // pred_reduction_ = rho * infea - get_obj_QP(): the raw objective of the SOC QP just solved (src/Algorithm.cpp:728);
            // qp_obj_soc mirrors the reference's qp_obj_ bookkeeping (:1197), which no test reads
            const double ared = P1_x - P1_t, pred = S.rho[b] * S.infea[b] - S.qp_obj[b];
            S.actual_red[b] = ared; S.pred_red[b] = pred;
            if (ared >= S.eta_s * pred && ared >= -S.tol) {
                S.acc[b] = 1;
                // update_radius reads p_k_->getInfNorm() (src/Algorithm.cpp:822): after an accepted correction that is the norm of the
                // corrected step p_k + s_k, which p_k holds since SOC_AFTER
                double np_ = 0.0;
                for (int i = 0; i < n; i++) np_ = fmax(np_, fabs(S.p_k[(size_t)b * n + i]));
                S.norm_p[b] = np_;
                S.infea[b] = infea_t;
                S.f_k[b] = S.f_trial[b];
                for (int i = 0; i < n; i++) S.x_k[(size_t)b * n + i] = S.x_trial[(size_t)b * n + i];
                for (int i = 0; i < m; i++) S.c_k[(size_t)b * m + i] = S.c_trial[(size_t)b * m + i];
                get_multipliers(S, b);
                S.upd[b] |= UP_A | UP_H | UP_BOUNDS | UP_G;
                for (int i = 0; i < m; i++) S.neg_lam[(size_t)b * m + i] = -S.lam_c[(size_t)b * m + i];
            } else {
                for (int i = 0; i < n; i++) S.p_k[(size_t)b * n + i] = S.p_tmp[(size_t)b * n + i];
            }
        } else if (S.rej[b] == 2) {
            for (int i = 0; i < n; i++) S.p_k[(size_t)b * n + i] = S.p_tmp[(size_t)b * n + i];
        }
        break;
    }
    case SQPB200_PH_INIT: {
        // lets one DeviceBatchedSQP object (handles, buffers, compiled NLP) serve batch after batch
        init_instance(S, b);
        break;
    }
    case SQPB200_PH_FINAL: {
        label_final(S, b);
        break;
    }
    case PH_RETIRE: {
        const long long id = X.d.slot_id[b];
        if (id < 0 || (S.exitflag[b] == EX_UNKNOWN && S.iter[b] != S.iter_max)) break;
        label_final(S, b);
        for (int i = 0; i < n; i++) X.d.x[id * n + i] = S.x_k[(size_t)b * n + i];
        X.d.obj[id] = S.f_k[b]; X.d.exitflag[id] = S.exitflag[b]; X.d.iter[id] = S.iter[b]; X.d.qp_iter[id] = S.qp_iter[b];
        X.d.kkt_err[id] = S.kkt_err[b]; X.d.rho[id] = S.rho[b]; X.d.delta[id] = S.delta[b];
        X.d.slot_id[b] = -1;
        break;
    }
    case PH_REFILL: {
        X.d.refill[b] = 0;
        if (X.d.slot_id[b] >= 0) break;
        const unsigned long long id = atomicAdd(X.d.head, 1ULL);
        if (id >= (unsigned long long)X.d.N) break;
        X.d.slot_id[b] = (long long)id;
        // shift_starting_point (src/SQPTNLP.cpp:140-153): max with the lower bound, then min with the upper one, as reset() does
        const double* x0 = X.d.x0_all + id * n;
        for (int i = 0; i < n; i++) {
            double v = x0[i];
            const double lo = S.x_l[(size_t)b * n + i], hi = S.x_u[(size_t)b * n + i];
            v = v > lo ? v : lo;
            v = v < hi ? v : hi;
            S.x_k[(size_t)b * n + i] = v;
        }
        for (int i = 0; i < m; i++) {
            S.lam_c[(size_t)b * m + i] = X.d.lam_start[i];
            S.neg_lam[(size_t)b * m + i] = -X.d.lam_start[i];
        }
        X.d.refill[b] = 1;
        break;
    }
    case PH_INIT_REFILLED: {
        if (!X.d.refill[b]) break;
        S.f_k[b] = X.f_tmp[b];
        for (int i = 0; i < m; i++) S.c_k[(size_t)b * m + i] = X.c_tmp[(size_t)b * m + i];
        for (int i = 0; i < n; i++) S.grad[(size_t)b * n + i] = S.g_new[(size_t)b * n + i];
        for (int i = 0; i < S.zJ; i++) S.jac[(size_t)b * S.zJ + i] = S.j_new[(size_t)b * S.zJ + i];
        for (int i = 0; i < S.zH; i++) S.hess[(size_t)b * S.zH + i] = S.h_new[(size_t)b * S.zH + i];
        init_instance(S, b);
        break;
    }
    }
}

// sets the condition of a conditional node of a recorded loop: one thread, after the phase that counted
__global__ void sqp_branch_kernel(cudaGraphConditionalHandle hc, const int* counters, int br, const unsigned long long* head, long long N,
                                  int refill_min) {
    cudaGraphSetConditional(hc, branch_taken(br, counters, head ? *head : 0ULL, N, refill_min) ? 1u : 0u);
}

}  // namespace

static int launch_phase(const sqpb200_sqp_state* st, int phase, const StreamArgs& X, int* counters_host, cudaStream_t stream) {
    if (X.d.slot_id && phase == SQPB200_PH_FLAGS) {
        // a streamed solve also counts stopped slots (counters[6]) in PH_FLAGS
        if (cudaMemsetAsync(st->counters, 0, 8 * sizeof(int), stream) != cudaSuccess) return SQPB200_ERR_CUDA;
    } else if (phase == SQPB200_PH_FLAGS || phase == SQPB200_PH_AFTER_QP || phase == SQPB200_PH_PEN_CHECK || phase == SQPB200_PH_RATIO || phase == SQPB200_PH_SOC_PREP) {
        // counters: [0] active, [1] OR of Update_* flags, [2] need penalty update, [3] go, [4] accepted
        const int idx = phase == SQPB200_PH_FLAGS ? 0 : (phase == SQPB200_PH_AFTER_QP ? 2 : (phase == SQPB200_PH_PEN_CHECK ? 3 : (phase == SQPB200_PH_RATIO ? 4 : 5)));
        if (cudaMemsetAsync(st->counters + idx, 0, (phase == SQPB200_PH_FLAGS ? 2 : 1) * sizeof(int), stream) != cudaSuccess) return SQPB200_ERR_CUDA;
    }
    const int block = 128, grid = (st->B + block - 1) / block;
    sqp_phase_kernel<<<grid, block, 0, stream>>>(*st, phase, X);
    if (cudaGetLastError() != cudaSuccess) return SQPB200_ERR_CUDA;
    if (counters_host) {
        if (cudaMemcpyAsync(counters_host, st->counters, 8 * sizeof(int), cudaMemcpyDeviceToHost, stream) != cudaSuccess) return SQPB200_ERR_CUDA;
        if (cudaStreamSynchronize(stream) != cudaSuccess) return SQPB200_ERR_CUDA;
    }
    return 0;
}

int sqpb200_sqp_phase(const sqpb200_sqp_state* st, int phase, int* counters_host, void* stream) {
    if (!st || st->B <= 0 || phase < SQPB200_PH_FLAGS || phase > SQPB200_PH_INIT) return SQPB200_ERR_INVALID;
    return launch_phase(st, phase, StreamArgs{}, counters_host, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------------------------------
// Algorithm::Optimize (src/Algorithm.cpp:55-168) for the whole batch, sequenced from C++ with no interpreter between the
// launches (at 10^4 instances the device work of an outer iteration is a few tens of microseconds, so the host side is what
// is timed).  The caller has set the structures of both
// handles (sqpb200_set_structure_A / _H) and evaluated the start point; `stream` must be the stream of both handles.
// ---------------------------------------------------------------------------------------------------------------------
namespace {
struct OuterLoop {
    sqpb200_sqp_state* S;
    sqpb200_handle qp, lp;
    sqpb200_nlp nlp;
    cudaStream_t stream;
    int bounds_update_mode;
    int cnt[8];
    long long launches;
    int rc;
    StreamArgs X{};  // the streamed phases' arguments (zero outside a streamed solve) and the scratch buffers f_tmp / c_tmp
    bool recording = false;  // the launches are being recorded into a CUDA graph (sqpb200_sqp_graph_create / _launch)
    bool ph(int phase, bool read = false) {
        rc = launch_phase(S, phase, X, read && !recording ? cnt : nullptr, stream);
        launches++;
        return rc == 0;
    }
    bool cuda(cudaError_t e) {
        rc = e == cudaSuccess ? 0 : SQPB200_ERR_CUDA;
        return rc == 0;
    }
    bool set_branch(cudaGraphConditionalHandle hc, int br) {
        sqp_branch_kernel<<<1, 1, 0, stream>>>(hc, S->counters, br, X.d.head, X.d.N, X.d.refill_min);
        return cuda(cudaGetLastError());
    }
    // A branch point: `body` runs once (loop = false) or as long as the condition holds (loop = true; the body's last phase counts
    // again).  Synchronous solves test the counters read back last.  While the loop is recorded, the branch becomes a conditional
    // node (IF / WHILE) set by sqp_branch_kernel: the capture of the enclosing graph ends in front of the node, the body is recorded
    // into the node's body graph on the same stream, and the enclosing capture resumes behind the node.
    template <class F>
    bool branch(int br, bool loop, F body) {
        if (!recording) {
            while (branch_taken(br, cnt, 0, 0, 0)) {
                if (!body()) return false;
                if (!loop) break;
            }
            return true;
        }
        cudaStreamCaptureStatus cs;
        cudaGraph_t g, t;
        const cudaGraphNode_t* d = nullptr;
        size_t nd = 0;
        cudaGraphConditionalHandle hc;
        if (!cuda(cudaStreamGetCaptureInfo(stream, &cs, nullptr, &g)) || !cuda(cudaGraphConditionalHandleCreate(&hc, g, 0, 0)) ||
            !set_branch(hc, br) || !cuda(cudaStreamGetCaptureInfo(stream, &cs, nullptr, &g, &d, &nd)))
            return false;
        std::vector<cudaGraphNode_t> deps(d, d + nd);
        if (!cuda(cudaStreamEndCapture(stream, &t))) return false;
        cudaGraphNodeParams p = {};
        p.type = cudaGraphNodeTypeConditional;
        p.conditional.handle = hc;
        p.conditional.type = loop ? cudaGraphCondTypeWhile : cudaGraphCondTypeIf;
        p.conditional.size = 1;
        cudaGraphNode_t node;
        if (!cuda(cudaGraphAddNode(&node, g, deps.data(), deps.size(), &p)) ||
            !cuda(cudaStreamBeginCaptureToGraph(stream, p.conditional.phGraph_out[0], nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed)))
            return false;
        if (!body() || (loop && !set_branch(hc, br)) || !cuda(cudaStreamEndCapture(stream, &t))) return false;
        return cuda(cudaStreamBeginCaptureToGraph(stream, g, &node, nullptr, 1, cudaStreamCaptureModeRelaxed));
    }
    bool solve(sqpb200_handle h, int type, const unsigned char* mask, signed char* inst) {
        rc = inst ? sqpb200_solve_per_instance(h, type, 0, mask, inst) : sqpb200_solve_device_mask(h, type, 0, mask);
        return rc == 0;
    }
    bool bounds(sqpb200_handle h, int mode, const double* xk, const double* ck) {
        rc = sqpb200_qphandler_bounds(h, mode, S->n, S->m, S->delta, S->x_l, S->x_u, xk, S->c_l, S->c_u, ck, SQPB200_LOC_DEVICE);
        return rc == 0;
    }
    bool grad(sqpb200_handle h, const double* g, const double* rho) {
        rc = sqpb200_qphandler_g(h, S->n, S->m, g, rho, SQPB200_LOC_DEVICE);
        return rc == 0;
    }
    // an empty Jacobian (m = 0) still raises Update_A like the reference's setter; the pointer is then never dereferenced
    bool valsA(sqpb200_handle h) { rc = sqpb200_set_values_A(h, S->zJ > 0 ? S->jac : S->x_k, SQPB200_LOC_DEVICE, 0); return rc == 0; }
    bool valsH(sqpb200_handle h) { rc = S->zH > 0 ? sqpb200_set_values_H(h, S->hess, SQPB200_LOC_DEVICE, 0) : 0; return rc == 0; }
    // setupQP, src/Algorithm.cpp:645-697.  The reference refreshes only what its Update_* flags name; here every refresh is
    // issued every iteration (rewriting unchanged data with itself), so that the host does not have to read the flags back
    // before it can queue the QP solve.  What the flags decide -- init / hotstart of each instance's backend -- is taken from
    // the per-instance flags on the device (PH_FLAGS), not from which setters were called.
    bool setupQP(int* first) {
        if (!valsA(qp) || !valsH(qp)) return false;
        if (*first) {
            if (!bounds(qp, 0, S->x_k, S->c_k)) return false;
            *first = 0;
            S->clear_flags = 1;
        } else if (!bounds(qp, bounds_update_mode, S->x_k, S->c_k)) return false;
        return grad(qp, S->grad, S->rho);
    }
    // the reference's own form (only what the Update_* bits name): used with handle-level init / hotstart decisions, where the
    // setters that were called decide the mode of the whole batch
    bool setupQP_bits(int bits, int* first) {
        if (*first) {
            if (!valsA(qp) || !valsH(qp) || !bounds(qp, 0, S->x_k, S->c_k) || !grad(qp, S->grad, S->rho)) return false;
            *first = 0;
            S->clear_flags = 1;
            return true;
        }
        if ((bits & 1) && !valsA(qp)) return false;
        if ((bits & 2) && !valsH(qp)) return false;
        if (bits & 4) { if (!bounds(qp, bounds_update_mode, S->x_k, S->c_k)) return false; }
        else if (bits & 8) { if (!bounds(qp, 2, S->x_k, nullptr)) return false; }
        if ((bits & 16) && !grad(qp, nullptr, S->rho)) return false;
        if ((bits & 32) && !grad(qp, S->grad, nullptr)) return false;
        return true;
    }
    // update_penalty_parameter, src/Algorithm.cpp:886-1028
    bool penalty() {
        if (!bounds(lp, 0, S->x_k, S->c_k) || !grad(lp, nullptr, S->rho) || !valsA(lp)) return false;  // setupLP :700-704
        if (!solve(lp, SQPB200_LP, S->need, S->lp_inst) || !ph(SQPB200_PH_LP_AFTER) || !ph(SQPB200_PH_PEN_CHECK, true)) return false;
        return branch(BR_PEN_GO, true, [&] {
            return grad(qp, nullptr, S->rho_trial) && solve(qp, SQPB200_QP, S->go, S->qp_inst) && ph(SQPB200_PH_PEN_AFTER) &&
                   ph(SQPB200_PH_PEN_CHECK, true);
        }) && ph(SQPB200_PH_PEN_FINAL);
    }
    // second_order_correction, src/Algorithm.cpp:1140-1211
    bool soc() {
        if (!ph(SQPB200_PH_SOC_PREP, true)) return false;
        return branch(BR_SOC, false, [&] {
            if (!grad(qp, S->soc_g, nullptr) || !bounds(qp, bounds_update_mode, S->soc_x, S->soc_c)) return false;
            if (!solve(qp, SQPB200_QP, S->rej, S->qp_inst) || !ph(SQPB200_PH_SOC_AFTER)) return false;
            rc = sqpb200_nlp_eval(nlp, 0, S->B, S->x_trial, nullptr, S->f_trial, S->c_trial, nullptr, nullptr, nullptr, SQPB200_LOC_DEVICE, stream);
            if (rc) return false;
            launches++;
            if (!ph(SQPB200_PH_SOC_RATIO)) return false;
            return grad(qp, S->grad, nullptr) && bounds(qp, bounds_update_mode, S->x_k, S->c_k);
        });
    }
    // the start of an outer iteration of a per-instance-mode solve: flags, QP data, QP solve, its acceptance
    bool qp_step(int* first) {
        return ph(SQPB200_PH_FLAGS) && setupQP(first) && solve(qp, SQPB200_QP, S->active, S->qp_inst) && ph(SQPB200_PH_AFTER_QP);
    }
    // one outer iteration after the QP solve, for the instances that were active in PH_FLAGS
    bool rest_of_iteration(int second_order_correction) {
        if (!branch(BR_PENALTY, false, [&] { return penalty(); })) return false;
        if (!ph(SQPB200_PH_TRIAL)) return false;
        // get_trial_point_info :414-429
        rc = sqpb200_nlp_eval(nlp, 0, S->B, S->x_trial, nullptr, S->f_trial, S->c_trial, nullptr, nullptr, nullptr, SQPB200_LOC_DEVICE, stream);
        if (rc) return false;
        if (!ph(SQPB200_PH_RATIO)) return false;
        if (second_order_correction && !soc()) return false;
        rc = sqpb200_nlp_eval(nlp, 1, S->B, S->x_k, S->neg_lam, X.f_tmp, X.c_tmp, S->g_new, S->j_new, S->h_new, SQPB200_LOC_DEVICE, stream);
        if (rc) return false;
        launches += 2;
        return ph(SQPB200_PH_FINISH);
    }
    // free slots take the next starting points; initialization() for them: one evaluation of the whole batch (the generated evaluator
    // has no instance mask) into the scratch buffers, which nothing reads between PH_FINISH and the next evaluation before PH_FINISH
    bool refill() {
        if (!ph(PH_REFILL)) return false;
        rc = sqpb200_nlp_eval(nlp, 1, S->B, S->x_k, S->neg_lam, X.f_tmp, X.c_tmp, S->g_new, S->j_new, S->h_new, SQPB200_LOC_DEVICE, stream);
        if (rc) return false;
        launches++;
        X.d.rounds++;
        return ph(PH_INIT_REFILLED);
    }
};
}  // namespace

int sqpb200_sqp_optimize(sqpb200_sqp_state* st, sqpb200_handle qp, sqpb200_handle lp, sqpb200_nlp nlp, int second_order_correction,
                         int refresh_ubA, int* first, double* f_tmp, double* c_tmp, long long* launches, void* stream) {
    if (!st || !qp || !lp || !nlp || !first || st->B <= 0) return SQPB200_ERR_INVALID;
    OuterLoop L{st, qp, lp, nlp, (cudaStream_t)stream, refresh_ubA ? 3 : 1, {0, 0, 0, 0, 0, 0, 0, 0}, 0, 0};
    L.X.f_tmp = f_tmp; L.X.c_tmp = c_tmp;
    for (;;) {
        // one read-back per outer iteration: the number of active instances (PH_FLAGS) and of instances that need the penalty
        // update (PH_AFTER_QP) come back together, after the QP solve has been queued behind the data refresh
        if (st->qp_inst) {
            if (!L.ph(SQPB200_PH_FLAGS)) return L.rc;
            if (!L.setupQP(first)) return L.rc;
        } else {
            if (!L.ph(SQPB200_PH_FLAGS, true)) return L.rc;
            if (L.cnt[0] == 0) break;
            if (!L.setupQP_bits(L.cnt[1], first)) return L.rc;
        }
        if (!L.solve(qp, SQPB200_QP, st->active, st->qp_inst)) return L.rc;
        if (!L.ph(SQPB200_PH_AFTER_QP, true)) return L.rc;
        if (L.cnt[0] == 0) break;  // nobody was active: the iteration above touched nothing
        if (!L.rest_of_iteration(second_order_correction)) return L.rc;
    }
    if (!L.ph(SQPB200_PH_FINAL)) return L.rc;
    if (launches) *launches = L.launches;
    return 0;
}

static bool stream_desc_ok(const sqpb200_sqp_state* st, const sqpb200_sqp_stream* sd) {
    if (sd->N < 0 || sd->refill_min < 1 || !sd->slot_id || !sd->head || !sd->refill) return false;
    return sd->N == 0 || (sd->x0_all && sd->x && sd->obj && sd->kkt_err && sd->rho && sd->delta && sd->exitflag && sd->iter && sd->qp_iter &&
                          (st->m == 0 || sd->lam_start));
}

// The same loop over a queue of N starting points.  A slot whose instance has stopped keeps its state (nothing changes a stopped
// instance's results) until a refill round retires it to out[instance] and hands it the next starting point; the refilled slot
// then runs initialization() and starts cold in both backends (PH_INIT_REFILLED), so its trajectory is the one it has in any batch.
// Its first setupQP is an update_bounds (mode 3) where a fresh batch's is a set_bounds (mode 0): the two write the same lb, ub, lbA,
// ubA for an instance except the slack bounds (0, 1e18), which mode 0 set for every slot in the object's first iteration and which
// nothing else writes.
int sqpb200_sqp_optimize_stream(sqpb200_sqp_state* st, sqpb200_handle qp, sqpb200_handle lp, sqpb200_nlp nlp,
                                int second_order_correction, int refresh_ubA, int* first, double* f_tmp, double* c_tmp,
                                sqpb200_sqp_stream* sd, long long* launches, void* stream) {
    if (!st || !qp || !lp || !nlp || !first || !sd || st->B <= 0) return SQPB200_ERR_INVALID;
    // handle-level init / hotstart decisions: a refilled slot would inherit its handle's hot start
    if (!st->qp_inst || !st->lp_inst || !stream_desc_ok(st, sd)) return SQPB200_ERR_INVALID;
    cudaStream_t cs = (cudaStream_t)stream;
    OuterLoop L{st, qp, lp, nlp, cs, refresh_ubA ? 3 : 1, {0, 0, 0, 0, 0, 0, 0, 0}, 0, 0};
    L.X.d = *sd;
    L.X.d.rounds = 0;
    L.X.f_tmp = f_tmp; L.X.c_tmp = c_tmp;
    if (cudaMemsetAsync(sd->slot_id, 0xff, (size_t)st->B * sizeof(long long), cs) != cudaSuccess ||
        cudaMemsetAsync(sd->head, 0, sizeof(unsigned long long), cs) != cudaSuccess)
        return SQPB200_ERR_CUDA;
    if (!L.refill()) return L.rc;
    unsigned long long head = 0;
    for (;;) {
        if (!L.qp_step(first)) return L.rc;
        // the loop's one read-back per outer iteration: active and stopped slots (PH_FLAGS), penalty updates (PH_AFTER_QP), queue head
        if (cudaMemcpyAsync(L.cnt, st->counters, 8 * sizeof(int), cudaMemcpyDeviceToHost, cs) != cudaSuccess ||
            cudaMemcpyAsync(&head, sd->head, sizeof head, cudaMemcpyDeviceToHost, cs) != cudaSuccess || cudaStreamSynchronize(cs) != cudaSuccess)
            return SQPB200_ERR_CUDA;
        const bool queued = head < (unsigned long long)sd->N;
        if (L.cnt[0] == 0 && !queued) break;
        if (L.cnt[0] > 0 && !L.rest_of_iteration(second_order_correction)) return L.rc;
        if (queued && (L.cnt[CNT_STOPPED] >= sd->refill_min || L.cnt[0] == 0) && (!L.ph(PH_RETIRE) || !L.refill())) return L.rc;
    }
    if (!L.ph(PH_RETIRE)) return L.rc;
    sd->rounds = L.X.d.rounds;
    if (launches) *launches = L.launches;
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// The same loops recorded once as CUDA graphs, every host branch a conditional node (OuterLoop::branch), so that a solve is queued on
// the stream and returns without waiting.  What a recorded launch freezes and how the calls keep results bit-identical:
//   - the state goes in by value: the loop is recorded with clear_flags = 1 and with setupQP's update_bounds (first = 0), so the
//     first iteration -- PH_FLAGS with the caller's clear_flags, setupQP(first), the QP solve, PH_AFTER_QP -- is queued as ordinary
//     launches in front of the graph, and PH_FINAL (PH_RETIRE) behind it;
//   - the streamed descriptor goes in by value too: a streamed launch records its loop again (a graph per call);
//   - a recorded solve neither allocates nor reads back (sqpb200_solve_prepare before, solve_impl skips the capacity read-back).
// The loop is recorded on a private stream, both handles moved there meanwhile: the caller's stream may be the legacy default
// stream, which cannot be captured.
// ---------------------------------------------------------------------------------------------------------------------
struct sqpb200_sqp_graph_s {
    sqpb200_sqp_state* st;
    sqpb200_handle qp, lp;
    sqpb200_nlp nlp;
    int second_order_correction, bounds_update_mode;
    double *f_tmp, *c_tmp;
    cudaStream_t stream;                      // the caller's: where launches are queued
    cudaStream_t rec = nullptr;               // where the loops are recorded
    cudaGraphExec_t optimize = nullptr, streamed = nullptr;
};

// records fn(L) into *out (replacing what it held)
template <class F>
static int record(sqpb200_sqp_graph g, const StreamArgs& X, cudaGraphExec_t* out, F fn) {
    sqpb200_sqp_state S = *g->st;
    S.clear_flags = 1;
    OuterLoop L{&S, g->qp, g->lp, g->nlp, g->rec, g->bounds_update_mode, {0, 0, 0, 0, 0, 0, 0, 0}, 0, 0};
    L.X = X;
    L.recording = true;
    cudaGraph_t top = nullptr;
    int rc = sqpb200_set_stream(g->qp, g->rec);
    if (!rc) rc = sqpb200_set_stream(g->lp, g->rec);
    if (!rc && cudaGraphCreate(&top, 0) != cudaSuccess) rc = SQPB200_ERR_CUDA;
    if (!rc && cudaStreamBeginCaptureToGraph(g->rec, top, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed) != cudaSuccess) rc = SQPB200_ERR_CUDA;
    if (!rc && !fn(L)) rc = L.rc ? L.rc : SQPB200_ERR_CUDA;
    // a failure may leave a capture open, in a body graph
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(g->rec, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone) {
        cudaGraph_t t;
        if (cudaStreamEndCapture(g->rec, &t) != cudaSuccess && !rc) rc = SQPB200_ERR_CUDA;
    }
    const int r1 = sqpb200_set_stream(g->qp, g->stream), r2 = sqpb200_set_stream(g->lp, g->stream);
    if (!rc) rc = r1 ? r1 : r2;
    cudaGraphExec_t e = nullptr;
    if (!rc && cudaGraphInstantiate(&e, top, 0) != cudaSuccess) rc = SQPB200_ERR_CUDA;
    if (!rc) {
        if (*out) cudaGraphExecDestroy(*out);  // an exec still running is freed when it completes
        *out = e;
    }
    if (top) cudaGraphDestroy(top);
    return rc;
}

int sqpb200_sqp_graph_create(sqpb200_sqp_state* st, sqpb200_handle qp, sqpb200_handle lp, sqpb200_nlp nlp, int second_order_correction,
                             int refresh_ubA, double* f_tmp, double* c_tmp, void* stream, sqpb200_sqp_graph* out) {
    if (!out) return SQPB200_ERR_INVALID;
    *out = nullptr;
    if (!st || !qp || !lp || !nlp || st->B <= 0 || !st->qp_inst || !st->lp_inst) return SQPB200_ERR_INVALID;
    int rc = sqpb200_solve_prepare(qp);
    if (!rc) rc = sqpb200_solve_prepare(lp);
    if (rc) return rc;
    sqpb200_sqp_graph g = new sqpb200_sqp_graph_s{st, qp, lp, nlp, second_order_correction, refresh_ubA ? 3 : 1, f_tmp, c_tmp,
                                                  (cudaStream_t)stream};
    if (cudaStreamCreateWithFlags(&g->rec, cudaStreamNonBlocking) != cudaSuccess) { delete g; return SQPB200_ERR_CUDA; }
    StreamArgs X{};
    X.f_tmp = f_tmp; X.c_tmp = c_tmp;
    rc = record(g, X, &g->optimize, [&](OuterLoop& L) {
        int first = 0;
        return L.branch(BR_ACTIVE, true, [&] { return L.rest_of_iteration(second_order_correction) && L.qp_step(&first); });
    });
    if (rc) { sqpb200_sqp_graph_destroy(g); return rc; }
    *out = g;
    return 0;
}

int sqpb200_sqp_graph_launch(sqpb200_sqp_graph g, int* first, sqpb200_sqp_stream* sd) {
    if (!g || !first) return SQPB200_ERR_INVALID;
    StreamArgs X{};
    X.f_tmp = g->f_tmp; X.c_tmp = g->c_tmp;
    if (sd) {
        if (!stream_desc_ok(g->st, sd)) return SQPB200_ERR_INVALID;
        X.d = *sd;
        const int soc = g->second_order_correction;
        const int rc = record(g, X, &g->streamed, [&](OuterLoop& L) {
            int zero = 0;
            return L.branch(BR_STREAM_LOOP, true, [&] {
                return L.branch(BR_ACTIVE, false, [&] { return L.rest_of_iteration(soc); }) &&
                       L.branch(BR_REFILL, false, [&] { return L.ph(PH_RETIRE) && L.refill(); }) && L.qp_step(&zero);
            });
        });
        if (rc) return rc;
    }
    OuterLoop L{g->st, g->qp, g->lp, g->nlp, g->stream, g->bounds_update_mode, {0, 0, 0, 0, 0, 0, 0, 0}, 0, 0};
    L.X = X;
    if (sd && (cudaMemsetAsync(sd->slot_id, 0xff, (size_t)g->st->B * sizeof(long long), g->stream) != cudaSuccess ||
               cudaMemsetAsync(sd->head, 0, sizeof(unsigned long long), g->stream) != cudaSuccess))
        return SQPB200_ERR_CUDA;
    if ((sd && !L.refill()) || !L.qp_step(first)) return L.rc;
    if (cudaGraphLaunch(sd ? g->streamed : g->optimize, g->stream) != cudaSuccess) return SQPB200_ERR_CUDA;
    return L.ph(sd ? PH_RETIRE : SQPB200_PH_FINAL) ? 0 : L.rc;
}

int sqpb200_sqp_graph_destroy(sqpb200_sqp_graph g) {
    if (!g) return SQPB200_ERR_INVALID;
    if (g->optimize) cudaGraphExecDestroy(g->optimize);
    if (g->streamed) cudaGraphExecDestroy(g->streamed);
    if (g->rec) cudaStreamDestroy(g->rec);
    delete g;
    return 0;
}
