// BatchedAlgorithm.cpp -- see BatchedAlgorithm.hpp.  Host sequencing and memory only: every numerical step runs in libsqpb200.so.
#include "BatchedAlgorithm.hpp"

#include <cuda_runtime.h>

#include <cstring>
#include <stdexcept>

namespace sqpb200 {

namespace {

const double INF = 1.0e18;  // include/sqphot/Types.hpp:21

// ConstraintType of a bound pair (include/sqphot/Types.hpp:75-81), decided as classify_single_constraint does
// (src/Utils.cpp:29-45): both sides finite -> EQUAL (gap < 1e-8) or BOUNDED; its one-sided tests are `upper > INF` / `lower < -INF`
int constraint_class(double lo, double hi) {
    const int BOUNDED = 5, EQUAL = -5, BOUNDED_ABOVE = 9, BOUNDED_BELOW = 1, UNBOUNDED = 0;
    if (lo > -INF && hi < INF) return (hi - lo) < 1.0e-8 ? EQUAL : BOUNDED;
    if (lo > -INF && hi > INF) return BOUNDED_BELOW;
    if (hi < INF && lo < -INF) return BOUNDED_ABOVE;
    return UNBOUNDED;
}

void cuda_check(cudaError_t e, const char* what) {
    if (e != cudaSuccess) throw std::runtime_error(std::string(what) + ": " + cudaGetErrorString(e));
}

// one arena for the whole SoA state: every array starts 256-byte aligned
struct Carver {
    char* base = nullptr;
    size_t off = 0;
    size_t take(size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; }
};

template <typename T>
std::vector<T> tiled(const std::vector<T>& row, int B) {
    std::vector<T> out((size_t)B * row.size());
    for (int b = 0; b < B; b++) std::memcpy(out.data() + (size_t)b * row.size(), row.data(), row.size() * sizeof(T));
    return out;
}

}  // namespace

void BatchedAlgorithm::check(int rc, const char* what) const {
    if (rc < 0) {
        std::string msg = std::string(what) + " failed (" + std::to_string(rc) + ")";
        if (qp_) msg += std::string(": ") + sqpb200_last_error(qp_);
        if (lp_) msg += std::string(" / ") + sqpb200_last_error(lp_);
        throw std::runtime_error(msg);
    }
}

BatchedAlgorithm::BatchedAlgorithm(const BatchedNLP& nlp, const BatchedOptions& options, int batch, const double* x0, int device)
    : B_(batch), n_(nlp.n), m_(nlp.m), zJ_((int)nlp.J_row1.size()), zH_((int)nlp.H_row1.size()), device_(device), opt_(options), nlp_(nlp) {
    if (batch <= 0 || n_ <= 0 || m_ < 0 || (int)nlp.x_l.size() != n_ || (int)nlp.x_u.size() != n_ || (int)nlp.c_l.size() != m_ ||
        (int)nlp.c_u.size() != m_ || (int)nlp.x_start.size() != n_ || (int)nlp.lam_start.size() != m_ || nlp.J_col1.size() != nlp.J_row1.size() ||
        nlp.H_col1.size() != nlp.H_row1.size())
        throw std::invalid_argument("BatchedAlgorithm: inconsistent model sizes");
    if (sqpb200_device_count() <= 0) throw std::runtime_error("BatchedAlgorithm: no CUDA device (there is no CPU path)");
    cuda_check(cudaSetDevice(device_), "cudaSetDevice");
    const size_t B = (size_t)B_, n = (size_t)n_, m = (size_t)m_, zJ = (size_t)zJ_, zH = (size_t)zH_;

    // the two QP handlers of Algorithm::initialization (src/Algorithm.cpp:561-562): one QP backend, one LP backend
    sqpb200_options o;
    sqpb200_default_options(&o);
    o.qp_maxiter = opt_.qp_maxiter; o.lp_maxiter = opt_.lp_maxiter;
    check(sqpb200_create(B_, n_ + 2 * m_, m_, SQPB200_QP, device_, &o, &qp_), "sqpb200_create(QP)");
    check(sqpb200_create(B_, n_ + 2 * m_, m_, SQPB200_LP, device_, &o, &lp_), "sqpb200_create(LP)");
    // structures: first set_A / set_H call of setupQP / setupLP (src/QPhandler.cpp:310-334; I_info_A_ of :41-51: A = [J I -I])
    const int irow[2] = {1, 1}, jcol[2] = {n_ + 1, n_ + m_ + 1}, size[2] = {m_, m_};
    const double value[2] = {1.0, -1.0};
    check(sqpb200_set_structure_A(qp_, zJ_, nlp.J_row1.data(), nlp.J_col1.data(), 2, irow, jcol, size, value), "set_structure_A(QP)");
    check(sqpb200_set_structure_H(qp_, zH_, nlp.H_row1.data(), nlp.H_col1.data(), 1), "set_structure_H(QP)");
    check(sqpb200_set_structure_A(lp_, zJ_, nlp.J_row1.data(), nlp.J_col1.data(), 2, irow, jcol, size, value), "set_structure_A(LP)");

    // the batched evaluator (SQPTNLP::Eval_*, src/SQPTNLP.cpp:67-132)
    char log[4096];
    log[0] = 0;
    if (sqpb200_nlp_compile(nlp.cuda_source.c_str(), n_, m_, zJ_, zH_, log, (int)sizeof log, &eval_) != 0)
        throw std::runtime_error(std::string("sqpb200_nlp_compile: ") + sqpb200_nlp_last_error() + "\n" + log);
    if (sqpb200_nlp_load(eval_, device_) != 0) throw std::runtime_error(std::string("sqpb200_nlp_load: ") + sqpb200_nlp_last_error());

    // ---- SoA state in one arena
    std::memset(&S_, 0, sizeof S_);
    Carver c;
    struct Slot { void** p; size_t off; };
    std::vector<Slot> slots;
    auto want = [&](void* field, size_t bytes) { slots.push_back({(void**)field, c.take(bytes ? bytes : 8)}); };
    const size_t d = sizeof(double);
    want(&S_.J_row1, zJ * 4); want(&S_.J_col1, zJ * 4); want(&S_.H_row1, zH * 4); want(&S_.H_col1, zH * 4);
    want(&S_.x_l, B * n * d); want(&S_.x_u, B * n * d); want(&S_.c_l, B * m * d); want(&S_.c_u, B * m * d);
    want(&S_.bound_type, B * n * 4); want(&S_.cons_type, B * m * 4);
    want(&S_.x_k, B * n * d); want(&S_.c_k, B * m * d); want(&S_.f_k, B * d); want(&S_.grad, B * n * d); want(&S_.jac, B * zJ * d);
    want(&S_.hess, B * zH * d); want(&S_.lam_c, B * m * d); want(&S_.lam_x, B * n * d); want(&S_.neg_lam, B * m * d);
    want(&S_.delta, B * d); want(&S_.rho, B * d); want(&S_.eps1, B * d); want(&S_.infea, B * d); want(&S_.p_k, B * n * d);
    want(&S_.x_trial, B * n * d); want(&S_.c_trial, B * m * d); want(&S_.f_trial, B * d); want(&S_.infea_trial, B * d);
    want(&S_.infea_model, B * d); want(&S_.infea_model_tmp, B * d); want(&S_.rho_trial, B * d); want(&S_.infea_infty, B * d);
    want(&S_.actual_red, B * d); want(&S_.pred_red, B * d); want(&S_.kkt_err, B * d);
    want(&S_.g_new, B * n * d); want(&S_.j_new, B * zJ * d); want(&S_.h_new, B * zH * d); want(&S_.scratch, B * n * d);
    want(&S_.exitflag, B * 4); want(&S_.iter, B * 4); want(&S_.pen_trial, B * 4); want(&S_.qp_iter, B * 8);
    want(&S_.active, B); want(&S_.need, B); want(&S_.go, B); want(&S_.acc, B); want(&S_.upd, B); want(&S_.feasible_lp, B); want(&S_.rej, B);
    want(&S_.counters, 8 * 4);
    want(&S_.soc_g, B * n * d); want(&S_.soc_x, B * n * d); want(&S_.soc_c, B * m * d); want(&S_.p_tmp, B * n * d);
    want(&S_.qp_obj_tmp, B * d); want(&S_.qp_obj_soc, B * d); want(&S_.norm_p, B * d);
    want(&S_.qp_inst, B * 8); want(&S_.lp_inst, B * 8);
    want(&f_tmp_, B * d); want(&c_tmp_, B * m * d);
    cuda_check(cudaMalloc(&arena_, c.off), "cudaMalloc(state arena)");
    cuda_check(cudaMemset(arena_, 0, c.off), "cudaMemset(state arena)");
    for (auto& s : slots) *s.p = (char*)arena_ + s.off;

    S_.B = B_; S_.n = n_; S_.m = m_; S_.zJ = zJ_; S_.zH = zH_;
    S_.iter_max = opt_.iter_max; S_.penalty_update = opt_.penalty_update ? 1 : 0; S_.penalty_iter_max = opt_.penalty_iter_max; S_.clear_flags = 0;
    S_.eta_c = opt_.eta_c; S_.eta_s = opt_.eta_s; S_.eta_e = opt_.eta_e; S_.gamma_c = opt_.gamma_c; S_.gamma_e = opt_.gamma_e;
    S_.delta_min = opt_.delta_min; S_.delta_max = opt_.delta_max; S_.tol = opt_.tol; S_.penalty_update_tol = opt_.penalty_update_tol;
    S_.rho_max = opt_.rho_max; S_.increase_parm = opt_.increase_parm; S_.eps1_change_parm = opt_.eps1_change_parm; S_.eps2 = opt_.eps2;
    S_.opt_prim_fea_tol = opt_.opt_prim_fea_tol; S_.opt_dual_fea_tol = opt_.opt_dual_fea_tol; S_.opt_compl_tol = opt_.opt_compl_tol;
    S_.opt_stat_tol = opt_.opt_stat_tol;
    S_.delta0 = opt_.delta; S_.rho0 = opt_.rho; S_.eps10 = opt_.eps1;

    // model data: the same row for every instance
    auto up = [&](const void* dst, const void* src, size_t bytes) {
        if (bytes) cuda_check(cudaMemcpy(const_cast<void*>(dst), src, bytes, cudaMemcpyHostToDevice), "cudaMemcpy(model)");
    };
    up(S_.J_row1, nlp.J_row1.data(), zJ * 4); up(S_.J_col1, nlp.J_col1.data(), zJ * 4);
    up(S_.H_row1, nlp.H_row1.data(), zH * 4); up(S_.H_col1, nlp.H_col1.data(), zH * 4);
    up(S_.x_l, tiled(nlp.x_l, B_).data(), B * n * d); up(S_.x_u, tiled(nlp.x_u, B_).data(), B * n * d);
    up(S_.c_l, tiled(nlp.c_l, B_).data(), B * m * d); up(S_.c_u, tiled(nlp.c_u, B_).data(), B * m * d);
    std::vector<int> bt(n), ct(m);
    for (int i = 0; i < n_; i++) bt[i] = constraint_class(nlp.x_l[i], nlp.x_u[i]);
    for (int i = 0; i < m_; i++) ct[i] = constraint_class(nlp.c_l[i], nlp.c_u[i]);
    up(S_.bound_type, tiled(bt, B_).data(), B * n * 4); up(S_.cons_type, tiled(ct, B_).data(), B * m * 4);

    // result buffers of the two backends
    void *bq[6], *bl[6];
    check(sqpb200_device_buffers(qp_, bq), "device_buffers(QP)");
    check(sqpb200_device_buffers(lp_, bl), "device_buffers(LP)");
    S_.qp_x = (const double*)bq[0]; S_.qp_y = (const double*)bq[1]; S_.qp_obj = (const double*)bq[2]; S_.qp_status = (const int*)bq[3];
    S_.qp_iters = (const int*)bq[4]; S_.qp_kkt = (const double*)bq[5];
    S_.lp_x = (const double*)bl[0]; S_.lp_status = (const int*)bl[3]; S_.lp_iters = (const int*)bl[4];

    initialization(x0);
}

BatchedAlgorithm::~BatchedAlgorithm() {
    cudaSetDevice(device_);
    cudaDeviceSynchronize();
    if (eval_) sqpb200_nlp_destroy(eval_);
    if (qp_) sqpb200_destroy(qp_);
    if (lp_) sqpb200_destroy(lp_);
    if (arena_) cudaFree(arena_);
}

// Algorithm::initialization (src/Algorithm.cpp:438-472): starting point shifted into its bounds (shift_starting_point,
// src/SQPTNLP.cpp:140-153), multipliers, f / c / gradient / Jacobian / Hessian at the start in one launch, then the per-instance
// state (infeasibility of the start, delta, rho, eps1, flags, backend state machines) by the SQPB200_PH_INIT phase
void BatchedAlgorithm::initialization(const double* x0) {
    const size_t B = (size_t)B_, n = (size_t)n_, m = (size_t)m_;
    std::vector<double> x(B * n);
    for (size_t b = 0; b < B; b++)
        for (size_t i = 0; i < n; i++) {
            double v = x0 ? x0[b * n + i] : nlp_.x_start[i];
            v = v > nlp_.x_l[i] ? v : nlp_.x_l[i];   // max(x, x_l)
            v = v < nlp_.x_u[i] ? v : nlp_.x_u[i];   // then min(., x_u)
            x[b * n + i] = v;
        }
    cuda_check(cudaMemcpy(S_.x_k, x.data(), B * n * 8, cudaMemcpyHostToDevice), "cudaMemcpy(x0)");
    if (m) {
        std::vector<double> lam = tiled(nlp_.lam_start, B_), neg(lam.size());
        for (size_t i = 0; i < lam.size(); i++) neg[i] = -lam[i];
        cuda_check(cudaMemcpy(S_.lam_c, lam.data(), B * m * 8, cudaMemcpyHostToDevice), "cudaMemcpy(lambda)");
        cuda_check(cudaMemcpy(S_.neg_lam, neg.data(), B * m * 8, cudaMemcpyHostToDevice), "cudaMemcpy(-lambda)");
    }
    if (sqpb200_nlp_eval(eval_, 1, B_, S_.x_k, S_.neg_lam, S_.f_k, S_.c_k, S_.grad, S_.jac, S_.hess, SQPB200_LOC_DEVICE, nullptr) != 0)
        throw std::runtime_error(std::string("sqpb200_nlp_eval: ") + sqpb200_nlp_last_error());
    S_.clear_flags = 0;
    check(sqpb200_sqp_phase(&S_, SQPB200_PH_INIT, nullptr, nullptr), "sqpb200_sqp_phase(INIT)");
    launches_ += 2;
    first_ = 1;
}

void BatchedAlgorithm::reset(const double* x0) {
    initialization(x0);
    check(sqpb200_reset(qp_), "sqpb200_reset(QP)");
    check(sqpb200_reset(lp_), "sqpb200_reset(LP)");
}

namespace {
// per-instance results [count] from device arrays
BatchedResult download(size_t count, size_t n, const double* x, const double* obj, const double* kkt, const double* rho, const double* delta,
                       const int* exitflag, const int* iter, const long long* qp_iter) {
    BatchedResult r;
    r.x.resize(count * n); r.obj.resize(count); r.KKT_error.resize(count); r.rho.resize(count); r.delta.resize(count);
    r.exitflag.resize(count); r.iter.resize(count); r.qp_iter.resize(count);
    auto down = [&](void* dst, const void* src, size_t bytes) { if (bytes) cuda_check(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost), "cudaMemcpy(result)"); };
    down(r.x.data(), x, count * n * 8); down(r.obj.data(), obj, count * 8); down(r.KKT_error.data(), kkt, count * 8);
    down(r.rho.data(), rho, count * 8); down(r.delta.data(), delta, count * 8);
    down(r.exitflag.data(), exitflag, count * 4); down(r.iter.data(), iter, count * 4); down(r.qp_iter.data(), qp_iter, count * 8);
    return r;
}
}  // namespace

BatchedResult BatchedAlgorithm::Optimize() {
    long long nl = 0;
    check(sqpb200_sqp_optimize(&S_, qp_, lp_, eval_, opt_.second_order_correction ? 1 : 0, /*refresh_ubA=*/1, &first_, f_tmp_, c_tmp_, &nl,
                               nullptr), "sqpb200_sqp_optimize");
    launches_ += nl;
    cuda_check(cudaDeviceSynchronize(), "cudaDeviceSynchronize");
    BatchedResult r = download(B_, n_, S_.x_k, S_.f_k, S_.kkt_err, S_.rho, S_.delta, S_.exitflag, S_.iter, S_.qp_iter);
    r.launches = launches_;
    return r;
}

BatchedResult BatchedAlgorithm::OptimizeStream(const double* x0_all, long long N, int refill_min, long long* rounds) {
    if (N < 0 || (N > 0 && !x0_all)) throw std::invalid_argument("OptimizeStream: no starting points");
    const size_t n = (size_t)n_, m = (size_t)m_, d = sizeof(double), Nz = (size_t)N, B = (size_t)B_;
    // inputs, results by instance and the queue in one arena
    Carver c;
    sqpb200_sqp_stream sd;
    std::memset(&sd, 0, sizeof sd);
    const size_t o_x0 = c.take(Nz * n * d), o_lam = c.take(m * d), o_x = c.take(Nz * n * d), o_obj = c.take(Nz * d), o_kkt = c.take(Nz * d),
                 o_rho = c.take(Nz * d), o_delta = c.take(Nz * d), o_ex = c.take(Nz * 4), o_it = c.take(Nz * 4), o_qi = c.take(Nz * 8),
                 o_slot = c.take(B * 8), o_head = c.take(8), o_refill = c.take(B);
    char* mem = nullptr;
    cuda_check(cudaMalloc((void**)&mem, c.off), "cudaMalloc(stream arena)");
    try {
        if (N > 0) cuda_check(cudaMemcpy(mem + o_x0, x0_all, Nz * n * d, cudaMemcpyHostToDevice), "cudaMemcpy(x0_all)");
        if (m) cuda_check(cudaMemcpy(mem + o_lam, nlp_.lam_start.data(), m * d, cudaMemcpyHostToDevice), "cudaMemcpy(lam_start)");
        sd.N = N;
        sd.refill_min = refill_min > 0 ? refill_min : (B_ / 16 > 0 ? B_ / 16 : 1);
        sd.x0_all = (const double*)(mem + o_x0); sd.lam_start = m ? (const double*)(mem + o_lam) : nullptr;
        sd.x = (double*)(mem + o_x); sd.obj = (double*)(mem + o_obj); sd.kkt_err = (double*)(mem + o_kkt); sd.rho = (double*)(mem + o_rho);
        sd.delta = (double*)(mem + o_delta); sd.exitflag = (int*)(mem + o_ex); sd.iter = (int*)(mem + o_it); sd.qp_iter = (long long*)(mem + o_qi);
        sd.slot_id = (long long*)(mem + o_slot); sd.head = (unsigned long long*)(mem + o_head); sd.refill = (unsigned char*)(mem + o_refill);
        long long nl = 0;
        check(sqpb200_sqp_optimize_stream(&S_, qp_, lp_, eval_, opt_.second_order_correction ? 1 : 0, /*refresh_ubA=*/1, &first_, f_tmp_, c_tmp_,
                                          &sd, &nl, nullptr), "sqpb200_sqp_optimize_stream");
        launches_ += nl;
        cuda_check(cudaDeviceSynchronize(), "cudaDeviceSynchronize");
        BatchedResult r = download(Nz, n, sd.x, sd.obj, sd.kkt_err, sd.rho, sd.delta, sd.exitflag, sd.iter, sd.qp_iter);
        r.launches = launches_;
        if (rounds) *rounds = sd.rounds;
        cudaFree(mem);
        return r;
    } catch (...) {
        cudaFree(mem);
        throw;
    }
}

}  // namespace sqpb200
