// BatchedAlgorithm.hpp -- the batched mode of the host C++ driver: the counterpart of the reference's `Algorithm`
// (include/sqphot/Algorithm.hpp:30-140, src/Algorithm.cpp) for `batch` independent NLP instances of one model.
//
// Where Algorithm keeps one x_k / delta / rho / exit flag, this class keeps [batch][...] SoA arrays in device memory (one arena) and
// never brings an iterate back to the host before the end: initialization() (src/Algorithm.cpp:438-472) is one batched NLP
// evaluation plus one state kernel, Optimize() (:55-168) is one call of sqpb200_sqp_optimize, which sequences the per-instance
// phases, the QP data updates, the QP / LP solves of the still-active instances and the NLP evaluations on one stream.  The class
// only talks to the C ABI of libsqpb200.so (include/sqpb200.h) and to the CUDA runtime for its own memory; it is the C++ twin
// of restartsqp_b200/sqp_device.py (tests/test_gpu_driver.py compares the two bit for bit).
//
// The model arrives as a BatchedNLP: sizes, bounds, starting point and sparsity patterns (what SQPTNLP::Get_nlp_info /
// Get_bounds_info / Get_starting_point / Get_Structure_* return, src/SQPTNLP.cpp:13-65) plus the CUDA source of its batched
// evaluator (compiled with NVRTC through sqpb200_nlp_compile; restartsqp_b200/nl_reader.py generates it from a `.nl` file).
#ifndef SQPB200_BATCHED_ALGORITHM_HPP
#define SQPB200_BATCHED_ALGORITHM_HPP

#include <string>
#include <vector>

#include <sqpb200.h>

namespace sqpb200 {

/** Options::setToDefault, src/Options.cpp:19-57 (the entries the batched loop reads). */
struct BatchedOptions {
    int iter_max = 1000, qp_maxiter = 1000, lp_maxiter = 100, penalty_iter_max = 200;
    bool penalty_update = true, second_order_correction = false;
    double eta_c = 0.25, eta_s = 1.0e-8, eta_e = 0.75, gamma_c = 0.5, gamma_e = 2.0;
    double delta = 1.0, delta_min = 1.0e-16, delta_max = 1.0e8;
    double opt_stat_tol = 1.0e-4, opt_compl_tol = 1.0e-4, opt_dual_fea_tol = 1.0e-4, opt_prim_fea_tol = 1.0e-4;
    double tol = 1.0e-8, penalty_update_tol = 1.0e-8, rho = 1.0, increase_parm = 10.0, rho_max = 1.0e6;
    double eps1 = 0.1, eps1_change_parm = 0.1, eps2 = 1.0e-6;
};

struct BatchedNLP {
    int n = 0, m = 0;                                   // NLPInfo nVar / nCon (include/sqphot/Types.hpp:100-105)
    std::vector<double> x_l, x_u, c_l, c_u;             // Get_bounds_info
    std::vector<double> x_start, lam_start;             // Get_starting_point (lam_start: constraint multipliers, m entries)
    std::vector<int> J_row1, J_col1, H_row1, H_col1;    // Get_Structure_Jacobian / _Hessian, 1-based triplets
    std::string cuda_source;                            // batched evaluator kernels for sqpb200_nlp_compile
};

/** Per-instance results (the getters of include/sqphot/Algorithm.hpp:70-100, one entry per instance). */
struct BatchedResult {
    std::vector<double> x;             // [batch][n] final iterates
    std::vector<double> obj;           // get_final_objective
    std::vector<double> KKT_error, rho, delta;
    std::vector<int> exitflag;         // get_exit_flag (Exitflag values; SQPB200_EXIT_QP_UNCHANGED = 7 in addition)
    std::vector<int> iter;             // Stats::iter
    std::vector<long long> qp_iter;    // Stats::qp_iter
    long long launches = 0;            // kernels launched by the loop
};

class BatchedAlgorithm {
public:
    /** x0: [batch][n] starting points (nullptr: every instance starts at nlp.x_start).  Throws std::runtime_error when the library
     *  reports an error (no CUDA device: there is no CPU path). */
    BatchedAlgorithm(const BatchedNLP& nlp, const BatchedOptions& options, int batch, const double* x0 = nullptr, int device = 0);
    ~BatchedAlgorithm();
    BatchedAlgorithm(const BatchedAlgorithm&) = delete;
    BatchedAlgorithm& operator=(const BatchedAlgorithm&) = delete;

    /** Algorithm::initialization for a new batch on the same object: handles, buffers and the compiled evaluator are kept. */
    void reset(const double* x0);
    /** Algorithm::Optimize for every instance. */
    BatchedResult Optimize();
    /** Algorithm::Optimize for N starting points x0_all[N][n] (host memory) streamed through the batch's instances as slots
     *  (sqpb200_sqp_optimize_stream): a slot whose instance has stopped takes the next starting point on the device.  Returns N
     *  entries in input order, each what one batch over all N gives.  refill_min: stopped slots that trigger a refill round
     *  (<= 0: batch / 16, at least 1).  rounds (if not null) receives the number of refill rounds, the initial fill included. */
    BatchedResult OptimizeStream(const double* x0_all, long long N, int refill_min = 0, long long* rounds = nullptr);

    int get_num_var() const { return n_; }
    int get_num_constr() const { return m_; }
    int get_batch() const { return B_; }

private:
    void initialization(const double* x0);
    void check(int rc, const char* what) const;

    int B_, n_, m_, zJ_, zH_, device_;
    BatchedOptions opt_;
    BatchedNLP nlp_;
    sqpb200_handle qp_ = nullptr, lp_ = nullptr;
    sqpb200_nlp eval_ = nullptr;
    sqpb200_sqp_state S_;
    void* arena_ = nullptr;
    double *f_tmp_ = nullptr, *c_tmp_ = nullptr;
    int first_ = 1;
    long long launches_ = 0;
};

}  // namespace sqpb200
#endif
