// oracle/algorithm_test.cpp -- TEST INFRASTRUCTURE.  The reference's OWN SQP loop -- src/Algorithm.cpp (initialization + Optimize),
// src/SQPTNLP.cpp and src/QPhandler.cpp, unmodified except for integration/restartsqp_cuda_backend.patch -- run on one instance of
// a model with the CUDA plugin as its QP / LP backend, the way test/simple_test.cpp:72-84 runs it with an AmplTNLP.  Ipopt and ASL
// are absent, so the NLP comes in as an Ipopt::TNLP (stand-in header of oracle/stubs_link, Ipopt's published callback signatures)
// over the C evaluator that restartsqp_b200/nl_reader.py generates from the `.nl` file (the same arithmetic the oracle of the loop,
// oracle/oracle_sqp.c, evaluates): this is what PINS that oracle -- and through it the device-resident loop -- against the
// reference's real Algorithm::Optimize.
//
//   algorithm_nl[_twin] <model file> <evaluator .so> <instance> [qore] [soc]
// Default backend: the patched Options default, CUDA_B200 (CudaQPInterface through QPhandler's non-QORE branches, which leave ubA
// stale after the first iteration: SURVEY.md 8a quirk 2).  `qore`: CUDA_B200_QORE_LAYOUT (CudaQOREInterface through QPhandler's QORE
// branches, which refresh both constraint sides -- the reference's own default backend is QORE, src/Options.cpp:24-25).
//
// model file: restartsqp_b200.nl_reader.write_model_file (sizes, bounds, start, patterns, starting points as hex floats);
// evaluator: the library oracle_py.SqpOracle compiled for the model (its `evaluator` path; nlp_fc, nlp_all).  Output: exitflag iter qp_iter obj x..., doubles as hex floats.
#include <dlfcn.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

#define private public  // the reference keeps its iterate private and offers no getter; the test reads Algorithm::x_k_
#include <sqphot/Algorithm.hpp>
#undef private

using namespace SQPhotstart;

typedef void (*nlp_fc_t)(const double* x, double* f, double* c);
typedef void (*nlp_all_t)(const double* x, const double* lam, double* f, double* c, double* grad, double* jac, double* hess);

static double next_double(std::istream& in) {
    std::string t;
    in >> t;
    if (t == "inf") return 1.0e19;
    if (t == "-inf") return -1.0e19;
    return strtod(t.c_str(), nullptr);
}

struct Model {
    int n = 0, m = 0;
    std::vector<double> x_l, x_u, c_l, c_u, x_start, lam_start;
    std::vector<int> J_row1, J_col1, H_row1, H_col1;
};

class NlTNLP : public Ipopt::TNLP {
public:
    NlTNLP(const Model& md, nlp_fc_t fc, nlp_all_t all) : md_(md), fc_(fc), all_(all), c_(md.m + 1), g_(md.n + 1), j_(md.J_row1.size() + 1),
                                                           h_(md.H_row1.size() + 1), zero_(md.m + 1, 0.0) {}
    bool get_nlp_info(Ipopt::Index& n, Ipopt::Index& m, Ipopt::Index& nnz_jac_g, Ipopt::Index& nnz_h_lag, IndexStyleEnum& index_style) override {
        n = md_.n; m = md_.m; nnz_jac_g = (int)md_.J_row1.size(); nnz_h_lag = (int)md_.H_row1.size(); index_style = FORTRAN_STYLE;
        return true;
    }
    bool get_bounds_info(Ipopt::Index n, double* x_l, double* x_u, Ipopt::Index m, double* g_l, double* g_u) override {
        for (int i = 0; i < n; i++) { x_l[i] = md_.x_l[i]; x_u[i] = md_.x_u[i]; }
        for (int i = 0; i < m; i++) { g_l[i] = md_.c_l[i]; g_u[i] = md_.c_u[i]; }
        return true;
    }
    bool get_starting_point(Ipopt::Index n, bool, double* x, bool, double*, double*, Ipopt::Index m, bool, double* lambda) override {
        for (int i = 0; i < n; i++) x[i] = md_.x_start[i];
        if (lambda) for (int i = 0; i < m; i++) lambda[i] = md_.lam_start[i];
        return true;
    }
    bool eval_f(Ipopt::Index, const double* x, bool, double& obj) override { fc_(x, &obj, c_.data()); return true; }
    bool eval_g(Ipopt::Index, const double* x, bool, Ipopt::Index m, double* g) override {
        double f; fc_(x, &f, c_.data());
        for (int i = 0; i < m; i++) g[i] = c_[i];
        return true;
    }
    bool eval_grad_f(Ipopt::Index n, const double* x, bool, double* grad) override {
        double f; all_(x, zero_.data(), &f, c_.data(), g_.data(), j_.data(), h_.data());
        for (int i = 0; i < n; i++) grad[i] = g_[i];
        return true;
    }
    bool eval_jac_g(Ipopt::Index, const double* x, bool, Ipopt::Index, Ipopt::Index nele, Ipopt::Index* iRow, Ipopt::Index* jCol, double* values) override {
        if (!values) { for (int k = 0; k < nele; k++) { iRow[k] = md_.J_row1[k]; jCol[k] = md_.J_col1[k]; } return true; }
        double f; all_(x, zero_.data(), &f, c_.data(), g_.data(), j_.data(), h_.data());
        for (int k = 0; k < nele; k++) values[k] = j_[k];
        return true;
    }
    bool eval_h(Ipopt::Index, const double* x, bool, double, Ipopt::Index, const double* lambda, bool, Ipopt::Index nele, Ipopt::Index* iRow,
                Ipopt::Index* jCol, double* values) override {
        if (!values) { for (int k = 0; k < nele; k++) { iRow[k] = md_.H_row1[k]; jCol[k] = md_.H_col1[k]; } return true; }
        double f; all_(x, lambda ? lambda : zero_.data(), &f, c_.data(), g_.data(), j_.data(), h_.data());  // obj_factor is 1 at both call sites
        for (int k = 0; k < nele; k++) values[k] = h_[k];
        return true;
    }
private:
    Model md_;
    nlp_fc_t fc_;
    nlp_all_t all_;
    std::vector<double> c_, g_, j_, h_, zero_;
};

int main(int argc, char** argv) {
    if (argc < 4) { fprintf(stderr, "usage: %s <model file> <evaluator .so> <instance> [qore] [soc]\n", argv[0]); return 64; }
    const int inst = atoi(argv[3]);
    bool qore = false, soc = false;
    for (int i = 4; i < argc; i++) { qore |= !strcmp(argv[i], "qore"); soc |= !strcmp(argv[i], "soc"); }
    std::ifstream file(argv[1]);
    std::stringstream ss; ss << file.rdbuf();
    std::string all = ss.str();
    size_t cut = all.find("\n---SOURCE---\n");
    std::istringstream in(all.substr(0, cut));
    Model md;
    size_t zJ, zH, B;
    in >> md.n >> md.m >> zJ >> zH >> B;
    auto rd = [&](std::vector<double>& v, size_t k) { v.resize(k); for (size_t i = 0; i < k; i++) v[i] = next_double(in); };
    auto ri = [&](std::vector<int>& v, size_t k) { v.resize(k); for (size_t i = 0; i < k; i++) in >> v[i]; };
    rd(md.x_l, md.n); rd(md.x_u, md.n); rd(md.c_l, md.m); rd(md.c_u, md.m); rd(md.x_start, md.n); rd(md.lam_start, md.m);
    ri(md.J_row1, zJ); ri(md.J_col1, zJ); ri(md.H_row1, zH); ri(md.H_col1, zH);
    std::vector<double> x0; rd(x0, B * md.n);
    if (inst < 0 || (size_t)inst >= B) { fprintf(stderr, "instance out of range\n"); return 64; }
    for (int i = 0; i < md.n; i++) md.x_start[i] = x0[(size_t)inst * md.n + i];
    void* so = dlopen(argv[2], RTLD_NOW);
    if (!so) { fprintf(stderr, "dlopen: %s\n", dlerror()); return 65; }
    nlp_fc_t fc = (nlp_fc_t)dlsym(so, "nlp_fc");
    nlp_all_t al = (nlp_all_t)dlsym(so, "nlp_all");
    if (!fc || !al) { fprintf(stderr, "evaluator symbols missing\n"); return 65; }
    try {
        Algorithm alg;
        Ipopt::SmartPtr<Ipopt::TNLP> nlp = new NlTNLP(md, fc, al);
        alg.initialization(nlp, argv[1]);
        if (qore) {  // Algorithm creates its Options and its two QPhandlers itself (src/Algorithm.cpp:558-562): swap them before the first QP
            alg.options_->QPsolverChoice = alg.options_->LPsolverChoice = CUDA_B200_QORE_LAYOUT;
            alg.myQP_ = make_shared<QPhandler>(alg.nlp_->nlp_info_, QP, alg.jnlst_, alg.options_);
            alg.myLP_ = make_shared<QPhandler>(alg.nlp_->nlp_info_, LP, alg.jnlst_, alg.options_);
        }
        if (soc) alg.options_->second_order_correction = true;  // off by default, src/Options.cpp:26
        alg.Optimize();
        printf("%d %d %d %a", (int)alg.get_exit_flag(), alg.get_stats()->iter, alg.get_stats()->qp_iter, alg.get_final_objective());
        for (int i = 0; i < md.n; i++) printf(" %a", alg.x_k_->values(i));
        printf("\n");
    } catch (QP_INTERNAL_ERROR& e) {
        printf("create_failed %s\n", e.Message().c_str());
        return 2;
    } catch (Ipopt::IpoptException& e) {
        printf("exception %s\n", e.Message().c_str());
        return 3;
    }
    return 0;
}
