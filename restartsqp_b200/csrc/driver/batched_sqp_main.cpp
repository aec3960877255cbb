// batched_sqp_main.cpp -- command-line front end of the C++ batched driver, the counterpart of the reference's test/simple_test.cpp
// (:60-90: read a model, run Algorithm::Optimize, print exit flag / objective / iterations) for a batch of instances.
//
//   batched_sqp <model file> [--soc] [--iter-max K] [--repeat R] [--quiet] [--slots S [--refill-min K]]
//
// The model file is written by restartsqp_b200.nl_reader.write_model_file from a `.nl` file: sizes, bounds, starting point,
// sparsity patterns, B starting points and the CUDA source of the batched evaluator (numbers as C99 hex floats, so the hand-over
// is exact).  Output: one line per instance -- exitflag iter qp_iter obj x[0..n) -- with the doubles as hex floats, then a
// summary line with the solve time measured by CUDA events around Optimize().  --slots S: the B starting points are streamed
// through S instances (BatchedAlgorithm::OptimizeStream); the instance lines are the same, the summary adds the refill rounds.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>
#include <stdexcept>

#include "BatchedAlgorithm.hpp"

using namespace sqpb200;

namespace {

double next_double(std::istream& in) {
    std::string t;
    if (!(in >> t)) throw std::runtime_error("model file: unexpected end");
    if (t == "inf") return 1.0e19;
    if (t == "-inf") return -1.0e19;
    return std::strtod(t.c_str(), nullptr);  // accepts hex floats
}

template <typename T>
void read_ints(std::istream& in, std::vector<T>& v, size_t n) {
    v.resize(n);
    for (size_t i = 0; i < n; i++) if (!(in >> v[i])) throw std::runtime_error("model file: unexpected end");
}

void read_doubles(std::istream& in, std::vector<double>& v, size_t n) {
    v.resize(n);
    for (size_t i = 0; i < n; i++) v[i] = next_double(in);
}

}  // namespace

int main(int argc, char** argv) {
    if (argc < 2) {
        fprintf(stderr, "usage: %s <model file> [--soc] [--iter-max K] [--repeat R] [--quiet] [--slots S [--refill-min K]]\n", argv[0]);
        return 64;
    }
    BatchedOptions opt;
    int repeat = 1, slots = 0, refill_min = 0;
    bool quiet = false;
    for (int i = 2; i < argc; i++) {
        if (!strcmp(argv[i], "--soc")) opt.second_order_correction = true;
        else if (!strcmp(argv[i], "--iter-max") && i + 1 < argc) opt.iter_max = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--repeat") && i + 1 < argc) repeat = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--quiet")) quiet = true;
        else if (!strcmp(argv[i], "--slots") && i + 1 < argc) slots = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--refill-min") && i + 1 < argc) refill_min = atoi(argv[++i]);
    }
    if (slots < 0 || refill_min < 0) { fprintf(stderr, "batched_sqp: --slots and --refill-min take positive counts\n"); return 64; }
    try {
        std::ifstream file(argv[1]);
        if (!file) throw std::runtime_error(std::string("cannot open ") + argv[1]);
        std::stringstream ss;
        ss << file.rdbuf();
        const std::string all = ss.str();
        const std::string marker = "\n---SOURCE---\n";
        const size_t cut = all.find(marker);
        if (cut == std::string::npos) throw std::runtime_error("model file: no ---SOURCE--- marker");
        std::istringstream in(all.substr(0, cut));
        BatchedNLP nlp;
        nlp.cuda_source = all.substr(cut + marker.size());
        size_t zJ, zH, B;
        if (!(in >> nlp.n >> nlp.m >> zJ >> zH >> B)) throw std::runtime_error("model file: bad header");
        read_doubles(in, nlp.x_l, nlp.n); read_doubles(in, nlp.x_u, nlp.n); read_doubles(in, nlp.c_l, nlp.m); read_doubles(in, nlp.c_u, nlp.m);
        read_doubles(in, nlp.x_start, nlp.n); read_doubles(in, nlp.lam_start, nlp.m);
        read_ints(in, nlp.J_row1, zJ); read_ints(in, nlp.J_col1, zJ); read_ints(in, nlp.H_row1, zH); read_ints(in, nlp.H_col1, zH);
        std::vector<double> x0;
        read_doubles(in, x0, B * (size_t)nlp.n);

        // streamed: the slots start at the model's starting point; OptimizeStream gives each its first instance
        BatchedAlgorithm alg(nlp, opt, slots ? slots : (int)B, slots ? nullptr : x0.data());
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0); cudaEventCreate(&e1);
        BatchedResult r;
        float ms = 0.f;
        long long rounds = 0;
        for (int k = 0; k < repeat; k++) {
            if (k && !slots) alg.reset(x0.data());
            cudaEventRecord(e0, nullptr);
            r = slots ? alg.OptimizeStream(x0.data(), (long long)B, refill_min, &rounds) : alg.Optimize();
            cudaEventRecord(e1, nullptr);
            cudaEventSynchronize(e1);
            cudaEventElapsedTime(&ms, e0, e1);
        }
        cudaEventDestroy(e0); cudaEventDestroy(e1);
        size_t optimal = 0;
        for (size_t b = 0; b < B; b++) {
            optimal += r.exitflag[b] == 0;
            if (quiet) continue;
            printf("%d %d %lld %a", r.exitflag[b], r.iter[b], r.qp_iter[b], r.obj[b]);
            for (int i = 0; i < nlp.n; i++) printf(" %a", r.x[b * nlp.n + i]);
            printf("\n");
        }
        printf("summary instances %zu optimal %zu optimize_ms %.3f solves_per_s %.1f launches %lld", B, optimal, ms,
               ms > 0 ? 1000.0 * B / ms : 0.0, r.launches);
        if (slots) printf(" slots %d refill_rounds %lld", slots, rounds);
        printf("\n");
    } catch (const std::exception& e) {
        fprintf(stderr, "batched_sqp: %s\n", e.what());
        return strstr(e.what(), "no CUDA device") ? 2 : 1;
    }
    return 0;
}
