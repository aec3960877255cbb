// qp_kernel.cuh -- batched FP64 active-set QP/LP solver for sm_100a (row D of SURVEY.md 8a).
//
// One solver template, QPT<TEAM>, three ways to run it:
//   * TEAM = 32: one QP per warp, a CTA hosts CTA_THREADS/32 QPs (qp_solve_kernel);
//   * TEAM = 16 / 8: sub-warp teams for QPs with nV <= 16 / <= 8 (two / four QPs per warp, team-masked barriers and shuffles);
//   * TEAM = 512: one QP per thread-block cluster (qp_solve_large_kernel, QPs too large for shared memory): the slice lives in
//     global memory, rank 0 of the cluster runs the method and the other CTAs take their share of the refactorisation (TMA-staged
//     FP64 DMMA tiles) and of the large O(n^2) primitives; the projected Cholesky factor is carried through additions.
// For TEAM <= 32 everything a QP needs for the whole solve lives in the team's slice of shared memory: the factors (Q of the
// TQ factorisation; T and the projected Cholesky factor R packed into one array), current and target homotopy data, iterate and
// work vectors, matrix values and the working-set index lists.  The sparsity pattern (shared by the batch) is staged once per
// CTA as 16-bit indices, and the launch arguments are copied to static shared memory, so the solver's
// out-of-line functions carry no per-thread state at all: no local-memory traffic, no global loads inside
// the active-set loop.  HBM is touched only for the compulsory input (matrix values, g, bounds), the output
// (x, y, working set, status, KKT residuals) and, for hot starts, one save/restore of the slice.
//
// The algorithm is the online active-set strategy as the reference drives it through qpOASES
// (call sites src/qpOASESInterface.cpp:155-206, 231-268, 221-222, 843-844, options :765): same
// steps, thresholds and tie-breaks as the CPU oracle (oracle/oracle_qp.c), which is only a
// checker and is never called from here.  The library is compiled with -fmad=false and every sum
// below runs in the oracle's order, so the results of the warp and sub-warp kernels are bit-identical with the oracle (the
// cluster kernel sums on the tensor cores and updates its factor: same working sets, 1e-8).
//
// Parallelisation inside the warp (32 lanes):
//   * sparse products: one lane per output entry (CSC columns for H and A', a CSR view for A),
//     accumulation in storage order (= the reference's SpHbMat::times order);
//   * Givens sweeps: the rotation chain is a scalar recurrence; every lane applies the whole
//     chain to its own rows of Q / T, so the sweep needs no barrier per rotation when the
//     chain is known up front (additions), and one barrier per rotation otherwise (removals);
//   * triangular solves: column-oriented substitution, lanes over the trailing vector;
//   * projected Hessian + Cholesky: one sparse product per null-space column, row-wise Cholesky
//     with lanes over the columns of the current row;
//   * ratio tests: lane-local scan in index order + (ratio, position) lexicographic min reduction,
//     which reproduces the sequential "first index wins ties" rule.
//
// A multi-warp-per-QP variant inside one CTA (named-barrier teams of 64..256 threads) was prototyped in round 1; with
// out-of-line functions CTA-level barriers lost synchronisation intermittently on sm_100a / CUDA 12.9 and
// the inlined build deadlocked at large grids, so between the warp and the whole CTA there is no intermediate team size.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "tma.cuh"

namespace sqpb200 {

#define QP_EPS 2.221e-16
#define QP_INFTY 1.0e20
#define QP_ZERO 1.0e-25
#define QP_BOUND_RELAX 1.0e4
#define QP_EPS_NUM (-1.0e3 * QP_EPS)
#define QP_EPS_DEN (1.0e3 * QP_EPS)
#define QP_EPS_FLIP (1.0e3 * QP_EPS)
#define QP_EPS_REG (1.0e3 * QP_EPS)
#define QP_EPS_LI (1.0e5 * QP_EPS)

enum { ST_OPTIMAL = 20, ST_INTERNAL = 21, ST_INFEASIBLE = 22, ST_UNBOUNDED = 23, ST_NOTINIT = 25, ST_HOMOTOPY = 28,
       ST_CAPACITY = 31 /* internal: factor capacity exceeded, instance is re-solved by the rescue launch */ };
enum { MODE_COLD = 0, MODE_HOT_FIXED = 1, MODE_HOT_VARIED = 2,
       MODE_REINIT = 3 /* FIXED <-> VARIED flip of the matrix status: init from the previous solution (src/qpOASESInterface.cpp:202-207) */ };
enum { FLAG_FLIPPING = 1, FLAG_RAMPING = 2, FLAG_DRIFT = 4, FLAG_KEEP_STATE = 8,
       FLAG_FORCE_GUESS = 16 /* test hook: take handle_error's infeasible branch whatever the first attempt returned */,
       FLAG_NO_CARRY = 32 /* one-QP-per-cluster kernel: recompute R after every addition (as the warp kernel does) instead of updating it */ };

struct QPKernelArgs {
    int batch, nV, nC;
    int cap, ld;      // factor capacity (max simultaneously free variables) and its odd leading dimension
    int large;        // 1: one-QP-per-CTA layout (adds the nFR x nZ scratch matrix W of the blocked refactorisation)
    int rescue;       // 1: only instances whose status is ST_CAPACITY are (re)solved, from their pre-solve state
    int is_lp, has_H;
    int max_iter, flags, mode;
    int zA, zH;
    // shared sparsity pattern (global memory; staged once per CTA into shared memory as 16-bit indices)
    const int *Ap, *Ai;            // CSC of A (nC x nV)
    const int *Arp, *Aci, *Aperm;  // CSR view of A: rowptr, column index, position in the CSC value array
    const int *Hp, *Hi;            // CSC of H (nV x nV, full symmetric)
    // per-instance inputs, instance-major
    const double *Aval, *Hval;
    const double *gN, *lbN, *ubN, *lbAN, *ubAN;
    const unsigned char* mask;
    signed char* inst_state;  // optional [batch][8]: per-instance init/hotstart state machine {first_solved, varied, old_ms, new_ms, last_mode}
    const int* gpat;   // TEAM > 32: the pattern as 32-bit indices in global memory, laid out by the p* offsets below
    double* gwork;     // TEAM > 32: [batch][slice_doubles] global-memory slices (persist between solves: hot start in place)
    // outputs
    double *x, *y, *obj, *kkt;
    int *status, *iters;
    long long* prof;         // optional [16] cycle counters per solver phase (filled only by -DQP_PROFILE builds)
    signed char *wsB, *wsC;  // raw working set (+1 upper, -1 lower, 0 inactive)
    int *WB, *WC;            // translated ActiveType
    // resident hot-start state: [batch][state_doubles]: the slice without its factors, then Q, R, T packed
    double* state;
    int state_doubles;
    int slice_doubles;  // doubles per QP slice
    int pat_shorts;     // 16-bit words of the staged pattern
    // slice layout: offsets in doubles from the slice base (filled by qp_fill_layout)
    int oQ, oRT, ox, og, olb, oub, odx, oAx, olbA, oubA, odAx, oy, ody, ot1, ot2, ot3, ow, oa, oyv, ozv, oAv, oHv;
    int ogN, olbN, oubN, olbAN, oubAN;  // target data of the homotopy
    int oW;                             // large layout only: scratch matrix (cap x ld)
    int oP;                             // end of the persistent part of the slice (what a hot start restores)
    int nW;                             // doubles from ot1 to the end of zv (chunk buffer of the warp kernel's refactorisation)
    int *ncap, *caplist;                // instances whose solve overflowed the factor capacity (count, list[batch]): the rescue launch's work list
    int* maxfr;                         // optional: running maximum of free variables seen by this handle (atomicMax)
    int oS;                             // start of the 16-bit index arrays (sB, FR, posFR, sC, AC, posAC)
    // pattern layout: offsets in 16-bit words from the pattern base
    int pAp, pAi, pArp, pAci, pAperm, pHp, pHi;
};

// Slice layout of one QP in shared memory.  Header (4 doubles = 8 ints): nFR, nAC, ramp_offset, initialised, then (cluster build of
// the one-QP-per-CTA kernel) the command and status words the leader CTA shares with its helper CTAs.
// The factors come last and are sized by the capacity `cap` <= nV (the number of simultaneously free variables
// stays far below nV on l1-penalty QPs: most slacks sit at zero), which is what sets the occupancy.
__host__ __device__ inline void qp_fill_layout(QPKernelArgs& a) {
    const int nV = a.nV, nC = a.nC, nT = nV + nC;
    if (a.cap <= 0 || a.cap > nV) a.cap = nV;
    // warp kernel: odd leading dimension (conflict-free row and column walks in shared memory); one-QP-per-CTA kernel: the
    // factors live in global memory and their rows are the source of 16-byte aligned TMA bulk copies -> multiple of 8 doubles
    a.ld = a.large ? ((a.cap + 7) & ~7) : ((a.cap % 2 == 0) ? a.cap + 1 : a.cap);
    int o = a.large ? 8 : 4;  // one-QP-per-CTA kernel: 8 more ints for the arguments of the operations the leader hands to its cluster
    // persistent part = the hot-start image (independent of the factor capacity): iterate, current homotopy data, matrix
    // values, working-set index lists
    a.ox = o; o += nV; a.og = o; o += nV; a.olb = o; o += nV; a.oub = o; o += nV;
    a.oAx = o; o += nC; a.olbA = o; o += nC; a.oubA = o; o += nC;
    a.oy = o; o += nT;
    a.oAv = o; o += a.zA; a.oHv = o; o += a.zH;
    a.oS = o;
    const int shorts = 3 * nV + 3 * nC;
    o += (shorts * 2 + 7) / 8;
    a.oP = o;
    // per-solve part: homotopy targets and work vectors, each sized by its use (the slice size sets the occupancy)
    const int mx_vc = nV > nC ? nV : nC, mx_cc = nC > a.cap ? nC : a.cap;
    a.odx = o; o += nV; a.ogN = o; o += nV; a.olbN = o; o += nV; a.oubN = o; o += nV;
    a.odAx = o; o += nC; a.olbAN = o; o += nC; a.oubAN = o; o += nC;
    a.ody = o; o += nT;
    a.ot1 = o; o += nV; a.ot2 = o; o += mx_vc; a.ot3 = o; o += mx_cc; a.ow = o; o += nT; a.oa = o; o += nV;
    a.oyv = o; o += a.cap; a.ozv = o; o += a.cap;
    a.nW = o - a.ot1;  // t1 .. zv are contiguous and dead during a refactorisation: its chunk buffer
    if (a.large) o = (o + 15) & ~15;  // 128-byte aligned factor rows
    a.oQ = o; o += a.cap * a.ld;
    a.oRT = o; o += a.cap * a.ld;
    a.oW = o; if (a.large) o += a.cap * a.ld;
    if (a.large) o = (o + 15) & ~15;
    a.slice_doubles = o;
    a.state_doubles = a.oP + 2 * nV * nV;  // capacity-independent image: persistent part, then Q, R, T packed
    int p = 0;
    a.pAp = p; p += nV + 1; a.pAi = p; p += a.zA; a.pArp = p; p += nC + 1; a.pAci = p; p += a.zA; a.pAperm = p; p += a.zA;
    a.pHp = p; p += nV + 1; a.pHi = p; p += a.zH;
    a.pat_shorts = (p + 3) & ~3;
}

#ifdef __CUDACC__

// launch arguments, copied once per CTA; every out-of-line function reads its context from here
__shared__ QPKernelArgs sA;
extern __shared__ __align__(128) double qp_smem[];

struct MinKey {
    double t;
    int pos;
};
__device__ __forceinline__ bool key_less(double t1, int p1, double t2, int p2) { return t1 < t2 || (t1 == t2 && p1 < p2); }

// x / d from the reciprocal ri = 1/d (formed in parallel ahead of a substitution chain) with one Newton correction: three
// dependent operations on the critical path instead of a full division.  Same sequence as the oracle's quot(); a bare x*ri is
// not accurate enough (the rho = 1e8 scaled dumps then need 3x the iterations).
__device__ __forceinline__ double quot(double x, double d, double ri) {
    const double q0 = x * ri;
    const double r = __fma_rn(-q0, d, x);
    return __fma_rn(r, ri, q0);
}

#define QP_FN __noinline__
// loop unrolling of the solver's loops: 1 = smallest code (10.6 k SASS instructions).  Measured with unroll 4 (59 k
// instructions): 1.3x-3x slower on every dumped QP (instruction-cache misses), so 1 is what ships.
#define QP_U1 _Pragma("unroll 1")
// Phase timers of a -DQP_PROFILE build (tools/large_try.py, tools/per_fixture.py print them): the first thread of every team adds
// the clock64() cycles it spent in phase i to A.prof[i].  Phase boundaries are team barriers, so one thread's clock is the team's.
#ifdef QP_PROFILE
#define PROF_T0 long long prof_t0_ = clock64();
#define PROF_RESET prof_t0_ = clock64();
#define PROF2_T0 long long prof_t2_ = clock64();
#define PROF2_ADD(i) do { long long t_ = clock64(); if (lane == 0 && sA.prof) atomicAdd((unsigned long long*)&sA.prof[i], (unsigned long long)(t_ - prof_t2_)); prof_t2_ = t_; } while (0)
#define PROF_ADD(i) do { long long t_ = clock64(); if (lane == 0 && sA.prof) atomicAdd((unsigned long long*)&sA.prof[i], (unsigned long long)(t_ - prof_t0_)); prof_t0_ = t_; } while (0)
#else
#define PROF_T0
#define PROF_RESET
#define PROF2_T0
#define PROF2_ADD(i) do { } while (0)
#define PROF_ADD(i) do { } while (0)
#endif
enum { PR_STEPDIR = 0, PR_RATIO = 1, PR_STEP = 2, PR_REMOVE = 3, PR_EXTEND = 4, PR_WVEC = 5, PR_ADD = 6, PR_REFAC_W = 7, PR_REFAC_M = 8,
       PR_REFAC_CHOL = 9, PR_DRIFT = 10, PR_ENSURE_LI = 11, PR_RSOLVE = 12, PR_SETUP = 13, PR_EPILOGUE = 14, PR_TOTAL = 15 };

// TEAM = threads that cooperate on one QP.  <= 32: one warp (TEAM = 32) or a sub-warp team of 16 / 8 lanes per QP (QPs with
// nV <= 16 / <= 8: a 5-variable QP keeps 5 of 32 lanes busy, so two or four of them share a warp; each team synchronises with
// its own lane mask and the teams of a warp may diverge freely), everything in the team's shared-memory slice, pattern
// staged as 16-bit indices.  > 32: the whole CTA works on one QP (large QPs, SURVEY 8d config 4); the slice lives in
// global memory (sSlice; factors streamed through L1/L2), the pattern is read as 32-bit indices from global memory and
// the team barrier is __syncthreads().
template <int TEAM> struct PatIdx { typedef int type; };
template <> struct PatIdx<32> { typedef short type; };
template <> struct PatIdx<16> { typedef short type; };
template <> struct PatIdx<8> { typedef short type; };
// lane mask of the calling team inside its warp (TEAM <= 32)
template <int TEAM> __device__ __forceinline__ unsigned team_mask() {
    if (TEAM >= 32) return 0xffffffffu;
    return ((1u << (TEAM & 31)) - 1u) << ((threadIdx.x & 31) & ~(TEAM - 1));
}
__shared__ double* sSlice;     // TEAM > 32: this CTA's slice in global memory
__shared__ int sClusterSize;   // TEAM > 32: CTAs that share this QP (thread-block cluster), 1 without a cluster launch
__shared__ uint32_t sPhase;    // TEAM > 32: phase bits of the TMA ring's mbarriers
__shared__ __align__(8) uint64_t sFull[3];  // TEAM > 32: "stage filled" mbarriers of the TMA ring
__shared__ double sRedT[32];   // TEAM > 32: scratch of the team-wide min reduction
__shared__ int sRedP[32];

// Context of the calling team.  hdr: [0]=nFR [1]=nAC [2]=ramp_offset [3]=initialised.
#define QP_CTX                                                                                     \
    const int lane = (TEAM <= 32) ? (int)(threadIdx.x & (TEAM - 1)) : (int)threadIdx.x;            \
    double* const slice = (TEAM <= 32) ? qp_smem + (size_t)(threadIdx.x / TEAM) * sA.slice_doubles : sSlice; \
    int* const hdr = reinterpret_cast<int*>(slice);                                                \
    const int nV = sA.nV, nC = sA.nC, ld = sA.ld, cap = sA.cap;                                    \
    (void)lane; (void)hdr; (void)nV; (void)nC; (void)ld; (void)cap;
#define QP_PAT                                                                                     \
    const pidx* const pat = (TEAM <= 32)                                                           \
        ? reinterpret_cast<const pidx*>(qp_smem + (size_t)(blockDim.x / TEAM) * sA.slice_doubles) \
        : reinterpret_cast<const pidx*>(sA.gpat);

#define V_(name) (slice + sA.o##name)
#define S_(k) (reinterpret_cast<short*>(slice + sA.oS) + (k))
#define sB_ S_(0)
#define FR_ S_(nV)
#define posFR_ S_(2 * nV)
#define sC_ S_(3 * nV)
#define AC_ S_(3 * nV + nC)
#define posAC_ S_(3 * nV + 2 * nC)
#define R_(a_, b_) RT[(a_) * ld + (b_)]
#define T_(i, j) RT[(cap - 1 - (i)) * ld + (j)]
// inner sequential sums: not unrolled in the warp kernel (instruction-cache footprint), unrolled 8x in the CTA kernel so
// that the loads of consecutive terms overlap (the additions stay in order: no reassociation without fast-math)
#define DOT_UNROLL _Pragma("unroll (TEAM <= 32 ? 1 : 8)")
#define SYNC() do { if (TEAM <= 32) __syncwarp(team_mask<TEAM>()); else __syncthreads(); } while (0)

template <int TEAM>
struct QPT {
    typedef typename PatIdx<TEAM>::type pidx;
    // ---------------------------------------------------------------- sparse products
    // One entry of each product, summed in storage order.  The mul* functions below run one lane per entry and end in a
    // barrier; the fused phases (step_direction, drift_correction, ramping, ensure_li) call these directly so that an entry
    // is formed by the lane that consumes it, with the same terms in the same order.
    static __device__ __forceinline__ double H_row(const pidx* pat, const double* Hv, const double* v, int c) {  // ((H + reg I) v)[c]
        const pidx *Hp = pat + sA.pHp, *Hi = pat + sA.pHi;
        const double reg = sA.is_lp ? QP_EPS_REG : 0.0;
        double s = 0.0;
        if (sA.has_H && !sA.is_lp) {
            int e1 = Hp[c + 1];
            QP_U1 for (int e = Hp[c]; e < e1; e++) s += Hv[e] * v[Hi[e]];
        }
        if (reg != 0.0) s += reg * v[c];
        return s;
    }
    static __device__ __forceinline__ double A_row(const pidx* pat, const double* Av, const double* v, int r) {  // (A v)[r]
        const pidx *Arp = pat + sA.pArp, *Aci = pat + sA.pAci, *Aperm = pat + sA.pAperm;
        double s = 0.0;
        int k1 = Arp[r + 1];
        QP_U1 for (int k = Arp[r]; k < k1; k++) s += Av[Aperm[k]] * v[Aci[k]];
        return s;
    }
    static __device__ __forceinline__ double AT_col(const pidx* pat, const double* Av, const double* yc, int c) {  // (A' yc)[c]
        const pidx *Ap = pat + sA.pAp, *Ai = pat + sA.pAi;
        double s = 0.0;
        int e1 = Ap[c + 1];
        QP_U1 for (int e = Ap[c]; e < e1; e++) s += Av[e] * yc[Ai[e]];
        return s;
    }
    static __device__ QP_FN void mulH(const double* v, double* out) {  // out = (H + reg I) v (H symmetric: column gather)
        QP_CTX QP_PAT
        const double* Hv = V_(Hv);
        QP_U1 for (int c = lane; c < nV; c += TEAM) out[c] = H_row(pat, Hv, v, c);
        SYNC();
    }
    static __device__ QP_FN void mulH_noreg(const double* v, double* out) {  // out = H v (objective / KKT epilogue)
        QP_CTX QP_PAT
        const pidx *Hp = pat + sA.pHp, *Hi = pat + sA.pHi;
        const double* Hv = V_(Hv);
        const bool has_H = sA.has_H && !sA.is_lp;
        QP_U1 for (int c = lane; c < nV; c += TEAM) {
            double s = 0.0;
            if (has_H) {
                int e1 = Hp[c + 1];
                QP_U1 for (int e = Hp[c]; e < e1; e++) s += Hv[e] * v[Hi[e]];
            }
            out[c] = s;
        }
        SYNC();
    }
    static __device__ QP_FN void mulA(const double* v, double* out) {
        QP_CTX QP_PAT
        const double* Av = V_(Av);
        QP_U1 for (int r = lane; r < nC; r += TEAM) out[r] = A_row(pat, Av, v, r);
        SYNC();
    }
    static __device__ QP_FN void mulAT(const double* yc, double* out) {
        QP_CTX QP_PAT
        const double* Av = V_(Av);
        QP_U1 for (int c = lane; c < nV; c += TEAM) out[c] = AT_col(pat, Av, yc, c);
        SYNC();
    }
    // A[r][c] via the CSR view (duplicates summed)
    static __device__ __forceinline__ double A_entry(const pidx* pat, const double* Av, int r, int c) {
        const pidx *Arp = pat + sA.pArp, *Aci = pat + sA.pAci, *Aperm = pat + sA.pAperm;
        double s = 0.0;
        int k1 = Arp[r + 1];
        QP_U1 for (int k = Arp[r]; k < k1; k++)
            if (Aci[k] == c) s += Av[Aperm[k]];
        return s;
    }

    // ---------------------------------------------------------------- reductions
    // lexicographic (t, pos) minimum over the team, returned to every thread
    static __device__ __forceinline__ MinKey team_min(double t, int pos) {
        const unsigned tm = team_mask<TEAM>();
        QP_U1 for (int o = (TEAM < 32 ? TEAM : 32) / 2; o > 0; o >>= 1) {
            double t2_ = __shfl_xor_sync(tm, t, o);
            int p2 = __shfl_xor_sync(tm, pos, o);
            if (key_less(t2_, p2, t, pos)) { t = t2_; pos = p2; }
        }
        if (TEAM > 32) {
            __syncthreads();  // previous use of the scratch is over
            if ((threadIdx.x & 31) == 0) { sRedT[threadIdx.x >> 5] = t; sRedP[threadIdx.x >> 5] = pos; }
            __syncthreads();
            t = sRedT[0]; pos = sRedP[0];
            QP_U1 for (int k = 1; k < TEAM / 32; k++)
                if (key_less(sRedT[k], sRedP[k], t, pos)) { t = sRedT[k]; pos = sRedP[k]; }
        }
        MinKey r; r.t = t; r.pos = pos;
        return r;
    }

    // ---------------------------------------------------------------- Givens
    static __device__ __forceinline__ void givens(double a_, double b_, double& c, double& s, double& r) {
        if (a_ == 0.0) { c = 1.0; s = 0.0; r = b_; return; }
        double h = sqrt(a_ * a_ + b_ * b_);
        c = b_ / h; s = a_ / h; r = h;
    }

    // ---------------------------------------------------------------- projected Cholesky
    static __device__ QP_FN void proj_column(int b) {  // t2 = (H+regI) * (column b of Q scattered to full space)
        QP_CTX
        double *t1 = V_(t1), *t2 = V_(t2);
        const double* Q = V_(Q);
        const short* posFR = posFR_;
        QP_U1 for (int i = lane; i < nV; i += TEAM) { int p = posFR[i]; t1[i] = (p >= 0) ? Q[p * ld + b] : 0.0; }
        SYNC();
        mulH(t1, t2);
    }
    // returns 0 ok, 1+j on failure (uniform)
    static __device__ QP_FN int recompute_R() {
        QP_CTX
        const int nFR = hdr[0], nAC = hdr[1], nZ = nFR - nAC;
        if (nZ <= 0) return 0;
        double* RT = V_(RT);
        if (sA.is_lp) {
            double sr = sqrt(QP_EPS_REG);
            QP_U1 for (int k = lane; k < nZ * nZ; k += TEAM) { int a_ = k / nZ, b_ = k % nZ; R_(a_, b_) = (a_ == b_) ? sr : 0.0; }
            if constexpr (TEAM > 32) {  // block inverses used by the triangular solves
                double* W = V_(W);
                for (int k = lane; k < nZ * 64; k += TEAM) { const int a_ = k >> 6, c_ = k & 63; if (c_ < ld) W[(size_t)a_ * ld + c_] = (c_ == (a_ & 63)) ? 1.0 / sr : 0.0; }
            }
            SYNC();
            return 0;
        }
        if constexpr (TEAM > 32) return recompute_R_blocked();
        PROF_T0
        // M = Z'(HZ), several null-space columns at a time so that all 32 lanes have work (one lane per entry of W = HZ, then
        // one lane per entry of M) instead of one column per pass with nV- and (b+1)-wide loops.  W lives in the seven work
        // vectors t1,t2,t3,w,a,yv,zv (sA.nW doubles), which are contiguous and unused here.  Per entry the same terms in the same order as the
        // column-by-column form: W[p][b] = sum over the entries of H's column FR[p], M[a][b] = sum over p ascending.
        {
            QP_PAT
            const double *Q = V_(Q), *Hv = V_(Hv);
            double* Wc = V_(t1);
            const short *FR = FR_, *posFR = posFR_;
            const pidx *Hp = pat + sA.pHp, *Hi = pat + sA.pHi;
            const bool has_H = sA.has_H != 0;
            int CH = sA.nW / nFR;
            if (CH > nZ) CH = nZ;
            QP_U1 for (int b0 = 0; b0 < nZ; b0 += CH) {
                const int cw = (nZ - b0 < CH) ? nZ - b0 : CH;
                QP_U1 for (int e = lane; e < nFR * cw; e += TEAM) {
                    const int p = e / cw, bb = e - p * cw;
                    double s = 0.0;
                    if (has_H) {
                        const int c = FR[p], e1 = Hp[c + 1];
                        QP_U1 for (int h = Hp[c]; h < e1; h++) {
                            const int pr = posFR[Hi[h]];
                            s += Hv[h] * ((pr >= 0) ? Q[pr * ld + b0 + bb] : 0.0);
                        }
                    }
                    Wc[e] = s;
                }
                SYNC();
                QP_U1 for (int e = lane; e < (b0 + cw) * cw; e += TEAM) {
                    const int a_ = e / cw, bb = e - a_ * cw;
                    if (a_ <= b0 + bb) {
                        double s = 0.0;
                        QP_U1 for (int p = 0; p < nFR; p++) s += Q[p * ld + a_] * Wc[p * cw + bb];
                        R_(a_, b0 + bb) = s;
                    }
                }
                SYNC();
            }
        }
        PROF_ADD(PR_REFAC_M);
        // row-wise Cholesky: R'R = M, same per-element summation order as the column version
        QP_U1 for (int i = 0; i < nZ; i++) {
            QP_U1 for (int j = i + lane; j < nZ; j += TEAM) {
                double s = R_(i, j);
                DOT_UNROLL for (int k = 0; k < i; k++) s -= R_(k, i) * R_(k, j);
                R_(i, j) = s;
            }
            SYNC();
            double d = R_(i, i);
            SYNC();  // all lanes hold d before anyone rewrites R(i,i): the branch below is warp-uniform
            if (!(d > QP_ZERO)) return 1 + i;
            double dd = sqrt(d);
            QP_U1 for (int j = i + lane; j < nZ; j += TEAM) R_(i, j) = (j == i) ? dd : R_(i, j) / dd;
            QP_U1 for (int j = lane; j < i; j += TEAM) R_(i, j) = 0.0;
            SYNC();
        }
        PROF_ADD(PR_REFAC_CHOL);
        return 0;
    }

    // =====================================================================================================================
    // One-QP-per-CTA kernel (TEAM == 512), B200 form of the O(n^3) part and of the triangular solves.  Parity gate for
    // this kernel is north_star's (identical working sets, 1e-8 relative): sums run on the FP64 tensor cores, whose
    // accumulation order differs from the oracle's.
    //
    //   * contraction tiles C(64x64) (+|-)= X' Y on FP64 DMMA (mma.sync.m8n8k4.f64; 16 warps x (16x16) sub-tiles), operands
    //     staged by 1-D TMA bulk copies (one per 512-byte tile row, issued by warp 0) into a 3-stage shared-memory ring
    //     with mbarrier completion: no thread waits on a global load, every tile row is fetched from L2 once;
    //   * refactorisation: W = H Z (sparse x dense), M = Z'W (DMMA), left-looking block Cholesky with 64-row blocks:
    //     block-row update (DMMA), diagonal block factorised AND inverted in shared memory, panel = Dinv' S (DMMA);
    //   * the 64x64 inverses of the diagonal blocks stay in the (then dead) scratch matrix W and turn the triangular
    //     solves into mat-vecs: per 64 unknowns one strip product and one product with the block inverse;
    //   * thread-block cluster: the CTAs of a cluster share one QP.  Rank 0 runs the active-set method; ranks > 0 wait
    //     at a cluster barrier and take their share of the W rows and of the DMMA tiles of every refactorisation, so a
    //     batch smaller than the SM count still fills the GPU (batch 64 -> 2 CTAs per QP, 16 -> 8).
    // =====================================================================================================================
    static constexpr int LT_KC = 32, LT_STAGES = 3, LT_LD = 68, LT_NB = 64;
    static constexpr int LT_STAGE_DOUBLES = LT_KC * LT_LD;            // one operand of one stage
    static constexpr int LT_D_LD = 65;
    // dynamic shared memory map of the large kernel (doubles from qp_smem)
    static constexpr int LS_X = 0, LS_Y = LT_STAGES * LT_STAGE_DOUBLES, LS_D = 2 * LT_STAGES * LT_STAGE_DOUBLES,
                         LS_DI = LS_D + LT_NB * LT_D_LD, LS_RED = LS_DI + LT_NB * LT_D_LD, LS_TV = LS_RED + 8 * LT_NB,
                         LS_TOTAL = LS_TV + 2 * LT_NB;

    static __device__ __forceinline__ void large_sync() {  // leader + helpers: orders generic and TMA accesses to the factors
        asm volatile("fence.proxy.async;" ::: "memory");
        if (sClusterSize > 1) asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
        else __syncthreads();
    }
    static __device__ __forceinline__ void dmma(double (&c)[2], double a, double b) {
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
    }
    // C[a*ld + b] (+|-)= sum_{k<K} X[k*ld + a] * Y[k*ld + b] for a, b < 64 (X, Y, C point at the tile origins; X and Y rows must
    // be 16-byte aligned); stores only a < na, b < nb and, if TRI, ga + a <= gb + b.  Called by all threads of the CTA.
    template <int SIGN, bool TRI>
    static __device__ __forceinline__ void mma_tile(const double* X, int xw, const double* Y, int yw, int K, double* C, int na, int nb,
                                                    int ld, bool init_zero, int ga, int gb) {
        static_assert(TEAM == 512, "tile mapping assumes 16 warps");
        uint32_t ph = sPhase;  // mbarrier phase bits of the ring, carried from tile to tile (uniform over the CTA)
        double* Xs = qp_smem + LS_X;
        double* Ys = qp_smem + LS_Y;
        const int tid = threadIdx.x, warp = tid >> 5, l = tid & 31, g = l >> 2, t = l & 3;
        const int ra = (warp >> 2) * 16, cb = (warp & 3) * 16;
        double acc[2][2][2];
#pragma unroll
        for (int mi = 0; mi < 2; mi++)
#pragma unroll
            for (int ni = 0; ni < 2; ni++)
#pragma unroll
                for (int j = 0; j < 2; j++) {
                    const int a = ra + mi * 8 + g, b = cb + ni * 8 + t * 2 + j;
                    acc[mi][ni][j] = (!init_zero && a < na && b < nb && (!TRI || ga + a <= gb + b)) ? C[a * ld + b] : 0.0;
                }
        const int nch = (K + LT_KC - 1) / LT_KC;
        auto issue = [&](int chunk, int s) {  // warp 0: one bulk copy per operand row
            const int rows = (K - chunk * LT_KC < LT_KC) ? K - chunk * LT_KC : LT_KC;
            if (l == 0) mbar_expect_tx(&sFull[s], (uint32_t)rows * (uint32_t)(xw + yw) * 8u);
            __syncwarp();
            if (l < rows) {
                const size_t kr = (size_t)(chunk * LT_KC + l) * ld;
                bulk_g2s(Xs + s * LT_STAGE_DOUBLES + l * LT_LD, X + kr, (uint32_t)xw * 8u, &sFull[s]);
                bulk_g2s(Ys + s * LT_STAGE_DOUBLES + l * LT_LD, Y + kr, (uint32_t)yw * 8u, &sFull[s]);
            }
        };
        if (warp == 0)
            for (int c = 0; c < LT_STAGES && c < nch; c++) issue(c, c);
        for (int c = 0; c < nch; c++) {
            const int s = c % LT_STAGES;
            while (!mbar_try_wait(&sFull[s], (ph >> s) & 1u)) {}
            ph ^= 1u << s;
            const int rows = (K - c * LT_KC < LT_KC) ? K - c * LT_KC : LT_KC;
            const double* xs = Xs + s * LT_STAGE_DOUBLES + ra + g;
            const double* ys = Ys + s * LT_STAGE_DOUBLES + cb + g;
            const int k4n = (rows + 3) >> 2;
#pragma unroll 2
            for (int k4 = 0; k4 < k4n; k4++) {
                const int kr = k4 * 4 + t;
                double a0 = xs[kr * LT_LD], a1 = xs[kr * LT_LD + 8], b0 = ys[kr * LT_LD], b1 = ys[kr * LT_LD + 8];
                if (kr >= rows) { a0 = 0.0; a1 = 0.0; b0 = 0.0; b1 = 0.0; }
                if (SIGN < 0) { a0 = -a0; a1 = -a1; }
                dmma(acc[0][0], a0, b0); dmma(acc[0][1], a0, b1); dmma(acc[1][0], a1, b0); dmma(acc[1][1], a1, b1);
            }
            __syncthreads();  // stage s consumed by every warp
            if (warp == 0 && c + LT_STAGES < nch) issue(c + LT_STAGES, s);
        }
#pragma unroll
        for (int mi = 0; mi < 2; mi++)
#pragma unroll
            for (int ni = 0; ni < 2; ni++)
#pragma unroll
                for (int j = 0; j < 2; j++) {
                    const int a = ra + mi * 8 + g, b = cb + ni * 8 + t * 2 + j;
                    if (a < na && b < nb && (!TRI || ga + a <= gb + b)) C[a * ld + b] = acc[mi][ni][j];
                }
        if (tid == 0) sPhase = ph;
        __syncthreads();
    }
    // ---- coalesced O(n^2) primitives of the one-QP-per-CTA kernel.  The factors are row-major in global memory: a thread
    // that walks "its" row (the warp kernel's lane-per-row loops) makes every warp load touch 32 different lines, which at
    // nFR ~ 10^3 turns each sweep into an L2-latency chain.  Here the fast index always runs over the lanes.
    static __device__ __forceinline__ double team_sum(double v) {  // sum over the CTA, returned to every thread
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) sRedT[threadIdx.x >> 5] = v;
        __syncthreads();
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < TEAM / 32; k++) t += sRedT[k];
        return t;
    }
    // out[j] = sgn * sum_{p < nP} M[p * ld + j] * v[p] for j0 <= j < j1: blocks of 64 columns (even-aligned), a lane on two adjacent
    // columns (one 16-byte load per row), warp w on the rows w, w + 16, ...; eight loads in flight per lane
    static __device__ __forceinline__ void col_sums(const double* M, int ld, int nP, int j0, int j1, const double* v, double* out, double sgn,
                                                    int rank = 0, int cs = 1) {
        double* red16 = qp_smem;  // [16][64] (the tile ring is idle outside the refactorisation)
        const int tid = threadIdx.x, warp = tid >> 5, l = tid & 31;
        for (int jb = (j0 & ~1) + 64 * rank; jb < j1; jb += 64 * cs) {
            const int j = jb + 2 * l;
            double s0 = 0.0, s1 = 0.0;
            if (j < j1) {
                const double* base = M + j;
#pragma unroll 8
                for (int pp = warp; pp < nP; pp += TEAM / 32) {
                    const double2 m = *reinterpret_cast<const double2*>(base + (size_t)pp * ld);
                    const double vp = v[pp];
                    s0 += m.x * vp; s1 += m.y * vp;
                }
            }
            red16[warp * 64 + 2 * l] = s0; red16[warp * 64 + 2 * l + 1] = s1;
            __syncthreads();
            if (tid < 64 && jb + tid >= j0 && jb + tid < j1) {
                double t = 0.0;
#pragma unroll
                for (int q = 0; q < TEAM / 32; q++) t += red16[q * 64 + tid];
                out[jb + tid] = sgn * t;
            }
            __syncthreads();
        }
    }
    // s_p = sum_{j0 <= j < j1} M[p * ld + j] * v[j] for p < nP, a warp on four rows at a time, a lane on two adjacent columns
    // (16-byte loads); out[idx ? idx[p] : p] (+)= s_p
    static __device__ __forceinline__ void row_sums(const double* M, int ld, int nP, int j0, int j1, const double* v, double* out,
                                                    const short* idx, bool accumulate, int rank = 0, int cs = 1) {
        const int warp = threadIdx.x >> 5, l = threadIdx.x & 31, ja = j0 & ~1;
        for (int pr = (warp + (TEAM / 32) * rank) * 4; pr < nP; pr += (TEAM / 32) * cs * 4) {
            double s4[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll 2
            for (int j = ja + 2 * l; j < j1; j += 64) {
                const bool lo = j >= j0, hi = j + 1 < j1;
                const double v0 = lo ? v[j] : 0.0, v1 = hi ? v[j + 1] : 0.0;
#pragma unroll
                for (int q = 0; q < 4; q++)
                    if (pr + q < nP) {
                        const double2 m = *reinterpret_cast<const double2*>(M + (size_t)(pr + q) * ld + j);
                        s4[q] += (lo ? m.x * v0 : 0.0) + (hi ? m.y * v1 : 0.0);
                    }
            }
#pragma unroll
            for (int q = 0; q < 4; q++) {
                double sq = s4[q];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
                if (l == 0 && pr + q < nP) { const int k = idx ? idx[pr + q] : pr + q; out[k] = accumulate ? out[k] + sq : sq; }
            }
        }
        __syncthreads();
    }
    // the rotation chain (c_j, s_j), j < cnt - 1, acting on columns (j, j + 1), applied to rows p < nP of M: per row
    //   qa = q[0]; for j: qb = q[j+1]; q[j] = c qa - s qb; qa = s qa + c qb;  q[cnt-1] = qa
    // Warp w owns 32-row groups; a group moves through shared memory in 32-column tiles (coalesced loads and stores, the
    // chain runs lane-per-row out of the tile).
    // The chain runs over the logical columns j = 0 .. cnt-1, stored at column base + dir * j (dir = -1: the right-to-left
    // chains of the removals, whose rotation i acts on (c, c+1) with c decreasing: same recurrence with (c_j, -s_j)).
    // tri: M is upper triangular (row r zero left of column r), so the chain of a row group starts at its first fill-in.
    // Groups of 16 rows (8 while that leaves warps without work); the chain runs on the first lanes.  The 16 row loads of the
    // next tile are issued before the chain of the current one, so a warp always has a tile in flight (a solve is bound by
    // load latency: with loads only between the chains an SM moved ~11 GB/s here).
    static __device__ __forceinline__ void rot_rows(double* M, int ld, int nP, int cnt, const double* cs, const double* sn, int rank = 0,
                                                    int ncta = 1, int base = 0, int dir = 1, bool tri = false) {
        if (cnt <= 0) return;
        const int warp = threadIdx.x >> 5, l = threadIdx.x & 31, nwarps = (TEAM / 32) * ncta;
        constexpr int GM = 16;
        int G = GM;
        while (G > 8 && (nP + G - 1) / G < nwarps) G >>= 1;
        double* tile = qp_smem + (size_t)warp * (GM * 33 + 64);
        double* rotc = tile + GM * 33;  // (c, s) of the tile's 32 rotations: the chain must not wait for global loads
        for (int r0 = (warp + (TEAM / 32) * rank) * G; r0 < nP; r0 += nwarps * G) {
            const int nr = (nP - r0 < G) ? nP - r0 : G;
            const int jt0 = (tri && r0 > 0) ? ((r0 - 1) & ~31) : 0;
            double qa = (l < nr) ? M[(size_t)(r0 + l) * ld + base + dir * jt0] : 0.0;
            double v[GM], cj, sj;
            // originals of columns jt+1 .. jt+32 of the group's rows, and the rotations jt .. jt+31
            auto issue = [&](int jt) {
                const int j = jt + 1 + l;
#pragma unroll
                for (int u = 0; u < GM; u++) v[u] = (u < nr && j < cnt) ? M[(size_t)(r0 + u) * ld + base + dir * j] : 0.0;
                cj = (j < cnt) ? cs[j - 1] : 1.0; sj = (j < cnt) ? sn[j - 1] : 0.0;
            };
            issue(jt0);
            for (int jt = jt0; jt < cnt; jt += 32) {
#pragma unroll
                for (int u = 0; u < GM; u++) tile[u * 33 + l] = v[u];
                rotc[l] = cj; rotc[32 + l] = sj;
                __syncwarp();
                if (jt + 32 < cnt) issue(jt + 32);
                if (l < nr) {
                    const int cmax = (cnt - jt < 32) ? cnt - jt : 32;       // columns of this tile
                    const int crot = (cnt - 1 - jt < 32) ? cnt - 1 - jt : 32;  // rotations of this tile (the last column has none)
                    double* tl = tile + l * 33;
                    int c = 0;
                    for (; c + 8 <= crot; c += 8) {  // operands of eight rotations first, then the dependent chain (s qa + c qb)
                        double co[8], si[8], qb[8];
#pragma unroll
                        for (int u = 0; u < 8; u++) { co[u] = rotc[c + u]; si[u] = rotc[32 + c + u]; qb[u] = tl[c + u]; }
#pragma unroll
                        for (int u = 0; u < 8; u++) { tl[c + u] = co[u] * qa - si[u] * qb[u]; qa = si[u] * qa + co[u] * qb[u]; }
                    }
                    for (; c < crot; c++) { const double co = rotc[c], si = rotc[32 + c], qb = tl[c]; tl[c] = co * qa - si * qb; qa = si * qa + co * qb; }
                    if (c < cmax) tl[c] = qa;
                }
                __syncwarp();
                for (int rr = 0; rr < nr; rr++) { const int j = jt + l; if (j < cnt) M[(size_t)(r0 + rr) * ld + base + dir * j] = tile[rr * 33 + l]; }
                __syncwarp();
            }
        }
        __syncthreads();
    }
    // ---- blocked substitutions with the reverse-triangular factor T (one-QP-per-CTA kernel).  In the index pair (i, k) with
    // d_k = nFR - 1 - k, L(i, k) = T(i, d_k) is lower triangular.  Blocks of 32: the diagonal block goes to shared memory and is
    // solved by warp 0 with shuffles (one quot() + one shuffle per unknown); the coupling with the other blocks is a
    // warp-per-row product with coalesced loads.  The column-by-column form above needs two CTA barriers and a global-memory
    // round trip per unknown, which at nAC ~ 500 was half of the step-direction time.
    // T v = b: v indexed by Q column (v[d_k]); b by AC position, destroyed.
    static __device__ __forceinline__ void solve_T_blocked(double* b, double* v) {
        QP_CTX
        const int nFR = hdr[0], nAC = hdr[1];
        const double* RT = V_(RT);
        double* Dt = qp_smem + LS_D;  // [32][33]
        const int tid = threadIdx.x, warp = tid >> 5, l = tid & 31;
        for (int i0 = 0; i0 < nAC; i0 += 32) {
            const int nb = (nAC - i0 < 32) ? nAC - i0 : 32;
            // left-looking: b_I -= L(I, 0:i0) v_{0:i0}; row i of the strip is contiguous: columns d_{i0-1} .. d_0 = nFR-i0 .. nFR-1
            for (int r = warp; r < nb; r += TEAM / 32) {
                const int i = i0 + r;
                double s0 = 0.0;
                for (int cc = nFR - i0 + l; cc < nFR; cc += 32) s0 += T_(i, cc) * v[cc];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                if (l == 0) b[i] -= s0;
            }
            for (int e = tid; e < 32 * 32; e += TEAM) {  // Dt[r][k] = L(i0 + r, i0 + k), k <= r
                const int r = e >> 5, k = e & 31;
                if (r < nb && k <= r) Dt[r * 33 + k] = T_(i0 + r, nFR - 1 - i0 - k);
            }
            __syncthreads();
            if (warp == 0) {
                double bl = (l < nb) ? b[i0 + l] : 0.0;
                const double piv = (l < nb) ? Dt[l * 33 + l] : 1.0, ri = 1.0 / piv;
                double mine = 0.0;
                for (int k = 0; k < nb; k++) {
                    const double lk = (l > k && l < nb) ? Dt[l * 33 + k] : 0.0;
                    const double vk = __shfl_sync(0xffffffffu, quot(bl, piv, ri), k);
                    if (l == k) mine = vk;
                    bl -= lk * vk;
                }
                if (l < nb) v[nFR - 1 - i0 - l] = mine;
            }
            __syncthreads();
        }
    }
    // T' u = r: r indexed by Q column (destroyed), u by AC position.
    static __device__ __forceinline__ void solve_Tt_blocked(double* r, double* u) {
        QP_CTX
        const int nFR = hdr[0], nAC = hdr[1];
        const double* RT = V_(RT);
        double* Dt = qp_smem + LS_D;
        double* red = qp_smem + LS_RED;  // [16][32]
        const int tid = threadIdx.x, warp = tid >> 5, l = tid & 31;
        for (int i0 = ((nAC - 1) >> 5) << 5; i0 >= 0; i0 -= 32) {
            const int nb = (nAC - i0 < 32) ? nAC - i0 : 32, i1 = i0 + nb;
            // r'_k -= sum_{i >= i1} L(i, k) u_i for k in the block: lanes over k (columns d_k, contiguous), warps over i
            {
                double s0 = 0.0;
                if (l < nb) for (int i = i1 + warp; i < nAC; i += TEAM / 32) s0 += T_(i, nFR - 1 - i0 - l) * u[i];
                red[warp * 32 + l] = s0;
            }
            for (int e = tid; e < 32 * 32; e += TEAM) {
                const int rr = e >> 5, k = e & 31;
                if (rr < nb && k <= rr) Dt[rr * 33 + k] = T_(i0 + rr, nFR - 1 - i0 - k);
            }
            __syncthreads();
            if (warp == 0) {
                double t = 0.0;
#pragma unroll
                for (int q = 0; q < TEAM / 32; q++) t += red[q * 32 + l];
                double rl = (l < nb) ? r[nFR - 1 - i0 - l] - t : 0.0;
                const double piv = (l < nb) ? Dt[l * 33 + l] : 1.0, ri = 1.0 / piv;
                double mine = 0.0;
                for (int k = nb - 1; k >= 0; k--) {
                    const double lk = (l < k) ? Dt[k * 33 + l] : 0.0;
                    const double uk = __shfl_sync(0xffffffffu, quot(rl, piv, ri), k);
                    if (l == k) mine = uk;
                    rl -= lk * uk;
                }
                if (l < nb) u[i0 + l] = mine;
            }
            __syncthreads();
        }
    }
    // leader only: Cholesky factor of the nb x nb diagonal block at (i0, i0) and its inverse, both formed in shared memory; the
    // factor goes back to R, the inverse to W[i0 + r][c].  Returns 0 or 1 + failing pivot (uniform).
    // Elimination with the block in registers (thread (r0, j) owns rows r0, r0 + 8, ... of column j): per pivot the owners
    // publish the finished (unscaled) row, one barrier, and every thread updates its own entries with a_ki a_kj / a_kk; the
    // square roots are taken afterwards for all rows at once, so the pivot chain is one division + one barrier long.
    // X = D^{-1} for the upper triangular 64 x 64 block D in shared memory (leading dimension LT_D_LD; entries outside the
    // leading nb x nb part are taken as the identity), by recursive doubling: the eight 8 x 8 diagonal blocks by substitution
    // (one thread per column), then X12 = -X11 (D12 X22) for block pairs of size 8, 16, 32 -- every element of a product by its
    // own thread, two barriers per level instead of one warp-synchronous step per row of the block.  T: scratch, same shape.
    static __device__ __forceinline__ void tri_inv_block(const double* D, double* X, double* T, int nb) {
        const int tid = threadIdx.x;
        for (int k = tid; k < LT_NB * LT_NB; k += TEAM) { const int i = k >> 6, j = k & 63; X[i * LT_D_LD + j] = (i == j && i >= nb) ? 1.0 : 0.0; }
        __syncthreads();
        if (tid < nb) X[tid * LT_D_LD + tid] = 1.0 / D[tid * LT_D_LD + tid];
        __syncthreads();
        if (tid < nb) {
            const int c = tid, g0 = c & ~7;
            for (int r = c - 1; r >= g0; r--) {
                double sacc = 0.0;
#pragma unroll 4
                for (int l = r + 1; l <= c; l++) sacc += D[r * LT_D_LD + l] * X[l * LT_D_LD + c];
                X[r * LT_D_LD + c] = -sacc * X[r * LT_D_LD + r];
            }
        }
        __syncthreads();
#pragma unroll 1
        for (int sz = 8; sz < LT_NB; sz <<= 1) {
            const int lg = (sz == 8) ? 3 : ((sz == 16) ? 4 : 5);
            // T = D12 X22 (X22 upper triangular: k <= j)
            for (int e = tid; e < 32 * sz; e += TEAM) {
                const int j = e & (sz - 1), i = (e >> lg) & (sz - 1), pr = e >> (2 * lg), a0 = pr * 2 * sz, b0 = a0 + sz;
                const double* dr = D + (a0 + i) * LT_D_LD + b0;
                const double* xc = X + b0 * LT_D_LD + b0 + j;
                double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
                int k = 0;
#pragma unroll 2
                for (; k + 3 <= j; k += 4) {
                    s0 += dr[k] * xc[k * LT_D_LD]; s1 += dr[k + 1] * xc[(k + 1) * LT_D_LD];
                    s2 += dr[k + 2] * xc[(k + 2) * LT_D_LD]; s3 += dr[k + 3] * xc[(k + 3) * LT_D_LD];
                }
                for (; k <= j; k++) s0 += dr[k] * xc[k * LT_D_LD];
                T[(a0 + i) * LT_D_LD + b0 + j] = (a0 + i < nb && b0 + j < nb) ? (s0 + s1) + (s2 + s3) : 0.0;
            }
            __syncthreads();
            // X12 = -X11 T (X11 upper triangular: k >= i)
            for (int e = tid; e < 32 * sz; e += TEAM) {
                const int j = e & (sz - 1), i = (e >> lg) & (sz - 1), pr = e >> (2 * lg), a0 = pr * 2 * sz, b0 = a0 + sz;
                const double* xr = X + (a0 + i) * LT_D_LD + a0;
                const double* tc = T + a0 * LT_D_LD + b0 + j;
                double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
                int k = i;
#pragma unroll 2
                for (; k + 3 < sz; k += 4) {
                    s0 += xr[k] * tc[k * LT_D_LD]; s1 += xr[k + 1] * tc[(k + 1) * LT_D_LD];
                    s2 += xr[k + 2] * tc[(k + 2) * LT_D_LD]; s3 += xr[k + 3] * tc[(k + 3) * LT_D_LD];
                }
                for (; k < sz; k++) s0 += xr[k] * tc[k * LT_D_LD];
                X[(a0 + i) * LT_D_LD + b0 + j] = -((s0 + s1) + (s2 + s3));
            }
            __syncthreads();
        }
    }
    static __device__ __forceinline__ int diag_block(int i0, int nb) {
        QP_CTX
        double *RT = V_(RT), *W = V_(W);
        double* D = qp_smem + LS_D;
        double* DI = qp_smem + LS_DI;
        double* sc = qp_smem + LS_RED;  // [0..1]: 1 / pivot (double-buffered), [2]: failure flag, [64..127]: 1 / R_kk
        const int tid = threadIdx.x, j = tid & 63, r0 = tid >> 6;
        double a[8];
#pragma unroll
        for (int q = 0; q < 8; q++) {
            const int i = r0 + 8 * q;
            a[q] = (i < nb && j < nb && i <= j) ? R_(i0 + i, i0 + j) : 0.0;
            DI[i * LT_D_LD + j] = 0.0;
        }
        if (tid == 0) sc[2] = 0.0;
        __syncthreads();
        for (int k = 0; k < nb; k++) {
            if ((k & 7) == r0 && j >= k && j < nb) {
                const double v = a[k >> 3];
                D[k * LT_D_LD + j] = v;
                if (j == k) { if (v > QP_ZERO) sc[k & 1] = 1.0 / v; else sc[2] = (double)(1 + i0 + k); }
            }
            __syncthreads();
            if (sc[2] != 0.0) return (int)sc[2];
            const double inv = sc[k & 1], dkj = D[k * LT_D_LD + j] * inv;
#pragma unroll
            for (int q = 0; q < 8; q++) {
                const int i = r0 + 8 * q;
                if (i > k && i <= j && j < nb) a[q] -= D[k * LT_D_LD + i] * dkj;
            }
        }
        __syncthreads();
        if (tid < nb) { const double d = sqrt(D[tid * LT_D_LD + tid]); sc[64 + tid] = 1.0 / d; sc[128 + tid] = d; }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 8; q++) {
            const int i = r0 + 8 * q;
            if (i < nb && j < nb && i <= j) {
                const double v = (i == j) ? sc[128 + i] : D[i * LT_D_LD + j] * sc[64 + i];
                D[i * LT_D_LD + j] = v;
                R_(i0 + i, i0 + j) = v;
            }
        }
        __syncthreads();
        // inverse of the (upper triangular) factor
        if (nb < LT_NB) {  // the last block: identity outside the leading nb x nb part
#pragma unroll
            for (int q = 0; q < 8; q++) { const int i = r0 + 8 * q; if (i < j && j >= nb) D[i * LT_D_LD + j] = 0.0; }
            if (tid >= nb && tid < LT_NB) D[tid * LT_D_LD + tid] = 1.0;
            __syncthreads();
        }
        tri_inv_block(D, DI, qp_smem, nb);
#pragma unroll
        for (int q = 0; q < 8; q++) {
            const int i = r0 + 8 * q;
            if (i < nb && j < nb) W[(size_t)(i0 + i) * ld + j] = DI[i * LT_D_LD + j];
        }
        __syncthreads();
        return 0;
    }
    // Executed by every CTA of the cluster (rank, cs): the refactorisation R'R = Z'(H + reg I)Z with all its cluster barriers.
    static __device__ __noinline__ int refac_body(int rank, int cs) {
        QP_CTX QP_PAT
        volatile int* vh = hdr;
        const int nFR = vh[0], nAC = vh[1], nZ = nFR - nAC;
        double *RT = V_(RT), *W = V_(W);
        const double *Q = V_(Q), *Hv = V_(Hv);
        const short *FR = FR_, *posFR = posFR_;
        const pidx *Hp = pat + sA.pHp, *Hi = pat + sA.pHi;
        const bool has_H = sA.has_H && !sA.is_lp;
        PROF_T0
        // A: W[p][b] = (H z_b)[FR[p]], entries split over the cluster; a thread owns four columns b, b + 32, b + 64, b + 96 of
        // one row p so that every index / value load of H's column is shared by four outputs (lanes still walk b: coalesced)
        {
            const int nb4 = (nZ + 127) / 128;  // groups of 128 columns
            const int l32 = lane & 31;
            for (int e = rank * (TEAM / 32) + (lane >> 5); e < nFR * nb4; e += cs * (TEAM / 32)) {
                const int p = e / nb4, b0 = (e - p * nb4) * 128 + l32;
                double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
                if (has_H) {
                    const int c = FR[p], e1 = Hp[c + 1];
                    for (int h = Hp[c]; h < e1; h++) {
                        const int pr = posFR[Hi[h]];
                        if (pr >= 0) {
                            const double hv = Hv[h];
                            const double* q = Q + (size_t)pr * ld + b0;
                            if (b0 < nZ) s0 += hv * q[0];
                            if (b0 + 32 < nZ) s1 += hv * q[32];
                            if (b0 + 64 < nZ) s2 += hv * q[64];
                            if (b0 + 96 < nZ) s3 += hv * q[96];
                        }
                    }
                }
                double* w = W + (size_t)p * ld + b0;
                if (b0 < nZ) w[0] = s0;
                if (b0 + 32 < nZ) w[32] = s1;
                if (b0 + 64 < nZ) w[64] = s2;
                if (b0 + 96 < nZ) w[96] = s3;
            }
        }
        large_sync();
        PROF_ADD(PR_REFAC_W);
        // B: M = Z'W, upper-triangle tiles dealt round-robin to the CTAs of the cluster
        {
            int t = 0;
            for (int b0 = 0; b0 < nZ; b0 += LT_NB)
                for (int a0 = 0; a0 <= b0; a0 += LT_NB, t++)
                    if (t % cs == rank) {
                        const int xw = (ld - a0 < LT_NB) ? ld - a0 : LT_NB, yw = (ld - b0 < LT_NB) ? ld - b0 : LT_NB;
                        mma_tile<1, true>(Q + a0, xw, W + b0, yw, nFR, RT + (size_t)a0 * ld + b0, (nZ - a0 < LT_NB) ? nZ - a0 : LT_NB,
                                          (nZ - b0 < LT_NB) ? nZ - b0 : LT_NB, ld, true, a0, b0);
                    }
        }
        large_sync();
        PROF_ADD(PR_REFAC_M);
        // C: left-looking block Cholesky
        int fail = 0;
        for (int i0 = 0; i0 < nZ; i0 += LT_NB) {
            const int i1 = (i0 + LT_NB < nZ) ? i0 + LT_NB : nZ, nbk = i1 - i0;
            if (i0 > 0) {
                int t = 0;
                for (int b0 = 0; b0 < nZ - i0; b0 += LT_NB, t++)
                    if (t % cs == rank) {
                        const int xw = (ld - i0 < LT_NB) ? ld - i0 : LT_NB, yw = (ld - i0 - b0 < LT_NB) ? ld - i0 - b0 : LT_NB;
                        mma_tile<-1, true>(RT + i0, xw, RT + i0 + b0, yw, i0, RT + (size_t)i0 * ld + i0 + b0, nbk,
                                           (nZ - i0 - b0 < LT_NB) ? nZ - i0 - b0 : LT_NB, ld, false, 0, b0);
                    }
                large_sync();
            }
            if (rank == 0) {
                const int f = diag_block(i0, nbk);
                if (lane == 0) hdr[5] = f;
            }
            large_sync();
            fail = vh[5];
            if (fail) break;
            {
                int t = 0;
                for (int b0 = i1; b0 < nZ; b0 += LT_NB, t++)
                    if (t % cs == rank) {
                        const int yw = (ld - b0 < LT_NB) ? ld - b0 : LT_NB;
                        mma_tile<1, false>(W + (size_t)i0 * ld, (ld < LT_NB) ? ld : LT_NB, RT + (size_t)i0 * ld + b0, yw, nbk, RT + (size_t)i0 * ld + b0, nbk,
                                           (nZ - b0 < LT_NB) ? nZ - b0 : LT_NB, ld, true, 0, 0);
                    }
            }
            if (i1 < nZ) large_sync();
        }
        PROF_ADD(PR_REFAC_CHOL);
        return fail;
    }
    // ---- operations the leader shares with its helper CTAs: arguments go through the slice header (ints 4..15), offsets are
    // in doubles from the slice base.  Worth two cluster barriers only when the operand is large.
    enum { OP_REFAC = 1, OP_EXIT = 2, OP_COLSUMS = 3, OP_ROWSUMS = 4, OP_ROTROWS = 5, OP_DINV = 6 };
    static constexpr int DIST_MIN_ELEMS = 1 << 16;  // below ~0.5 MB of factor data the leader works alone (measured: 1 << 16 beats 1 << 17 by 3-6 %, 1 << 19 loses 10-20 %)
    static __device__ __forceinline__ void run_op(int cmd, int rank, int cs) {
        QP_CTX
        volatile int* vh = hdr;
        const int oM = vh[8], nP = vh[9], i0 = vh[10], i1 = vh[11], oA = vh[12], oB = vh[13], flag = vh[14];
        if (cmd == OP_COLSUMS) col_sums(slice + oM, ld, nP, i0, i1, slice + oA, slice + oB, flag ? -1.0 : 1.0, rank, cs);
        else if (cmd == OP_ROWSUMS) row_sums(slice + oM, ld, nP, i0, i1, slice + oA, slice + oB, (flag & 1) ? FR_ : nullptr, (flag & 2) != 0, rank, cs);
        else if (cmd == OP_ROTROWS) rot_rows(slice + oM, ld, nP, i0, slice + oA, slice + oB, rank, cs, i1, (flag & 1) ? -1 : 1, (flag & 2) != 0);
        else if (cmd == OP_DINV) dinv_blocks(nP, rank, cs);
    }
    static __device__ __forceinline__ void dist_op(int cmd, int oM, int nP, int i0, int i1, int oA, int oB, int flag) {
        QP_CTX
        if (lane == 0) { hdr[4] = cmd; hdr[8] = oM; hdr[9] = nP; hdr[10] = i0; hdr[11] = i1; hdr[12] = oA; hdr[13] = oB; hdr[14] = flag; }
        __syncthreads();
        large_sync();
        run_op(cmd, 0, sClusterSize);
        large_sync();
    }
    // the three primitives with automatic choice between the leader alone and the whole cluster
    static __device__ __forceinline__ void col_sums_auto(int oM, int nP, int j0, int j1, int oV, int oOut, bool negate) {
        QP_CTX
        if (sClusterSize > 1 && (long long)nP * (j1 - j0) >= DIST_MIN_ELEMS) dist_op(OP_COLSUMS, oM, nP, j0, j1, oV, oOut, negate ? 1 : 0);
        else col_sums(slice + oM, ld, nP, j0, j1, slice + oV, slice + oOut, negate ? -1.0 : 1.0);
    }
    static __device__ __forceinline__ void row_sums_auto(int oM, int nP, int j0, int j1, int oV, int oOut, bool via_FR, bool accumulate) {
        QP_CTX
        if (sClusterSize > 1 && (long long)nP * (j1 - j0) >= DIST_MIN_ELEMS) dist_op(OP_ROWSUMS, oM, nP, j0, j1, oV, oOut, (via_FR ? 1 : 0) | (accumulate ? 2 : 0));
        else row_sums(slice + oM, ld, nP, j0, j1, slice + oV, slice + oOut, via_FR ? FR_ : nullptr, accumulate);
    }
    static __device__ __forceinline__ void rot_rows_auto(int oM, int nP, int cnt, int oC, int oS_, int base = 0, int dir = 1, bool tri = false) {
        QP_CTX
        if (sClusterSize > 1 && (long long)nP * cnt >= DIST_MIN_ELEMS) dist_op(OP_ROTROWS, oM, nP, cnt, base, oC, oS_, (dir < 0 ? 1 : 0) | (tri ? 2 : 0));
        else rot_rows(slice + oM, ld, nP, cnt, slice + oC, slice + oS_, 0, 1, base, dir, tri);
    }
    // ---- Cholesky factor of the projected Hessian carried through an addition (one-QP-per-cluster kernel only).  The warp
    // kernel and the oracle recompute R after every addition, as qpOASES does under setToReliable
    // (enableCholeskyRefactorisation = 1); that is O(nZ^3) per working-set change.  Here the addition's rotation chain G (the
    // one that was just applied to the null-space columns of Q) is applied to the columns of R, the last column is dropped
    // (Z loses it) and the upper Hessenberg rest is brought back to triangular form by row rotations: R_new'R_new =
    // (Z G)'H(Z G) restricted to the kept columns, the same matrix a recomputation factorises, in O(nZ^2) (qpOASES's own
    // update under its default options).  A full recomputation still runs every REFAC_EVERY additions, after an exchange
    // step (R is one column short there) and after a flipped bound.
    static constexpr int REFAC_EVERY = 64;
    // inverses of the 64 x 64 diagonal blocks of R (n x n) into W, block b by CTA b % cs
    static __device__ __forceinline__ void dinv_blocks(int n, int rank, int cs) {
        QP_CTX
        const double* RT = V_(RT);
        double* W = V_(W);
        double* D = qp_smem + LS_D;
        double* DI = qp_smem + LS_DI;
        const int tid = threadIdx.x, j = tid & 63, r0 = tid >> 6;
        for (int i0 = rank * LT_NB; i0 < n; i0 += cs * LT_NB) {
            const int nb = (n - i0 < LT_NB) ? n - i0 : LT_NB;
#pragma unroll
            for (int q = 0; q < 8; q++) {
                const int i = r0 + 8 * q;
                D[i * LT_D_LD + j] = (i < nb && j < nb && i <= j) ? R_(i0 + i, i0 + j) : ((i == j) ? 1.0 : 0.0);
            }
            __syncthreads();
            tri_inv_block(D, DI, qp_smem, nb);
#pragma unroll
            for (int q = 0; q < 8; q++) {
                const int i = r0 + 8 * q;
                if (i < nb && j < nb) W[(size_t)(i0 + i) * ld + j] = DI[i * LT_D_LD + j];
            }
            __syncthreads();
        }
    }
    // rows 0..nZ-1, columns 0..nZ-2 of R hold an upper Hessenberg matrix: row rotation k (rows k, k+1) removes (k+1, k).
    // A thread owns the columns tid, tid + TEAM, ... and carries "its" entries of the running row k+1 in registers; the rows
    // k+1 .. k+4 are in flight in four register sets (the loop is unrolled by four so that the sets rotate without moves: an
    // L2 round trip per rotation otherwise); one barrier per rotation (the owner of column k publishes (c, s) through shared
    // memory).
    template <int NQ, int DEPTH>
    static __device__ __noinline__ void retriangularise(int nZ) {
        QP_CTX
        double* RT = V_(RT);
        double* sc = qp_smem + LS_RED;
        const int tid = threadIdx.x, m = nZ - 1;
        const int nact = (m < TEAM) ? ((m + 31) & ~31) : TEAM;
        if (tid >= nact) { __syncthreads(); return; }
        double cur[NQ], buf[DEPTH][NQ];  // buf[r % DEPTH]: row r
#pragma unroll
        for (int q = 0; q < NQ; q++) {
            const int j = tid + TEAM * q;
            cur[q] = (j < m) ? R_(0, j) : 0.0;
#pragma unroll
            for (int r = 1; r <= DEPTH; r++) buf[r % DEPTH][q] = (j < m && j + 1 >= r && r < nZ) ? R_(r, j) : 0.0;
        }
        for (int k0 = 0; k0 < m; k0 += DEPTH) {
#pragma unroll
            for (int u = 0; u < DEPTH; u++) {
                const int k = k0 + u;
                if (k >= m) break;
                double* nxt = buf[(u + 1) % DEPTH];  // row k+1 (k0 is a multiple of DEPTH)
                if (tid == (k & (TEAM - 1))) {
                    double a = 0.0, b = 0.0;
#pragma unroll
                    for (int q = 0; q < NQ; q++) if (q == k / TEAM) { a = cur[q]; b = nxt[q]; }
                    const double h2 = a * a + b * b;
                    double* o = sc + 2 * (k & 1);
                    if (h2 > 0.0) { const double ih = rsqrt(h2); o[0] = a * ih; o[1] = b * ih; } else { o[0] = 1.0; o[1] = 0.0; }
                }
                asm volatile("bar.sync 1, %0;" ::"r"(nact) : "memory");  // the warps that own a column
                const double c = sc[2 * (k & 1)], sn = sc[2 * (k & 1) + 1];
#pragma unroll
                for (int q = 0; q < NQ; q++) {
                    const int j = tid + TEAM * q;
                    if (j >= k && j < m) {
                        const double a = cur[q], b = nxt[q];
                        R_(k, j) = fma(c, a, sn * b);
                        if (j == k) { R_(k + 1, k) = 0.0; cur[q] = 0.0; }
                        else cur[q] = fma(c, b, -sn * a);
                    }
                    // row k + 1 + DEPTH takes the place of row k + 1
                    nxt[q] = (j >= k + DEPTH && j < m && k + 1 + DEPTH < nZ) ? R_(k + 1 + DEPTH, j) : 0.0;
                }
                // row k + 32 towards L2, one 128-byte line per thread
                if (k + 32 < nZ && tid * 16 < m && tid * 16 + 16 > k + 30) asm volatile("prefetch.global.L2 [%0];" ::"l"(&R_(k + 32, tid * 16)));
            }
        }
        __syncthreads();
    }
    // The same elimination with four rotations per barrier (m <= 4 * TEAM): a thread owns the four adjacent columns
    // 4 tid .. 4 tid + 3, so the owner of columns k0 .. k0+3 forms the rotations k0 .. k0+3 one after the other out of its own
    // registers (applying each to its four columns before the next) and publishes all four at once; the other threads then
    // apply the four rotations to their columns.  Rows k0+5 .. k0+8 are loaded while the group k0 is processed.
    static __device__ __noinline__ void retriangularise4(int nZ) {
        QP_CTX
        double* RT = V_(RT);
        double* sc = qp_smem + LS_RED;  // (c, s) of a group: 8 doubles, double-buffered
        const int tid = threadIdx.x, m = nZ - 1, j0 = 4 * tid;
        const int nact = (((m + 3) >> 2) + 31) & ~31;  // threads that own a column < m, whole warps
        if (tid >= nact) { __syncthreads(); return; }
        const bool full = j0 + 3 < m;
        auto load4 = [&](int r, double (&v)[4]) {
            if (r > m || j0 >= m || j0 + 4 < r) { v[0] = v[1] = v[2] = v[3] = 0.0; return; }  // row r is zero left of column r-1
            const double* p = &R_(r, j0);
            if (full) { const double2 a = *reinterpret_cast<const double2*>(p), b = *reinterpret_cast<const double2*>(p + 2); v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; }
            else {
#pragma unroll
                for (int q = 0; q < 4; q++) v[q] = (j0 + q < m) ? p[q] : 0.0;
            }
        };
        auto store4 = [&](int r, const double (&v)[4]) {
            if (j0 >= m || j0 + 3 < r) return;  // nothing on or right of the diagonal
            double* p = &R_(r, j0);
            if (full) { *reinterpret_cast<double2*>(p) = make_double2(v[0], v[1]); *reinterpret_cast<double2*>(p + 2) = make_double2(v[2], v[3]); }
            else {
#pragma unroll
                for (int q = 0; q < 4; q++) if (j0 + q < m) p[q] = v[q];
            }
        };
        double cur[4], rows[2][4][4];  // rows[g & 1][u]: row k0 + 1 + u of group g = k0 / 4
        load4(0, cur);
#pragma unroll
        for (int u = 0; u < 4; u++) load4(1 + u, rows[0][u]);
        for (int kk = 0; kk < m; kk += 8) {
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int k0 = kk + 4 * h;
                if (k0 >= m) break;
                double (&rw)[4][4] = rows[h];
#pragma unroll
                for (int u = 0; u < 4; u++) load4(k0 + 5 + u, rows[h ^ 1][u]);
                // rows k0 + 33 .. k0 + 36 towards L2, one 128-byte line per thread
#pragma unroll
                for (int u = 0; u < 4; u++)
                    if (k0 + 33 + u <= m && tid * 16 < m && tid * 16 + 16 > k0 + 31) asm volatile("prefetch.global.L2 [%0];" ::"l"(&R_(k0 + 33 + u, tid * 16)));
                double* o = sc + 8 * ((k0 >> 2) & 1);
                const bool owner = (tid == (k0 >> 2));
                if (owner) {
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        if (k0 + u < m) {
                            const double a = cur[u], b = rw[u][u], h2 = a * a + b * b;
                            double c = 1.0, sn = 0.0;
                            if (h2 > 0.0) { const double ih = rsqrt(h2); c = a * ih; sn = b * ih; }
                            o[2 * u] = c; o[2 * u + 1] = sn;
                            double top[4];
#pragma unroll
                            for (int v = 0; v < 4; v++) { top[v] = fma(c, cur[v], sn * rw[u][v]); cur[v] = fma(c, rw[u][v], -sn * cur[v]); }
                            cur[u] = 0.0;
                            store4(k0 + u, top);
                        }
                    }
                    if (k0 + 4 <= m) R_(k0 + 4, k0 + 3) = 0.0;  // the last eliminated entry lies in the next group's first row
                }
                asm volatile("bar.sync 1, %0;" ::"r"(nact) : "memory");
                if (!owner && j0 > k0) {
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        if (k0 + u < m) {
                            const double c = o[2 * u], sn = o[2 * u + 1];
                            double top[4];
#pragma unroll
                            for (int v = 0; v < 4; v++) { top[v] = fma(c, cur[v], sn * rw[u][v]); cur[v] = fma(c, rw[u][v], -sn * cur[v]); }
                            store4(k0 + u, top);
                        }
                    }
                }
            }
        }
        __syncthreads();
    }
    // R (nZ x nZ) -> factor of the working set that has just lost its last null-space column; (c_j, s_j) of the addition's chain
    // are still in t2 / t3
    static __device__ __noinline__ void update_R_after_add(int nZ) {
        QP_CTX
        const int m = nZ - 1;
        if (m <= 0) return;
        PROF_T0
        rot_rows_auto(sA.oRT, nZ, nZ, sA.ot2, sA.ot3, 0, 1, true);
        PROF_ADD(PR_REFAC_W);  // (profile build: the three slots of the recomputation show the update's steps)
        // (a panel variant -- one warp eliminating 32 columns out of registers, then all threads applying the 32 rotations to
        // their columns -- measured no faster: the chain of dependent FP64 operations per rotation, ~0.3 us, is what bounds all
        // three forms)
        if (m <= TEAM) retriangularise<1, 4>(nZ);
        else if (m <= 4 * TEAM) retriangularise4(nZ);
        else retriangularise<8, 4>(nZ);
        PROF_ADD(PR_REFAC_M);
        if (sClusterSize > 1 && m > LT_NB) dist_op(OP_DINV, 0, m, 0, 0, 0, 0, 0);
        else dinv_blocks(m, 0, 1);
        PROF_ADD(PR_REFAC_CHOL);
    }
    static constexpr int UPDATE_MAX_NZ = 8 * TEAM;
    static __device__ QP_FN int recompute_R_blocked() {
        QP_CTX
        if (lane == 0) hdr[4] = 1;  // command: refactorise
        __syncthreads();
        large_sync();               // releases the helper CTAs
        return refac_body(0, sClusterSize);
    }
    // ranks > 0 of the cluster
    static __device__ void helper_loop(int rank, int cs) {
        QP_CTX
        volatile int* vh = hdr;
        for (;;) {
            large_sync();
            const int cmd = vh[4];
            if (cmd == OP_EXIT) return;
            if (cmd == OP_REFAC) refac_body(rank, cs);
            else { run_op(cmd, rank, cs); large_sync(); }
        }
    }
    // R' u = z (n unknowns, in place) with the block inverses; col >= 0: also R(k, col) = u_k
    static __device__ QP_FN void fwd_solve_R_blocked(double* z, int n, int col) {
        QP_CTX
        double* RT = V_(RT);
        const double* W = V_(W);
        double* red = qp_smem + LS_RED;
        double* red16 = qp_smem;  // [16][64]: the tile ring is idle during the substitutions
        double* tv = qp_smem + LS_TV;
        const int tid = threadIdx.x, c = tid & 63, sl = tid >> 6, warp = tid >> 5, l = tid & 31;
        for (int i0 = 0; i0 < n; i0 += LT_NB) {
            const int nb = (n - i0 < LT_NB) ? n - i0 : LT_NB;
            // the block inverse goes to registers first: its loads are in flight during the strip product
            double dreg[8];
#pragma unroll
            for (int q = 0; q < 8; q++) { const int k = sl + 8 * q; dreg[q] = (c < nb && k <= c) ? W[(size_t)(i0 + k) * ld + c] : 0.0; }
            // strip product: a lane owns the columns i0 + 2l, i0 + 2l + 1 (one 16-byte load per row), warp w the rows w, w + 16, ...
            {
                double s0 = 0.0, s1 = 0.0;
                if (2 * l < nb) {
                    const double* base = &R_(0, i0 + 2 * l);
#pragma unroll 8
                    for (int k = warp; k < i0; k += TEAM / 32) {
                        const double2 v = *reinterpret_cast<const double2*>(base + (size_t)k * ld);
                        const double zk = z[k];
                        s0 += v.x * zk; s1 += v.y * zk;
                    }
                }
                if (l < 32) { red16[warp * LT_NB + 2 * l] = s0; red16[warp * LT_NB + 2 * l + 1] = s1; }
            }
            __syncthreads();
            if (tid < LT_NB) {
                double tsum = 0.0;
#pragma unroll
                for (int q = 0; q < TEAM / 32; q++) tsum += red16[q * LT_NB + tid];
                tv[tid] = (tid < nb) ? z[i0 + tid] - tsum : 0.0;
            }
            __syncthreads();
            // u_c = sum_{k <= c} Dinv[k][c] t_k
            {
                double s = 0.0;
#pragma unroll
                for (int q = 0; q < 8; q++) s += dreg[q] * tv[sl + 8 * q];
                red[sl * LT_NB + c] = s;
            }
            __syncthreads();
            if (tid < nb) {
                double u = 0.0;
#pragma unroll
                for (int q = 0; q < 8; q++) u += red[q * LT_NB + tid];
                z[i0 + tid] = u;
                if (col >= 0) R_(i0 + tid, col) = u;
            }
            __syncthreads();
        }
    }
    // R v = z (n unknowns, in place): one warp per row, lanes over the columns
    static __device__ QP_FN void bwd_solve_R_blocked(double* z, int n) {
        QP_CTX
        const double* RT = V_(RT);
        const double* W = V_(W);
        double* tv = qp_smem + LS_TV;
        const int tid = threadIdx.x, warp = tid >> 5, l = tid & 31;
        for (int i0 = ((n - 1) >> 6) << 6; i0 >= 0; i0 -= LT_NB) {
            const int nb = (n - i0 < LT_NB) ? n - i0 : LT_NB, i1 = i0 + nb;
            // the warp's rows of the block inverse first (row r: columns r + l, r + l + 32), in flight during the strip product
            double dreg[4][2];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int r = warp + (TEAM / 32) * q;
#pragma unroll
                for (int h = 0; h < 2; h++) { const int cc = r + l + 32 * h; dreg[q][h] = (r < nb && cc < nb) ? W[(size_t)(i0 + r) * ld + cc] : 0.0; }
            }
            {   // the warp's four rows (warp, warp + 16, ...) together, a lane on the columns k, k + 1 (16-byte loads; i1 is even)
                double s4[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll 2
                for (int k = i1 + 2 * l; k < n; k += 64) {
                    const double zk = z[k], zk1 = (k + 1 < n) ? z[k + 1] : 0.0;
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const int r = warp + (TEAM / 32) * q;
                        if (r < nb) { const double2 v = *reinterpret_cast<const double2*>(&R_(i0 + r, k)); s4[q] += v.x * zk + ((k + 1 < n) ? v.y * zk1 : 0.0); }
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    double sq = s4[q];
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
                    const int r = warp + (TEAM / 32) * q;
                    if (l == 0 && r < nb) tv[r] = z[i0 + r] - sq;
                }
            }
            __syncthreads();
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int r = warp + (TEAM / 32) * q;
                double s = 0.0;
#pragma unroll
                for (int h = 0; h < 2; h++) { const int cc = r + l + 32 * h; if (r < nb && cc < nb) s += dreg[q][h] * tv[cc]; }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                if (l == 0 && r < nb) z[i0 + r] = s;
            }
            __syncthreads();
        }
    }
    // after extend_R bordered R with column/row b (diagonal rho): extend the inverse of the last diagonal block
    static __device__ QP_FN void extend_Dinv(int b, double rho) {
        QP_CTX
        const double* RT = V_(RT);
        double* W = V_(W);
        const int i0 = (b >> 6) << 6, c = b - i0, tid = threadIdx.x;
        if (tid < c) {  // Dinv[r][c] = -(sum_{l = r..c-1} Dinv[r][l] R(i0 + l, b)) / rho
            double s = 0.0;
            for (int q = tid; q < c; q++) s += W[(size_t)(i0 + tid) * ld + q] * R_(i0 + q, b);
            W[(size_t)(i0 + tid) * ld + c] = -s / rho;
        } else if (tid == c) W[(size_t)(i0 + c) * ld + c] = 1.0 / rho;
        __syncthreads();
    }
    // border R with the new last null-space column; returns 1 if curvature acceptable
    static __device__ QP_FN int extend_R(int check_curvature) {
        QP_CTX
        const int nFR = hdr[0], nAC = hdr[1], nZ = nFR - nAC, b = nZ - 1;
        double *RT = V_(RT), *w = V_(w);
        if (sA.is_lp) {
            QP_U1 for (int a_ = lane; a_ < b; a_ += TEAM) { R_(a_, b) = 0.0; R_(b, a_) = 0.0; }
            if (lane == 0) R_(b, b) = sqrt(QP_EPS_REG);
            SYNC();
            if constexpr (TEAM > 32) extend_Dinv(b, sqrt(QP_EPS_REG));
            return 1;
        }
        const double *Q = V_(Q), *t2 = V_(t2);
        const short* FR = FR_;
        proj_column(b);
        if constexpr (TEAM > 32) {
            double* tmp = V_(a);  // dead between two homotopy steps
            for (int p = lane; p < nFR; p += TEAM) tmp[p] = t2[FR[p]];
            SYNC();
            col_sums_auto(sA.oQ, nFR, 0, b + 1, sA.oa, sA.ow, false);
        } else
        {
        QP_U1 for (int a_ = lane; a_ <= b; a_ += TEAM) {
            double s = 0.0;
            DOT_UNROLL for (int p = 0; p < nFR; p++) s += Q[p * ld + a_] * t2[FR[p]];
            w[a_] = s;
        }
        SYNC();
        }
        // r = R'^{-1} w[0..b): forward substitution, column oriented
        if constexpr (TEAM > 32) fwd_solve_R_blocked(w, b, b);
        else {
        double* rinv = V_(dy);  // dead between two homotopy steps
        QP_U1 for (int k = lane; k < b; k += TEAM) rinv[k] = 1.0 / R_(k, k);
        SYNC();
        QP_U1 for (int k = 0; k < b; k++) {
            double rk = quot(w[k], R_(k, k), rinv[k]);
            SYNC();
            if (lane == 0) R_(k, b) = rk;
            QP_U1 for (int i = k + 1 + lane; i < b; i += TEAM) w[i] -= R_(k, i) * rk;
            SYNC();
        }
        }
        double rho2 = w[b];
        if constexpr (TEAM > 32) {
            double part = 0.0;
            for (int k = lane; k < b; k += TEAM) part += R_(k, b) * R_(k, b);
            rho2 -= team_sum(part);
        } else
        {
        DOT_UNROLL for (int k = 0; k < b; k++) rho2 -= R_(k, b) * R_(k, b);
        }
        int ok = check_curvature ? (rho2 > QP_EPS_FLIP) : (rho2 > QP_ZERO);
        SYNC();  // every lane has read w[b] / R(.,b) before a caller may overwrite them (uniform decision)
        if (!ok) return 0;
        if (lane == 0) R_(b, b) = sqrt(rho2);
        QP_U1 for (int a_ = lane; a_ < b; a_ += TEAM) R_(b, a_) = 0.0;
        SYNC();
        if constexpr (TEAM > 32) extend_Dinv(b, sqrt(rho2));
        return 1;
    }

    // ---------------------------------------------------------------- working-set updates
    static __device__ QP_FN void constraint_w(int c, double& wz2, double& a2) {
        QP_CTX QP_PAT
        const int nFR = hdr[0], nAC = hdr[1], nZ = nFR - nAC;
        double *a = V_(a), *w = V_(w);
        const double *Q = V_(Q), *Av = V_(Av);
        const short* FR = FR_;
        QP_U1 for (int p = lane; p < nFR; p += TEAM) a[p] = A_entry(pat, Av, c, FR[p]);
        SYNC();
        if constexpr (TEAM > 32) {
            col_sums_auto(sA.oQ, nFR, 0, nFR, sA.oa, sA.ow, false);
            double s2p = 0.0, z2p = 0.0;
            for (int p = lane; p < nFR; p += TEAM) s2p += a[p] * a[p];
            for (int j = lane; j < nZ; j += TEAM) z2p += w[j] * w[j];
            a2 = team_sum(s2p); wz2 = team_sum(z2p);
            SYNC();
            return;
        }
        QP_U1 for (int j = lane; j < nFR; j += TEAM) {
            double s = 0.0;
            DOT_UNROLL for (int p = 0; p < nFR; p++) s += Q[p * ld + j] * a[p];
            w[j] = s;
        }
        SYNC();
        double s2 = 0.0, z2 = 0.0;
        DOT_UNROLL for (int p = 0; p < nFR; p++) s2 += a[p] * a[p];
        DOT_UNROLL for (int j = 0; j < nZ; j++) z2 += w[j] * w[j];
        wz2 = z2; a2 = s2;
        SYNC();
    }
    // Chain of rotations compressing w[0..cnt) into its last entry, rotation j acting on columns (j, j+1); writes
    // (c_j, s_j) to t2, t3 and returns the compressed value.  Formed from the running sums of squares
    // S_j = w_0^2 + ... + w_j^2 (each lane accumulates its own prefix left to right, exactly the oracle's sequence), so
    // the cnt-1 square roots and 2(cnt-1) divisions run in parallel instead of as one scalar recurrence.
    static __device__ QP_FN double rotation_chain(int cnt) {
        QP_CTX
        double *t2 = V_(t2), *t3 = V_(t3);
        const double* w = V_(w);
        QP_U1 for (int j = lane; j + 1 < cnt; j += TEAM) {
            double S = w[0] * w[0];
            bool anyprev = false;  // a non-zero entry before j: then a_j = sqrt(S_j), else a_j = w_j (signed)
            DOT_UNROLL for (int k = 1; k <= j; k++) { anyprev = anyprev || (w[k - 1] != 0.0); S = S + w[k] * w[k]; }
            const double a = anyprev ? sqrt(S) : w[j];
            if (a == 0.0) { t2[j] = 1.0; t3[j] = 0.0; }
            else { const double h = sqrt(S + w[j + 1] * w[j + 1]); t2[j] = w[j + 1] / h; t3[j] = a / h; }
        }
        // compressed value a_{cnt-1}
        double r;
        {
            const int j = cnt - 1;
            double S = w[0] * w[0];
            bool anyprev = false;
            DOT_UNROLL for (int k = 1; k <= j; k++) { anyprev = anyprev || (w[k - 1] != 0.0); S = S + w[k] * w[k]; }
            r = anyprev ? sqrt(S) : w[j];
        }
        SYNC();
        return r;
    }
    // carry_R (one-QP-per-cluster kernel): R is valid for the current working set and is updated instead of recomputed
    static __device__ QP_FN void add_constraint(int c, int status, bool carry_R = false) {
        QP_CTX
        const int nFR = hdr[0], nAC = hdr[1], nZ = nFR - nAC;
        double *Q = V_(Q), *RT = V_(RT);
        const double *t2 = V_(t2), *t3 = V_(t3), *w = V_(w);
        double r = rotation_chain(nZ);
        if constexpr (TEAM > 32) {
            rot_rows_auto(sA.oQ, nFR, nZ, sA.ot2, sA.ot3);
            if (carry_R) update_R_after_add(nZ);  // before the new row of T below: with nFR == cap it lands on row nZ-1 of R
        } else
        {
        QP_U1 for (int p = lane; p < nFR; p += TEAM) {
            double* q = Q + p * ld;
            double qa = q[0];
            QP_U1 for (int j = 0; j + 1 < nZ; j++) {
                double cs = t2[j], sn = t3[j], qb = q[j + 1];
                q[j] = cs * qa - sn * qb;
                qa = sn * qa + cs * qb;
            }
            if (nZ > 0) q[nZ - 1] = qa;
        }
        }
        QP_U1 for (int j = lane; j < nFR; j += TEAM) T_(nAC, j) = (j > nZ - 1) ? w[j] : ((j == nZ - 1) ? r : 0.0);
        if (lane == 0) { AC_[nAC] = (short)c; posAC_[c] = (short)nAC; sC_[c] = (short)status; hdr[1] = nAC + 1; }
        SYNC();
    }
    // The rotation chain of a removal, warp kernel with nAC <= TEAM.  Rotation i (i0 <= i < nAC) acts on the columns
    // (cL, cL+1), cL = c0 - i, of rows i.. of T (it zeroes T_(i, cL)) and of every row of Q.  Lane ii owns row ii of T and
    // carries in a register the entry of column cL+1 that rotation i-1 left; T_(ii, cL) is still untouched in shared memory.
    // Lane i's pair is broadcast and every lane forms (cs, sn) from it, stores the entry that became final and carries the
    // other one on.  Q is then rotated one lane per row, right to left, carrying Q[p][cL+1].  Every element sees the same
    // operations on the same operands in the same order as in the barrier-per-rotation loop of the callers (nAC > TEAM),
    // so the factors are bit-identical; the chain costs one broadcast and the givens() of one pair per rotation, and the
    // removal two barriers in all.  Ends without a barrier (the caller's next phase decides).  Needs nAC > i0.
    static __device__ QP_FN void removal_chain_regs(int i0, int c0) {
        QP_CTX
        const int nFR = hdr[0], nAC = hdr[1];
        double *Q = V_(Q), *RT = V_(RT), *t2 = V_(t2), *t3 = V_(t3);
        const unsigned tm = team_mask<TEAM>();
        constexpr int W = TEAM <= 32 ? TEAM : 32;
        const bool own = lane >= i0 && lane < nAC;
        double tb = own ? T_(lane, c0 - i0 + 1) : 0.0;  // running entry of column cL+1 of row `lane`
        QP_U1 for (int i = i0; i < nAC; i++) {
            const int cL = c0 - i;
            const bool act = own && lane >= i;
            const double ta = act ? T_(lane, cL) : 0.0;
            double cs, sn, r;
            givens(__shfl_sync(tm, ta, i, W), __shfl_sync(tm, tb, i, W), cs, sn, r);
            if (act) {
                T_(lane, cL + 1) = sn * ta + cs * tb;
                tb = cs * ta - sn * tb;
                if (lane == i) { T_(lane, cL) = 0.0; t2[i - i0] = cs; t3[i - i0] = sn; }
            }
        }
        SYNC();
        QP_U1 for (int p = lane; p < nFR; p += TEAM) {
            double* q = Q + p * ld;
            double qb = q[c0 - i0 + 1];
            QP_U1 for (int i = i0; i < nAC; i++) {
                const int cL = c0 - i;
                const double cs = t2[i - i0], sn = t3[i - i0], qa = q[cL];
                q[cL + 1] = sn * qa + cs * qb;
                qb = cs * qa - sn * qb;
            }
            q[c0 - nAC + 1] = qb;
        }
    }
    static __device__ QP_FN void remove_constraint(int c) {
        QP_CTX
        const int nFR = hdr[0], nAC = hdr[1];
        double *Q = V_(Q), *RT = V_(RT);
        short *AC = AC_, *posAC = posAC_;
        const int k = posAC[c];
        SYNC();  // every thread holds nAC and k before lane 0 rewrites them below (the loops may be empty)
        if (TEAM <= 32 && nAC <= TEAM) {
            if (k + 1 < nAC) removal_chain_regs(k + 1, nFR - 1);  // its pass over Q and the row shift of T below share a phase
        } else {
        QP_U1 for (int i = k + 1; i < nAC; i++) {
            int cL = nFR - 1 - i;
            double cs, sn, r;
            givens(T_(i, cL), T_(i, cL + 1), cs, sn, r);
            SYNC();
            QP_U1 for (int ii = i + lane; ii < nAC; ii += TEAM) {
                double ta = T_(ii, cL), tb = T_(ii, cL + 1);
                T_(ii, cL) = (ii == i) ? 0.0 : cs * ta - sn * tb;
                T_(ii, cL + 1) = sn * ta + cs * tb;
            }
            if constexpr (TEAM > 32) {  // Q is rotated afterwards, all rotations in one coalesced pass (rot_rows, right to left)
                if (lane == 0) { V_(t2)[i - k - 1] = cs; V_(t3)[i - k - 1] = -sn; }
            } else
            {
            QP_U1 for (int p = lane; p < nFR; p += TEAM) {
                double qa = Q[p * ld + cL], qb = Q[p * ld + cL + 1];
                Q[p * ld + cL] = cs * qa - sn * qb;
                Q[p * ld + cL + 1] = sn * qa + cs * qb;
            }
            }
            SYNC();
        }
        }
        if constexpr (TEAM > 32) rot_rows_auto(sA.oQ, nFR, nAC - k, sA.ot2, sA.ot3, nFR - 1 - k, -1);
        // shift rows k+1.. up by one (row i -> i-1): every thread moves its own columns, so no barrier between the rows
        QP_U1 for (int j = lane; j < nFR; j += TEAM)
            QP_U1 for (int i = k + 1; i < nAC; i++) T_(i - 1, j) = T_(i, j);
        SYNC();
        if (lane == 0) {
            QP_U1 for (int i = k + 1; i < nAC; i++) { AC[i - 1] = AC[i]; posAC[AC[i - 1]] = (short)(i - 1); }
            sC_[c] = 0; posAC[c] = -1; hdr[1] = nAC - 1;
        }
        SYNC();
    }
    static __device__ QP_FN double bound_w(int v) {
        QP_CTX
        const int nFR = hdr[0], nAC = hdr[1], nZ = nFR - nAC, p = posFR_[v];
        double* w = V_(w);
        const double* Q = V_(Q);
        QP_U1 for (int j = lane; j < nFR; j += TEAM) w[j] = Q[p * ld + j];
        SYNC();
        if constexpr (TEAM > 32) {
            double z2p = 0.0;
            for (int j = lane; j < nZ; j += TEAM) z2p += w[j] * w[j];
            const double z2s = team_sum(z2p);
            SYNC();
            return z2s;
        }
        double z2 = 0.0;
        DOT_UNROLL for (int j = 0; j < nZ; j++) z2 += w[j] * w[j];
        SYNC();
        return z2;
    }
    static __device__ QP_FN void add_bound(int v, int status, bool carry_R = false) {
        QP_CTX
        const int nFR = hdr[0], nAC = hdr[1], nZ = nFR - nAC;
        double *Q = V_(Q), *RT = V_(RT);
        const double *t2 = V_(t2), *t3 = V_(t3);
        short *FR = FR_, *posFR = posFR_;
        const int p = posFR[v];
        rotation_chain(nFR);
        if constexpr (TEAM > 32) {
            rot_rows_auto(sA.oQ, nFR, nFR, sA.ot2, sA.ot3);
            if (carry_R) update_R_after_add(nZ);  // the first nZ-1 rotations of the chain act inside the null space
        } else
        {
        QP_U1 for (int pp = lane; pp < nFR; pp += TEAM) {
            double* q = Q + pp * ld;
            double qa = q[0];
            QP_U1 for (int j = 0; j + 1 < nFR; j++) {
                double cs = t2[j], sn = t3[j], qb = q[j + 1];
                q[j] = cs * qa - sn * qb;
                qa = sn * qa + cs * qb;
            }
            q[nFR - 1] = qa;
        }
        }
        // T rows: row i is touched by rotations j >= nFR-2-i (and j >= nZ-1)
        QP_U1 for (int i = lane; i < nAC; i += TEAM) {
            int j0 = nFR - 2 - i; if (j0 < nZ - 1) j0 = nZ - 1; if (j0 < 0) j0 = 0;
            double ta = T_(i, j0);
            QP_U1 for (int j = j0; j + 1 < nFR; j++) {
                double cs = t2[j], sn = t3[j], tb = T_(i, j + 1);
                T_(i, j) = cs * ta - sn * tb;
                ta = sn * ta + cs * tb;
            }
            T_(i, nFR - 1) = ta;
        }
        SYNC();
        const int last = nFR - 1;
        if (p != last) {
            QP_U1 for (int j = lane; j < nFR - 1; j += TEAM) Q[p * ld + j] = Q[last * ld + j];
            if (lane == 0) { short vl = FR[last]; FR[p] = vl; posFR[vl] = (short)p; }
        }
        if (lane == 0) { posFR[v] = -1; sB_[v] = (short)status; hdr[0] = nFR - 1; }
        SYNC();
    }
    // returns 1 (warp-uniform) if the factors cannot hold one more free variable
    static __device__ QP_FN int remove_bound(int v) {
        QP_CTX QP_PAT
        int nFR = hdr[0];
        const int nAC = hdr[1];
        if (nFR + 1 > cap) return 1;
        double *Q = V_(Q), *RT = V_(RT);
        const double* Av = V_(Av);
        const pidx *Ap = pat + sA.pAp, *Ai = pat + sA.pAi;
        const short* AC = AC_;
        SYNC();  // all lanes have read hdr[0] before lane 0 updates it below
        QP_U1 for (int j = lane; j < nFR; j += TEAM) { Q[nFR * ld + j] = 0.0; Q[j * ld + nFR] = 0.0; }
        QP_U1 for (int i = lane; i < nAC; i += TEAM) {
            int r = AC[i];
            double s = 0.0;
            int e1 = Ap[v + 1];
            QP_U1 for (int e = Ap[v]; e < e1; e++)
                if (Ai[e] == r) s += Av[e];
            T_(i, nFR) = s;
        }
        if (lane == 0) { Q[nFR * ld + nFR] = 1.0; FR_[nFR] = (short)v; posFR_[v] = (short)nFR; sB_[v] = 0; hdr[0] = nFR + 1; if (nFR + 1 > hdr[6]) hdr[6] = nFR + 1; }
        nFR++;
        SYNC();
        if (TEAM <= 32 && nAC <= TEAM) {
            if (nAC > 0) { removal_chain_regs(0, nFR - 2); SYNC(); }
            return 0;
        }
        QP_U1 for (int i = 0; i < nAC; i++) {
            int cL = nFR - 2 - i;
            double cs, sn, r;
            givens(T_(i, cL), T_(i, cL + 1), cs, sn, r);
            SYNC();
            QP_U1 for (int ii = i + lane; ii < nAC; ii += TEAM) {
                double ta = T_(ii, cL), tb = T_(ii, cL + 1);
                T_(ii, cL) = (ii == i) ? 0.0 : cs * ta - sn * tb;
                T_(ii, cL + 1) = sn * ta + cs * tb;
            }
            if constexpr (TEAM > 32) {
                if (lane == 0) { V_(t2)[i] = cs; V_(t3)[i] = -sn; }
            } else
            {
            QP_U1 for (int p = lane; p < nFR; p += TEAM) {
                double qa = Q[p * ld + cL], qb = Q[p * ld + cL + 1];
                Q[p * ld + cL] = cs * qa - sn * qb;
                Q[p * ld + cL + 1] = sn * qa + cs * qb;
            }
            }
            SYNC();
        }
        if constexpr (TEAM > 32) rot_rows_auto(sA.oQ, nFR, nAC + 1, sA.ot2, sA.ot3, nFR - 1, -1);
        return 0;
    }

    // ---------------------------------------------------------------- T solves
    // T v = b : v indexed by Q column; row i has its diagonal at column nFR-1-i.  b (by AC position) is destroyed.
    static __device__ QP_FN void solve_T(double* b, double* v) {
        QP_CTX
        const int nFR = hdr[0], nAC = hdr[1];
        const double* RT = V_(RT);
        if constexpr (TEAM > 32) { solve_T_blocked(b, v); return; }
        if (TEAM <= 32 && nAC <= TEAM) {
            // whole right-hand side in registers (lane k holds b_k and its pivot): the substitution chain is one shuffle and
            // the three operations of quot() per unknown, no barrier and no shared-memory round trip.  Same operations on
            // the same operands in the same order as the loop below (and the oracle).
            const bool act = lane < nAC;
            double bk = act ? b[lane] : 0.0;
            const double piv = act ? T_(lane, nFR - 1 - lane) : 1.0, ri = 1.0 / piv;
            QP_U1 for (int i = 0; i < nAC; i++) {
                const int d = nFR - 1 - i;
                const double tkd = (lane > i && act) ? T_(lane, d) : 0.0;
                const double vi = __shfl_sync(team_mask<TEAM>(), quot(bk, piv, ri), i, TEAM <= 32 ? TEAM : 32);
                if (lane == i) v[d] = vi;
                if (lane > i && act) bk -= tkd * vi;
            }
            SYNC();
            return;
        }
        double* rinv = V_(dAx);  // pivot reciprocals, one per lane in parallel: the sequential part below only multiplies
        QP_U1 for (int i = lane; i < nAC; i += TEAM) rinv[i] = 1.0 / T_(i, nFR - 1 - i);
        SYNC();
        QP_U1 for (int i = 0; i < nAC; i++) {
            int d = nFR - 1 - i;
            double vi = quot(b[i], T_(i, d), rinv[i]);
            SYNC();
            if (lane == 0) v[d] = vi;
            QP_U1 for (int k = i + 1 + lane; k < nAC; k += TEAM) b[k] -= T_(k, d) * vi;
            SYNC();
        }
    }
    // T' u = r : r indexed by Q column (destroyed), u by AC position
    static __device__ QP_FN void solve_Tt(double* r, double* u) {
        QP_CTX
        const int nFR = hdr[0], nAC = hdr[1];
        const double* RT = V_(RT);
        if constexpr (TEAM > 32) { solve_Tt_blocked(r, u); return; }
        if (TEAM <= 32 && nAC <= TEAM) {  // register form, see solve_T
            const bool act = lane < nAC;
            double rk = act ? r[nFR - 1 - lane] : 0.0;
            const double piv = act ? T_(lane, nFR - 1 - lane) : 1.0, ri = 1.0 / piv;
            QP_U1 for (int i = nAC - 1; i >= 0; i--) {
                const double tik = (lane < i) ? T_(i, nFR - 1 - lane) : 0.0;
                const double ui = __shfl_sync(team_mask<TEAM>(), quot(rk, piv, ri), i, TEAM <= 32 ? TEAM : 32);
                if (lane == i) u[i] = ui;
                if (lane < i) rk -= tik * ui;
            }
            SYNC();
            return;
        }
        double* rinv = V_(dAx);
        QP_U1 for (int i = lane; i < nAC; i += TEAM) rinv[i] = 1.0 / T_(i, nFR - 1 - i);
        SYNC();
        QP_U1 for (int i = nAC - 1; i >= 0; i--) {
            int d = nFR - 1 - i;
            double ui = quot(r[d], T_(i, d), rinv[i]);
            SYNC();
            if (lane == 0) u[i] = ui;
            QP_U1 for (int k = lane; k < i; k += TEAM) { int dk = nFR - 1 - k; r[dk] -= T_(i, dk) * ui; }
            SYNC();
        }
    }

    // ---------------------------------------------------------------- step direction
    // dxFX: full-length vector holding the bound shift of every fixed variable; dbAC by AC position; dgvec: gradient shift.
    // Writes dx, dy and dAx = A dx.  The first loop reads only the entries of dxFX (and the caller's dbAC, dgvec) that the
    // same lane wrote, so the caller needs no barrier between setting them up and this call; a product is formed by the lane
    // that consumes its entry wherever the lane mappings allow it (same terms, same order as mulA / mulH / mulAT).
    static __device__ QP_FN void step_direction(const double* dgvec, const double* dxFX, double* dbAC) {
        QP_CTX QP_PAT
        const int nT = nV + nC;
        const int nFR = hdr[0], nAC = hdr[1], nZ = nFR - nAC;
        double *dx = V_(dx), *dy = V_(dy), *dAx = V_(dAx), *t1 = V_(t1), *t3 = V_(t3), *yv = V_(yv), *zv = V_(zv);
        const double *Q = V_(Q), *RT = V_(RT), *Av = V_(Av), *Hv = V_(Hv);
        const short *sB = sB_, *FR = FR_, *AC = AC_;
        QP_U1 for (int i = lane; i < nV; i += TEAM) dx[i] = (sB[i] != 0) ? dxFX[i] : 0.0;
        SYNC();
        if (nAC > 0) {
            QP_U1 for (int i = lane; i < nAC; i += TEAM) t3[i] = dbAC[i] - A_row(pat, Av, dx, AC[i]);
            SYNC();
            solve_T(t3, yv);
            if constexpr (TEAM > 32) row_sums_auto(sA.oQ, nFR, nZ, nFR, sA.oyv, sA.odx, true, false);
            else
            {
            QP_U1 for (int p = lane; p < nFR; p += TEAM) {
                double s = 0.0;
                DOT_UNROLL for (int j = nZ; j < nFR; j++) s += Q[p * ld + j] * yv[j];
                dx[FR[p]] = s;
            }
            SYNC();
            }
        }
        if (nZ > 0) {
            mulH(dx, t1);
            if constexpr (TEAM > 32) {
                for (int p = lane; p < nFR; p += TEAM) { const int v = FR[p]; yv[p] = t1[v] + dgvec[v]; }  // yv is dead here
                SYNC();
                col_sums_auto(sA.oQ, nFR, 0, nZ, sA.oyv, sA.ozv, true);
            } else
            {
            double* rinv = V_(dy);  // pivot reciprocals of the substitutions below (dy is dead here, rewritten below)
            QP_U1 for (int j = lane; j < nZ; j += TEAM) {
                double s = 0.0;
                DOT_UNROLL for (int p = 0; p < nFR; p++) { int v = FR[p]; s += Q[p * ld + j] * (t1[v] + dgvec[v]); }
                zv[j] = -s;
                rinv[j] = 1.0 / R_(j, j);
            }
            SYNC();
            }
            // R' u = rhs (forward), R z = u (backward); column oriented
            PROF2_T0
            if constexpr (TEAM > 32) {
                fwd_solve_R_blocked(zv, nZ, -1);
                bwd_solve_R_blocked(zv, nZ);
                PROF2_ADD(PR_RSOLVE);
            } else {
                const double* rinv = V_(dy);
                QP_U1 for (int k = 0; k < nZ; k++) {
                    double uk = quot(zv[k], R_(k, k), rinv[k]);
                    SYNC();
                    if (lane == 0) zv[k] = uk;
                    QP_U1 for (int i = k + 1 + lane; i < nZ; i += TEAM) zv[i] -= R_(k, i) * uk;
                    SYNC();
                }
                QP_U1 for (int k = nZ - 1; k >= 0; k--) {
                    double zk = quot(zv[k], R_(k, k), rinv[k]);
                    SYNC();
                    if (lane == 0) zv[k] = zk;
                    QP_U1 for (int i = lane; i < k; i += TEAM) zv[i] -= R_(i, k) * zk;
                    SYNC();
                }
                PROF2_ADD(PR_RSOLVE);
            }
            if constexpr (TEAM > 32) row_sums_auto(sA.oQ, nFR, 0, nZ, sA.ozv, sA.odx, true, true);
            else
            {
            QP_U1 for (int p = lane; p < nFR; p += TEAM) {
                double s = 0.0;
                DOT_UNROLL for (int j = 0; j < nZ; j++) s += Q[p * ld + j] * zv[j];
                dx[FR[p]] += s;
            }
            SYNC();
            }
        }
        QP_U1 for (int i = lane; i < nV; i += TEAM) t1[i] = H_row(pat, Hv, dx, i) + dgvec[i];
        QP_U1 for (int i = lane; i < nT; i += TEAM) dy[i] = 0.0;
        SYNC();
        if (nAC > 0) {
            if constexpr (TEAM > 32) {
                for (int p = lane; p < nFR; p += TEAM) zv[p] = t1[FR[p]];  // zv is dead here
                SYNC();
                col_sums_auto(sA.oQ, nFR, nZ, nFR, sA.ozv, sA.oyv, false);
            } else
            {
            QP_U1 for (int j = nZ + lane; j < nFR; j += TEAM) {
                double s = 0.0;
                DOT_UNROLL for (int p = 0; p < nFR; p++) s += Q[p * ld + j] * t1[FR[p]];
                yv[j] = s;
            }
            SYNC();
            }
            solve_Tt(yv, t3);
            QP_U1 for (int i = lane; i < nAC; i += TEAM) dy[nV + AC[i]] = t3[i];
            SYNC();
            QP_U1 for (int i = lane; i < nV; i += TEAM) if (sB[i] != 0) dy[i] = t1[i] - AT_col(pat, Av, dy + nV, i);
        } else {
            QP_U1 for (int i = lane; i < nV; i += TEAM) if (sB[i] != 0) dy[i] = t1[i];
        }
        QP_U1 for (int r = lane; r < nC; r += TEAM) dAx[r] = A_row(pat, Av, dx, r);
        SYNC();
    }

    // ---------------------------------------------------------------- drift correction / ramping
    // g = A'y_c + y_b - (H+regI) x, second phase: t1 = (H+regI) x is complete, and so is y.  One lane per column forms the
    // column's product with y_c and combines it with the entries of y and t1 that the same lane wrote in the first phase.
    static __device__ QP_FN void stationarity_gradient_tail() {
        QP_CTX QP_PAT
        double* g = V_(g);
        const double *t1 = V_(t1), *y = V_(y), *Av = V_(Av);
        QP_U1 for (int i = lane; i < nV; i += TEAM) g[i] = AT_col(pat, Av, y + nV, i) + y[i] - t1[i];
        SYNC();
    }
    static __device__ QP_FN void stationarity_gradient() {  // g = A'y_c + y_b - (H+regI) x
        QP_CTX
        mulH(V_(x), V_(t1));
        stationarity_gradient_tail();
    }
    // Two phases: (1) A x, the bounds and the clamped multipliers, each lane on the entries it owns, and t1 = (H+regI) x;
    // (2) the gradient (stationarity_gradient_tail).  The clamps of y depend only on the statuses and y itself, and lane r
    // updates lbA[r] / ubA[r] from the (A x)[r] it holds in a register.
    static __device__ QP_FN void drift_correction() {
        QP_CTX QP_PAT
        double *x = V_(x), *y = V_(y), *Ax = V_(Ax), *lb = V_(lb), *ub = V_(ub), *lbA = V_(lbA), *ubA = V_(ubA), *t1 = V_(t1);
        const double *Av = V_(Av), *Hv = V_(Hv);
        const short *sB = sB_, *sC = sC_;
        QP_U1 for (int i = lane; i < nV; i += TEAM) {
            int s = sB[i]; double xi = x[i];
            if (s < 0) { lb[i] = xi; if (ub[i] < xi) ub[i] = xi; if (y[i] < 0) y[i] = 0.0; }
            else if (s > 0) { ub[i] = xi; if (lb[i] > xi) lb[i] = xi; if (y[i] > 0) y[i] = 0.0; }
            else { if (lb[i] > xi) lb[i] = xi; if (ub[i] < xi) ub[i] = xi; y[i] = 0.0; }
            t1[i] = H_row(pat, Hv, x, i);
        }
        QP_U1 for (int i = lane; i < nC; i += TEAM) {
            int s = sC[i]; double ax = A_row(pat, Av, x, i);
            Ax[i] = ax;
            if (s < 0) { lbA[i] = ax; if (ubA[i] < ax) ubA[i] = ax; if (y[nV + i] < 0) y[nV + i] = 0.0; }
            else if (s > 0) { ubA[i] = ax; if (lbA[i] > ax) lbA[i] = ax; if (y[nV + i] > 0) y[nV + i] = 0.0; }
            else { if (lbA[i] > ax) lbA[i] = ax; if (ubA[i] < ax) ubA[i] = ax; y[nV + i] = 0.0; }
        }
        SYNC();
        stationarity_gradient_tail();
    }
    static __device__ QP_FN void ramping() {  // same two phases as drift_correction
        QP_CTX QP_PAT
        double *x = V_(x), *y = V_(y), *Ax = V_(Ax), *lb = V_(lb), *ub = V_(ub), *lbA = V_(lbA), *ubA = V_(ubA), *t1 = V_(t1);
        const double *Av = V_(Av), *Hv = V_(Hv);
        const short *sB = sB_, *sC = sC_;
        const int ramp_offset = hdr[2];
        const int nRamp = nV + nC + nC + nV;
        const double r0 = 0.5, r1 = 1.0;
        QP_U1 for (int i = lane; i < nV; i += TEAM) {
            double tP = (double)((i + ramp_offset) % nRamp) / (double)(nRamp - 1);
            double rP = (1.0 - tP) * r0 + tP * r1;
            double tD = (double)((nV + nC + i + ramp_offset) % nRamp) / (double)(nRamp - 1);
            double rD = (1.0 - tD) * r0 + tD * r1;
            double xi = x[i];
            double sca = fabs(xi) > 1.0 ? fabs(xi) : 1.0;
            int s = sB[i];
            if (s >= 0) lb[i] = xi - sca * rP;
            if (s <= 0) ub[i] = xi + sca * rP;
            if (s < 0) { lb[i] = xi; y[i] = rD; }
            if (s > 0) { ub[i] = xi; y[i] = -rD; }
            if (s == 0) y[i] = 0.0;
            t1[i] = H_row(pat, Hv, x, i);
        }
        QP_U1 for (int i = lane; i < nC; i += TEAM) {
            double tP = (double)((nV + i + ramp_offset) % nRamp) / (double)(nRamp - 1);
            double rP = (1.0 - tP) * r0 + tP * r1;
            double tD = (double)((nV + nC + nV + i + ramp_offset) % nRamp) / (double)(nRamp - 1);
            double rD = (1.0 - tD) * r0 + tD * r1;
            double ax = A_row(pat, Av, x, i);
            Ax[i] = ax;
            double sca = fabs(ax) > 1.0 ? fabs(ax) : 1.0;
            int s = sC[i];
            if (s >= 0) lbA[i] = ax - sca * rP;
            if (s <= 0) ubA[i] = ax + sca * rP;
            if (s < 0) { lbA[i] = ax; y[nV + i] = rD; }
            if (s > 0) { ubA[i] = ax; y[nV + i] = -rD; }
            if (s == 0) y[nV + i] = 0.0;
        }
        SYNC();  // also: every lane has read ramp_offset
        if (lane == 0) hdr[2] = ramp_offset + 1;
        stationarity_gradient_tail();
    }

    // ---------------------------------------------------------------- exchange (ensure LI)
    // element to add: constraint c (v<0) or bound v (c<0); w holds its Q-coordinates. 0 ok, 1 infeasible, 2 capacity
    static __device__ QP_FN int ensure_li(int c, int v, int status) {
        QP_CTX QP_PAT
        const int nFR = hdr[0], nAC = hdr[1], nZ = nFR - nAC;
        double *xiC = V_(zv), *xiB = V_(dx), *t3 = V_(t3), *y = V_(y), *w = V_(w);
        const double* Av = V_(Av);
        const short *sB = sB_, *sC = sC_, *AC = AC_, *posAC = posAC_;
        (void)nZ;
        solve_Tt(w, xiC);  // may destroy w[nZ..nFR): the caller forms w again after the exchange
        QP_U1 for (int i = lane; i < nC; i += TEAM) { int p = posAC[i]; t3[i] = (p >= 0) ? xiC[p] : 0.0; }
        SYNC();
        QP_U1 for (int i = lane; i < nV; i += TEAM) {
            if (sB[i] == 0) { xiB[i] = 0.0; continue; }
            double ai = (c >= 0) ? A_entry(pat, Av, c, i) : 0.0;
            xiB[i] = ai - AT_col(pat, Av, t3, i);
        }
        // no barrier: the scan reads only the xiB[i] this lane wrote, and xiC, complete since solve_Tt's barrier
        const double sgn = (status < 0) ? 1.0 : -1.0;
        double best = QP_INFTY; int bpos = 0x7fffffff;
        QP_U1 for (int i = lane; i < nAC; i += TEAM) {
            int ci = AC[i]; double xi = sgn * xiC[i], yy = y[nV + ci]; double t = QP_INFTY;
            if (sC[ci] < 0) { if (xi > QP_ZERO && yy >= 0.0) t = yy / xi; }
            else { if (xi < -QP_ZERO && yy <= 0.0) t = yy / xi; }
            if (t < QP_INFTY && key_less(t, i, best, bpos)) { best = t; bpos = i; }
        }
        QP_U1 for (int i = lane; i < nV; i += TEAM) {
            if (sB[i] == 0) continue;
            double xi = sgn * xiB[i], yy = y[i]; double t = QP_INFTY;
            if (sB[i] < 0) { if (xi > QP_ZERO && yy >= 0.0) t = yy / xi; }
            else { if (xi < -QP_ZERO && yy <= 0.0) t = yy / xi; }
            if (t < QP_INFTY && key_less(t, nC + i, best, bpos)) { best = t; bpos = nC + i; }
        }
        MinKey mk = team_min(best, bpos);
        if (mk.pos == 0x7fffffff) return 1;
        const double ymin = mk.t;
        const int kind = mk.pos >= nC ? 1 : 0;
        const int idx = kind ? mk.pos - nC : AC[mk.pos];
        SYNC();
        QP_U1 for (int i = lane; i < nAC; i += TEAM) y[nV + AC[i]] -= ymin * sgn * xiC[i];
        QP_U1 for (int i = lane; i < nV; i += TEAM) if (sB[i] != 0) y[i] -= ymin * sgn * xiB[i];
        SYNC();
        if (lane == 0) {
            if (c >= 0) y[nV + c] = sgn * ymin; else y[v] = sgn * ymin;
            if (kind == 0) y[nV + idx] = 0.0; else y[idx] = 0.0;
        }
        SYNC();
        if (kind == 0) remove_constraint(idx); else if (remove_bound(idx)) return 2;
        return 0;
    }

    // ---------------------------------------------------------------- homotopy
    static __device__ QP_FN int homotopy(int max_iter, int& iters) {
        QP_CTX
        const int nT = nV + nC;
        const int flags = sA.flags;
        int carried = 0;  // additions since R was last recomputed (one-QP-per-cluster kernel)
        double *x = V_(x), *y = V_(y), *Ax = V_(Ax), *g = V_(g), *lb = V_(lb), *ub = V_(ub), *lbA = V_(lbA), *ubA = V_(ubA);
        double *dx = V_(dx), *dy = V_(dy), *dAx = V_(dAx), *w = V_(w), *a = V_(a);
        const double *gN = V_(gN), *lbN = V_(lbN), *ubN = V_(ubN), *lbAN = V_(lbAN), *ubAN = V_(ubAN);
        short *sB = sB_, *sC = sC_, *AC = AC_;
        iters = 0;
        PROF_T0
        QP_U1 for (int it = 0;; it++) {
            const int nAC = hdr[1];
            // w[0..nV) <- bound shift of fixed variables, w[nV..) <- constraint shift by AC position, a <- dg
            QP_U1 for (int i = lane; i < nV; i += TEAM) {
                int s = sB[i];
                w[i] = s < 0 ? (lbN[i] - lb[i]) : (s > 0 ? (ubN[i] - ub[i]) : 0.0);
                a[i] = gN[i] - g[i];
            }
            QP_U1 for (int i = lane; i < nAC; i += TEAM) { int ci = AC[i]; w[nV + i] = sC[ci] < 0 ? (lbAN[ci] - lbA[ci]) : (ubAN[ci] - ubA[ci]); }
            step_direction(a, w, w + nV);  // reads w[i] of this lane before its first barrier (no barrier needed here); dAx too
            PROF_ADD(PR_STEPDIR);

            // ---- ratio tests: position = scan order of the sequential rule
            double best = 2.0; int bpos = 0x7fffffff;
#define CONSIDER(num, den, pos)                                                                   \
    {                                                                                             \
        double n_ = (num), d_ = (den);                                                            \
        if (d_ >= QP_EPS_DEN && n_ >= QP_EPS_NUM && n_ < d_) {                                    \
            double t_ = n_ / d_;                                                                  \
            if (t_ < 1.0 && key_less(t_, (pos), best, bpos)) { best = t_; bpos = (pos); }         \
        }                                                                                         \
    }
            QP_U1 for (int i = lane; i < nAC; i += TEAM) {
                int ci = AC[i];
                if (sC[ci] < 0) CONSIDER(y[nV + ci], -dy[nV + ci], i) else CONSIDER(-y[nV + ci], dy[nV + ci], i)
            }
            QP_U1 for (int i = lane; i < nV; i += TEAM) {
                int s = sB[i];
                if (s == 0) continue;
                if (s < 0) CONSIDER(y[i], -dy[i], nC + i) else CONSIDER(-y[i], dy[i], nC + i)
            }
            QP_U1 for (int i = lane; i < nC; i += TEAM) {
                if (sC[i] != 0) continue;
                double num = Ax[i] - lbA[i]; if (num < 0) num = 0;
                CONSIDER(num, (lbAN[i] - lbA[i]) - dAx[i], nC + nV + i)
                num = ubA[i] - Ax[i]; if (num < 0) num = 0;
                CONSIDER(num, dAx[i] - (ubAN[i] - ubA[i]), nC + nV + nC + i)
            }
            QP_U1 for (int i = lane; i < nV; i += TEAM) {
                if (sB[i] != 0) continue;
                double num = x[i] - lb[i]; if (num < 0) num = 0;
                CONSIDER(num, (lbN[i] - lb[i]) - dx[i], 2 * nC + nV + nC + i)
                num = ub[i] - x[i]; if (num < 0) num = 0;
                CONSIDER(num, dx[i] - (ubN[i] - ub[i]), 3 * nC + 2 * nV + i)
            }
#undef CONSIDER
            MinKey mk = team_min(best, bpos);
            double tau = 1.0; int bc_idx = -1, bc_isbound = 0, bc_status = 0;
            if (mk.pos != 0x7fffffff) {
                tau = mk.t;
                int p = mk.pos;
                if (p < nC) { bc_idx = AC[p]; bc_isbound = 0; bc_status = 0; }
                else if (p < nC + nV) { bc_idx = p - nC; bc_isbound = 1; bc_status = 0; }
                else if (p < 2 * nC + nV) { bc_idx = p - nC - nV; bc_isbound = 0; bc_status = -1; }
                else if (p < 3 * nC + nV) { bc_idx = p - 2 * nC - nV; bc_isbound = 0; bc_status = 1; }
                else if (p < 3 * nC + 2 * nV) { bc_idx = p - 3 * nC - nV; bc_isbound = 1; bc_status = -1; }
                else { bc_idx = p - 3 * nC - 2 * nV; bc_isbound = 1; bc_status = 1; }
            }
            SYNC();
            PROF_ADD(PR_RATIO);
            // ---- step
            if (bc_idx < 0) {
                QP_U1 for (int i = lane; i < nV; i += TEAM) { x[i] += dx[i]; g[i] = gN[i]; lb[i] = lbN[i]; ub[i] = ubN[i]; }
                QP_U1 for (int i = lane; i < nT; i += TEAM) y[i] += dy[i];
                QP_U1 for (int i = lane; i < nC; i += TEAM) { Ax[i] += dAx[i]; lbA[i] = lbAN[i]; ubA[i] = ubAN[i]; }
                SYNC();
                iters = it;
                return ST_OPTIMAL;
            }
            if (it >= max_iter) { iters = it; return ST_HOMOTOPY; }
            if (tau > 0.0) {
                QP_U1 for (int i = lane; i < nV; i += TEAM) {
                    x[i] += tau * dx[i]; g[i] += tau * a[i];
                    lb[i] += tau * (lbN[i] - lb[i]); ub[i] += tau * (ubN[i] - ub[i]);
                }
                QP_U1 for (int i = lane; i < nT; i += TEAM) y[i] += tau * dy[i];
                QP_U1 for (int i = lane; i < nC; i += TEAM) {
                    Ax[i] += tau * dAx[i];
                    lbA[i] += tau * (lbAN[i] - lbA[i]); ubA[i] += tau * (ubAN[i] - ubA[i]);
                }
                SYNC();
            }
            PROF_ADD(PR_STEP);
            // ---- change the working set
            if (bc_status == 0) {
                int flipped = 0;
                if (bc_isbound) {
                    int old = sB[bc_idx];
                    SYNC();
                    if (lane == 0) y[bc_idx] = 0.0;
                    SYNC();
                    if (remove_bound(bc_idx)) { iters = it; return ST_CAPACITY; }
                    PROF_ADD(PR_REMOVE);
                    const int ext_ok = extend_R(flags & FLAG_FLIPPING);
                    PROF_ADD(PR_EXTEND);
                    if (!ext_ok) {
                        if (!(flags & FLAG_FLIPPING)) { iters = it; return ST_UNBOUNDED; }
                        bound_w(bc_idx);
                        add_bound(bc_idx, -old);
                        if (lane == 0) { if (old < 0) ub[bc_idx] = x[bc_idx]; else lb[bc_idx] = x[bc_idx]; }
                        SYNC();
                        flipped = 1;
                    }
                } else {
                    int old = sC[bc_idx];
                    SYNC();
                    if (lane == 0) y[nV + bc_idx] = 0.0;
                    SYNC();
                    remove_constraint(bc_idx);
                    PROF_ADD(PR_REMOVE);
                    const int ext_ok = extend_R(flags & FLAG_FLIPPING);
                    PROF_ADD(PR_EXTEND);
                    if (!ext_ok) {
                        if (!(flags & FLAG_FLIPPING)) { iters = it; return ST_UNBOUNDED; }
                        double z2, a2;
                        constraint_w(bc_idx, z2, a2);
                        add_constraint(bc_idx, -old);
                        if (lane == 0) { if (old < 0) ubA[bc_idx] = Ax[bc_idx]; else lbA[bc_idx] = Ax[bc_idx]; }
                        SYNC();
                        flipped = 1;
                    }
                }
                if (flipped) {
                    PROF_ADD(PR_ADD);
                    if (recompute_R()) { iters = it; return ST_INTERNAL; }
                    PROF_RESET
                }
            } else {
                // one-QP-per-cluster kernel: R is carried through the addition (update_R_after_add) unless an exchange step left
                // it one column short or REFAC_EVERY updates have accumulated
                bool carry = false;
                if constexpr (TEAM > 32) carry = !sA.is_lp && carried < REFAC_EVERY && hdr[0] - hdr[1] <= UPDATE_MAX_NZ && !(sA.flags & FLAG_NO_CARRY);
                if (bc_isbound) {
                    double z2 = bound_w(bc_idx);
                    PROF_ADD(PR_WVEC);
                    if (!(z2 > QP_EPS_LI * QP_EPS_LI)) {
                        int e_ = ensure_li(-1, bc_idx, bc_status);
                        if (e_) { iters = it; return e_ == 2 ? ST_CAPACITY : ST_INFEASIBLE; }
                        bound_w(bc_idx);
                        carry = false;
                        PROF_ADD(PR_ENSURE_LI);
                    }
                    add_bound(bc_idx, bc_status, carry);
                    PROF_ADD(PR_ADD);
                } else {
                    double z2, a2;
                    constraint_w(bc_idx, z2, a2);
                    PROF_ADD(PR_WVEC);
                    if (!(z2 > QP_EPS_LI * QP_EPS_LI * a2) || a2 == 0.0) {
                        int e_ = ensure_li(bc_idx, -1, bc_status);
                        if (e_) { iters = it; return e_ == 2 ? ST_CAPACITY : ST_INFEASIBLE; }
                        constraint_w(bc_idx, z2, a2);
                        carry = false;
                        PROF_ADD(PR_ENSURE_LI);
                    }
                    add_constraint(bc_idx, bc_status, carry);
                    PROF_ADD(PR_ADD);
                }
                if (carry) carried++;
                else {
                    if (recompute_R()) { iters = it; return ST_INTERNAL; }
                    carried = 0;
                }
                PROF_RESET
            }
            if (tau <= QP_EPS && (flags & FLAG_RAMPING)) ramping();
            else if (flags & FLAG_DRIFT) drift_correction();
            PROF_ADD(PR_DRIFT);
        }
    }

    // ---------------------------------------------------------------- cold start / refactorise
    static __device__ QP_FN void cold_start_state() {
        QP_CTX
        double *x = V_(x), *y = V_(y), *Ax = V_(Ax), *g = V_(g), *lb = V_(lb), *ub = V_(ub), *lbA = V_(lbA), *ubA = V_(ubA);
        short *sB = sB_, *sC = sC_, *posFR = posFR_, *posAC = posAC_;
        QP_U1 for (int i = lane; i < nV; i += TEAM) {
            x[i] = 0.0; y[i] = 0.0; sB[i] = -1; posFR[i] = -1; g[i] = 0.0; lb[i] = 0.0; ub[i] = QP_BOUND_RELAX;
        }
        QP_U1 for (int i = lane; i < nC; i += TEAM) {
            y[nV + i] = 0.0; sC[i] = 0; posAC[i] = -1; Ax[i] = 0.0; lbA[i] = -QP_BOUND_RELAX; ubA[i] = QP_BOUND_RELAX;
        }
        if (lane == 0) { hdr[0] = 0; hdr[1] = 0; hdr[2] = 0; hdr[6] = 0; }
        SYNC();
    }
    // rebuild TQ and R for the kept working set with the new matrix values; 0 ok
    static __device__ QP_FN int refactorise() {
        QP_CTX
        const int nFR = hdr[0], nAC_old = hdr[1];
        double *Q = V_(Q), *dAx = V_(dAx), *dy = V_(dy), *y = V_(y);
        short *sC = sC_, *AC = AC_, *posAC = posAC_;
        // remember (constraint, status) by AC position in dAx (nC) and dy[nV..] (nC): neither is touched below
        QP_U1 for (int i = lane; i < nAC_old; i += TEAM) { int ci = AC[i]; dAx[i] = (double)ci; dy[nV + i] = (double)sC[ci]; }
        SYNC();
        QP_U1 for (int k = lane; k < nFR * nFR; k += TEAM) { int i = k / nFR, j = k % nFR; Q[i * ld + j] = (i == j) ? 1.0 : 0.0; }
        QP_U1 for (int i = lane; i < nAC_old; i += TEAM) { int ci = (int)dAx[i]; sC[ci] = 0; posAC[ci] = -1; }
        if (lane == 0) hdr[1] = 0;
        SYNC();
        QP_U1 for (int i = 0; i < nAC_old; i++) {
            int ci = (int)dAx[i]; int st = (int)dy[nV + i];
            double z2, a2;
            constraint_w(ci, z2, a2);
            if (!(z2 > QP_EPS_LI * QP_EPS_LI * a2) || a2 == 0.0) { if (lane == 0) y[nV + ci] = 0.0; SYNC(); continue; }
            add_constraint(ci, st);
        }
        return recompute_R();
    }

    // Auxiliary QP of an init from a guess (qpOASES solveInitialQP as reached from src/qpOASESInterface.cpp:202-207 and :716-729).
    // The caller has set x, y, A x, the wanted bound statuses sB and the wanted constraint statuses (as doubles in dy[nV..]).
    // Working set: bounds first, then the constraints in index order, linearly dependent ones left out; auxiliary bounds tight
    // on the active side and relaxed by boundRelaxation elsewhere -- a constraint left out for dependence keeps its wanted side
    // tight; gradient from stationarity.  Returns 0, 1 (projected Hessian not positive definite) or 2 (factor capacity).
    static __device__ QP_FN int aux_qp_from_guess() {
        QP_CTX
        double *x = V_(x), *Ax = V_(Ax), *lb = V_(lb), *ub = V_(ub), *lbA = V_(lbA), *ubA = V_(ubA), *Q = V_(Q);
        const double* want = V_(dy) + nV;
        short *sB = sB_, *sC = sC_, *FR = FR_, *posFR = posFR_, *posAC = posAC_;
        QP_U1 for (int i = lane; i < nV; i += TEAM) {
            const double xi = x[i];
            const int st = sB[i];
            posFR[i] = -1;
            lb[i] = (st < 0) ? xi : xi - QP_BOUND_RELAX;
            ub[i] = (st > 0) ? xi : xi + QP_BOUND_RELAX;
        }
        QP_U1 for (int i = lane; i < nC; i += TEAM) {
            const double ax = Ax[i], st = want[i];
            sC[i] = 0; posAC[i] = -1;
            lbA[i] = (st < 0.0) ? ax : ax - QP_BOUND_RELAX;
            ubA[i] = (st > 0.0) ? ax : ax + QP_BOUND_RELAX;
        }
        SYNC();
        if (lane == 0) {
            int nf = 0;
            QP_U1 for (int i = 0; i < nV; i++) if (sB[i] == 0) { if (nf < cap) FR[nf] = (short)i; posFR[i] = (short)nf; nf++; }
            hdr[0] = nf; hdr[1] = 0; hdr[2] = 0;
            if (nf > hdr[6]) hdr[6] = nf;
        }
        SYNC();
        const int nFR = hdr[0];
        if (nFR > cap) return 2;
        QP_U1 for (int k = lane; k < nFR * nFR; k += TEAM) { const int i = k / nFR, j = k % nFR; Q[i * ld + j] = (i == j) ? 1.0 : 0.0; }
        SYNC();
        QP_U1 for (int i = 0; i < nC; i++) {
            const int st = (int)want[i];
            if (st == 0 || hdr[1] >= hdr[0]) continue;
            double z2, a2;
            constraint_w(i, z2, a2);
            if (!(z2 > QP_EPS_LI * QP_EPS_LI * a2) || a2 == 0.0) continue;
            add_constraint(i, st);
        }
        stationarity_gradient();
        return recompute_R() ? 1 : 0;
    }
    // handle_error's infeasible branch (src/qpOASESInterface.cpp:716-729, 690-701): init with the primal guess
    // x0 = [0; max(0, lbA); -min(0, ubA)] (the slack-feasible point of the l1-penalty QP), y = 0; working set read off x0 and
    // A x0 with boundTolerance = 1e6*EPS.
    static __device__ QP_FN int guess_start_state() {
        QP_CTX
        double *x = V_(x), *y = V_(y), *Ax = V_(Ax), *want = V_(dy) + nV;
        const double *lbN = V_(lbN), *ubN = V_(ubN), *lbAN = V_(lbAN), *ubAN = V_(ubAN);
        short* sB = sB_;
        const double TOL = 1.0e6 * QP_EPS;
        const int o1 = nV - 2 * nC, o2 = nV - nC;
        QP_U1 for (int i = lane; i < nV; i += TEAM) { x[i] = 0.0; y[i] = 0.0; }
        SYNC();
        QP_U1 for (int i = lane; i < nC; i += TEAM) { x[o1 + i] = fmax(0.0, lbAN[i]); x[o2 + i] = -fmin(0.0, ubAN[i]); y[nV + i] = 0.0; }
        SYNC();
        mulA(x, Ax);
        QP_U1 for (int i = lane; i < nV; i += TEAM) { const double xi = x[i]; sB[i] = (short)((xi <= lbN[i] + TOL) ? -1 : ((xi >= ubN[i] - TOL) ? 1 : 0)); }
        QP_U1 for (int i = lane; i < nC; i += TEAM) { const double ax = Ax[i]; want[i] = (ax <= lbAN[i] + TOL) ? -1.0 : ((ax >= ubAN[i] - TOL) ? 1.0 : 0.0); }
        SYNC();
        return aux_qp_from_guess();
    }
    // The matrix-status flip (src/qpOASESInterface.cpp:202-207): init(H, g, A, ..., x_qp, y_qp, &bounds) -- primal and dual guess
    // = the previous solution, bound statuses = the previous ones, constraint statuses from the sign of the guessed multipliers
    // (y > EPS lower, y < -EPS upper: qpOASES obtainAuxiliaryWorkingSet with yOpt and without guessedConstraints), new matrices.
    static __device__ QP_FN int reinit_start_state() {
        QP_CTX
        double *x = V_(x), *y = V_(y), *Ax = V_(Ax), *want = V_(dy) + nV;
        QP_U1 for (int i = lane; i < nC; i += TEAM) { const double yi = y[nV + i]; want[i] = (yi > QP_EPS) ? -1.0 : ((yi < -QP_EPS) ? 1.0 : 0.0); }
        SYNC();
        mulA(x, Ax);
        return aux_qp_from_guess();
    }
    // qpOASESInterface::handle_error (src/qpOASESInterface.cpp:686-758), called when a solve did not end OPTIMAL -- after an init
    // as well as after a hot start (:160-162, :217-219).  `cold`: the failed attempt was an init.  Infeasible: re-init from the
    // slack-feasible guess.  Otherwise plain re-init; after a failed init that repeats the same deterministic solve, so only its
    // iteration count is added again (the reference adds nWSR of both runs to Stats::qp_iter, :752-753).
    static __device__ __forceinline__ int handle_error(int status, bool cold, int max_iter, int last_iters, int& total_iters) {
        QP_CTX
        int iters = 0;
        if ((status == ST_INFEASIBLE || (sA.flags & FLAG_FORCE_GUESS)) && nV >= 2 * nC) {
            const int e = guess_start_state();
            if (e == 2) return ST_CAPACITY;
            if (e == 1) return ST_INTERNAL;
            status = homotopy(max_iter, iters);
            total_iters += iters;
        } else if (!cold) {
            cold_start_state();
            status = homotopy(max_iter, iters);
            total_iters += iters;
        } else total_iters += last_iters;
        return status;
    }

    // ---------------------------------------------------------------- epilogue: objective + test_optimality
    static __device__ QP_FN void epilogue(int b, int status, int total_iters) {
        QP_CTX
        const int nT = nV + nC;
        // A x of the KKT test goes to the dead dAx buffer: the solver's own Ax (advanced incrementally by the homotopy) is part
        // of the hot-start state and must stay what the oracle keeps, or a later hotstart(g, lb, ub, lbA, ubA) starts its
        // ratio tests from a value that differs in the last bits
        double *x = V_(x), *y = V_(y), *Ax = V_(dAx), *t1 = V_(t1), *t2 = V_(t2);
        const double *gN = V_(gN), *lbN = V_(lbN), *ubN = V_(ubN), *lbAN = V_(lbAN), *ubAN = V_(ubAN);
        const short *sB = sB_, *sC = sC_;
        double* xo = sA.x + (size_t)b * nV;
        double* yo = sA.y + (size_t)b * nT;
        QP_U1 for (int i = lane; i < nV; i += TEAM) xo[i] = x[i];
        QP_U1 for (int i = lane; i < nT; i += TEAM) yo[i] = y[i];
        if (sA.wsB) for (int i = lane; i < nV; i += TEAM) sA.wsB[(size_t)b * nV + i] = (signed char)sB[i];
        if (sA.wsC) for (int i = lane; i < nC; i += TEAM) sA.wsC[(size_t)b * nC + i] = (signed char)sC[i];
        // Hx (unregularised) in t1, A x in Ax, A'y_c in t2
        mulH_noreg(x, t1);
        mulA(x, Ax);
        mulAT(y + nV, t2);
        if (lane == 0) {
            const double SQRT_M_EPS = 1.0e-8;
            double obj = 0.0;
            QP_U1 for (int i = 0; i < nV; i++) obj += 0.5 * x[i] * t1[i];
            QP_U1 for (int i = 0; i < nV; i++) obj += gN[i] * x[i];
            // getObjVal() of a problem that is not solved is INFTY (qpOASES QProblemB::getObjVal; the reference passes it on,
            // src/qpOASESInterface.cpp:324-327)
            sA.obj[b] = (status == ST_OPTIMAL) ? obj : QP_INFTY; sA.status[b] = status; sA.iters[b] = total_iters;
            // qpOASESInterface::get_working_set + test_optimality (src/qpOASESInterface.cpp:835-895, 498-684),
            // evaluated against the target data the caller supplied.
            double primal = 0.0, dual = 0.0, compl_ = 0.0, stat = 0.0;
            int* WB = sA.WB ? sA.WB + (size_t)b * nV : nullptr;
            int* WC = sA.WC ? sA.WC + (size_t)b * nC : nullptr;
            QP_U1 for (int i = 0; i < nV; i++) {
                double xi = x[i];
                primal += fmax(0.0, lbN[i] - xi);
                primal += -fmin(0.0, ubN[i] - xi);
            }
            QP_U1 for (int i = 0; i < nC; i++) {
                double ax = Ax[i];
                primal += fmax(0.0, lbAN[i] - ax);
                primal += -fmin(0.0, ubAN[i] - ax);
            }
            QP_U1 for (int i = 0; i < nV; i++) {
                int s = sB[i], W; double xi = x[i], yi = y[i];
                if (s > 0) W = (fabs(xi - lbN[i]) < SQRT_M_EPS) ? -99 : 1;
                else if (s < 0) W = (fabs(xi - ubN[i]) < SQRT_M_EPS) ? -99 : -1;
                else W = 0;
                if (WB) WB[i] = W;
                if (W == 0) dual += fabs(yi); else if (W == -1) dual += -fmin(0.0, yi); else if (W == 1) dual += fmax(0.0, yi);
            }
            QP_U1 for (int i = 0; i < nC; i++) {
                int s = sC[i], W; double ax = Ax[i], yi = y[nV + i];
                if (s > 0) W = (ax - lbAN[i] < SQRT_M_EPS) ? -99 : 1;       // :874 (comparison inside fabs)
                else if (s < 0) W = (ax - ubAN[i] < SQRT_M_EPS) ? -99 : -1;  // :880
                else W = 0;
                if (WC) WC[i] = W;
                if (W == 0) dual += fabs(yi); else if (W == -1) dual += -fmin(0.0, yi); else if (W == 1) dual += fmax(0.0, yi);
            }
            QP_U1 for (int i = 0; i < nV; i++) {
                double gap = t2[i];
                gap += y[i]; gap -= gN[i]; gap -= t1[i];
                stat += fabs(gap);
            }
            QP_U1 for (int i = 0; i < nV; i++) {
                int s = sB[i]; double xi = x[i], yi = y[i];
                int W = (s > 0) ? ((fabs(xi - lbN[i]) < SQRT_M_EPS) ? -99 : 1) : (s < 0 ? ((fabs(xi - ubN[i]) < SQRT_M_EPS) ? -99 : -1) : 0);
                if (W == 0) compl_ += fabs(yi); else if (W == -1) compl_ += fabs(yi * (xi - lbN[i])); else if (W == 1) compl_ += fabs(yi * (ubN[i] - xi));
            }
            QP_U1 for (int i = 0; i < nC; i++) {
                int s = sC[i]; double ax = Ax[i], yi = y[nV + i];
                int W = (s > 0) ? ((ax - lbAN[i] < SQRT_M_EPS) ? -99 : 1) : (s < 0 ? ((ax - ubAN[i] < SQRT_M_EPS) ? -99 : -1) : 0);
                if (W == 0) compl_ += fabs(yi); else if (W == -1) compl_ += fabs(yi * (ax - lbAN[i])); else if (W == 1) compl_ += fabs(yi * (ubAN[i] - ax));
            }
            if (sA.kkt) {
                double* k = sA.kkt + (size_t)b * 5;
                k[0] = primal; k[1] = dual; k[2] = stat; k[3] = compl_; k[4] = compl_ + stat + dual + primal;
            }
            hdr[3] = (status == ST_OPTIMAL) ? 1 : 0;
            if (sA.maxfr) atomicMax(sA.maxfr, hdr[6]);  // the handle learns the factor capacity its QPs need
        }
        SYNC();
    }
};

// Per-instance init / hotstart decision (src/qpOASESInterface.cpp:141-211 with get_Matrix_change_status :817-833), for batched
// drivers that keep the reference's semantics instance by instance: st = {first_solved, varied (Update_A || Update_H since the
// instance's last solve), old matrix status, new matrix status, mode chosen by the last launch}; matrix status -1 undefined,
// 0 fixed, 1 varied.  Every thread of the team computes the same mode; one thread stores the new state after a team barrier.
// The rescue launch re-uses the mode the main launch chose.
__device__ __forceinline__ int qp_instance_mode(const signed char* st, bool rescue, int& old_ms, int& new_ms) {
    old_ms = st[2]; new_ms = st[3];
    if (rescue) return st[4];
    const int first = st[0], varied = st[1] != 0;
    int mode = MODE_COLD;
    if (first) {
        if (old_ms < 0) old_ms = varied ? 1 : 0;
        else { if (new_ms >= 0) old_ms = new_ms; new_ms = varied ? 1 : 0; }
        if (new_ms < 0) mode = (old_ms == 0) ? MODE_HOT_FIXED : MODE_HOT_VARIED;
        else if (new_ms == 0 && old_ms == 0) mode = MODE_HOT_FIXED;
        else if (new_ms == 1 && old_ms == 1) mode = MODE_HOT_VARIED;
        else { mode = MODE_REINIT; new_ms = old_ms = -1; }  // status flip: init from the previous solution (:202-207)
    }
    return mode;
}
__device__ __forceinline__ void qp_instance_store(signed char* st, int mode, int old_ms, int new_ms) {
    st[0] = 1; st[1] = 0; st[2] = (signed char)old_ms; st[3] = (signed char)new_ms; st[4] = (signed char)mode;
}

// -------------------------------------------------------------------------------------------
// kernel: one QP per warp, CTA_THREADS/32 QPs per CTA
// -------------------------------------------------------------------------------------------
// WPS = warps per SM the register allocation is capped for: 16 (<= 128 registers; measured: 20 or 24 warps lose everywhere) or
// 32 (<= 64 registers, a few spills): 15-20 % faster on QPs small enough that shared memory lets 32 warps be resident
// (nV <~ 20), slower on the larger ones where shared memory caps the occupancy anyway -- capi.cu picks per problem size.
template <int TEAM> static __device__ __forceinline__ void qp_solve_one(const QPKernelArgs& A, const int b, const int team_id, const int lane);
template <int CTA_THREADS, int WPS, int TEAM = 32>
__global__ void __launch_bounds__(CTA_THREADS, (WPS * 32) / CTA_THREADS) qp_solve_kernel(const __grid_constant__ QPKernelArgs A) {
    constexpr int TEAMS = CTA_THREADS / TEAM;
    // stage the launch arguments and the 16-bit pattern once per CTA
    {
        const int* src = reinterpret_cast<const int*>(&A);
        int* dst = reinterpret_cast<int*>(&sA);
        for (int i = threadIdx.x; i < (int)(sizeof(QPKernelArgs) / 4); i += CTA_THREADS) dst[i] = src[i];
        short* pat = reinterpret_cast<short*>(qp_smem + (size_t)TEAMS * A.slice_doubles);
        const bool has_H = A.has_H && !A.is_lp;
        for (int i = threadIdx.x; i <= A.nV; i += CTA_THREADS) { pat[A.pAp + i] = (short)A.Ap[i]; if (has_H) pat[A.pHp + i] = (short)A.Hp[i]; }
        for (int i = threadIdx.x; i <= A.nC; i += CTA_THREADS) pat[A.pArp + i] = (short)A.Arp[i];
        for (int i = threadIdx.x; i < A.zA; i += CTA_THREADS) { pat[A.pAi + i] = (short)A.Ai[i]; pat[A.pAci + i] = (short)A.Aci[i]; pat[A.pAperm + i] = (short)A.Aperm[i]; }
        if (has_H) for (int i = threadIdx.x; i < A.zH; i += CTA_THREADS) pat[A.pHi + i] = (short)A.Hi[i];
    }
    __syncthreads();

    const int team_id = threadIdx.x / TEAM;
    const int lane = threadIdx.x & (TEAM - 1);
    if (A.rescue) {
        // rescue launch (small fixed grid): the instances the main launch listed as overflowing its factor capacity, re-solved
        // from their pre-solve state with full-size factors.  Usually the list is empty and every warp leaves at once.
        const int count = *A.ncap;
        for (int k = blockIdx.x * TEAMS + team_id; k < count; k += gridDim.x * TEAMS) { qp_solve_one<TEAM>(A, A.caplist[k], team_id, lane); __syncwarp(team_mask<TEAM>()); }
        return;
    }
    const int b = blockIdx.x * TEAMS + team_id;
    if (b >= A.batch) return;
    if (A.mask && !A.mask[b]) return;
    qp_solve_one<TEAM>(A, b, team_id, lane);
}

// one QP on the calling team of TEAM <= 32 lanes (slice `team_id` of the CTA's shared memory)
template <int TEAM> static __device__ __forceinline__ void qp_solve_one(const QPKernelArgs& A, const int b, const int team_id, const int lane) {
    const int nV = A.nV, nC = A.nC, cap = A.cap, ld = A.ld;
    double* slice = qp_smem + (size_t)team_id * A.slice_doubles;
    int* hdr = reinterpret_cast<int*>(slice);
    double *Q = slice + A.oQ, *RT = slice + A.oRT;

    int mode = A.mode;
    if (A.inst_state) {
        int oms, nms;
        mode = qp_instance_mode(A.inst_state + 8 * (size_t)b, A.rescue != 0, oms, nms);
        __syncwarp(team_mask<TEAM>());  // every lane has read the state
        if (lane == 0 && !A.rescue) qp_instance_store(A.inst_state + 8 * (size_t)b, mode, oms, nms);
    }
    int status = 0;
    if (mode != MODE_COLD) {
        // restore the pre-solve image: everything but the factors verbatim, then Q (nFR x nFR), R (nZ x nZ), T (nAC x nFR)
        const double* st = A.state + (size_t)b * A.state_doubles;
        for (int i = lane; i < A.oP; i += TEAM) slice[i] = st[i];
        __syncwarp(team_mask<TEAM>());
        const int nFR = hdr[0], nAC = hdr[1], nZ = nFR - nAC;
        if (!hdr[3]) mode = MODE_COLD;  // previous solve did not end optimal: plain re-init (handle_error)
        else if (nFR > cap) status = ST_CAPACITY;
        else {
            const double *Qp = st + A.oP, *Rp = Qp + nFR * nFR, *Tp = Rp + nZ * nZ;
            for (int k = lane; k < nFR * nFR; k += TEAM) Q[(k / nFR) * ld + (k % nFR)] = Qp[k];
            for (int k = lane; k < nZ * nZ; k += TEAM) R_(k / nZ, k % nZ) = Rp[k];
            for (int k = lane; k < nAC * nFR; k += TEAM) T_(k / nFR, k % nFR) = Tp[k];
        }
        __syncwarp(team_mask<TEAM>());
    }
    if (mode != MODE_HOT_FIXED) {
        const double* av = A.Aval + (size_t)b * A.zA;
        for (int i = lane; i < A.zA; i += TEAM) slice[A.oAv + i] = av[i];
        if (A.has_H && !A.is_lp) {
            const double* hv = A.Hval + (size_t)b * A.zH;
            for (int i = lane; i < A.zH; i += TEAM) slice[A.oHv + i] = hv[i];
        }
    }
    {  // target data of the homotopy
        const double *gN = A.gN + (size_t)b * nV, *lbN = A.lbN + (size_t)b * nV, *ubN = A.ubN + (size_t)b * nV;
        const double *lbAN = A.lbAN + (size_t)b * nC, *ubAN = A.ubAN + (size_t)b * nC;
        // |v| > 1e20 is clamped to qpOASES's infinity, as the oracle does
        for (int i = lane; i < nV; i += TEAM) {
            slice[A.ogN + i] = gN[i];
            slice[A.olbN + i] = fmin(fmax(lbN[i], -QP_INFTY), QP_INFTY);
            slice[A.oubN + i] = fmin(fmax(ubN[i], -QP_INFTY), QP_INFTY);
        }
        for (int i = lane; i < nC; i += TEAM) {
            slice[A.olbAN + i] = fmin(fmax(lbAN[i], -QP_INFTY), QP_INFTY);
            slice[A.oubAN + i] = fmin(fmax(ubAN[i], -QP_INFTY), QP_INFTY);
        }
    }
    __syncwarp(team_mask<TEAM>());

    int iters = 0, total_iters = 0;
    PROF_T0
    if (status != ST_CAPACITY) {
        bool fell_back = false;  // the kept working set could not be refactorised: the cold start below is the recovery attempt
        if (mode == MODE_HOT_VARIED) {
            if (QPT<TEAM>::refactorise()) { mode = MODE_COLD; fell_back = true; }  // projected Hessian of the kept set not PD
            else QPT<TEAM>::drift_correction();
        } else if (mode == MODE_REINIT) {
            const int e = QPT<TEAM>::reinit_start_state();
            if (e == 2) status = ST_CAPACITY;
            else if (e) { mode = MODE_COLD; fell_back = true; }  // that init fails before its homotopy: plain re-init
        }
        if (status != ST_CAPACITY) {
            if (mode == MODE_COLD) QPT<TEAM>::cold_start_state();
            status = QPT<TEAM>::homotopy(A.max_iter, iters);
            total_iters += iters;
            if (status != ST_CAPACITY && ((status != ST_OPTIMAL && !fell_back) || (A.flags & FLAG_FORCE_GUESS)))
                status = QPT<TEAM>::handle_error(status, mode == MODE_COLD, A.max_iter, iters, total_iters);
        }
    }
    if (status == ST_CAPACITY) {  // left to the rescue launch (full capacity), which restarts from the pre-solve state
        if (lane == 0) { A.status[b] = ST_CAPACITY; A.iters[b] = 0; if (A.ncap) A.caplist[atomicAdd(A.ncap, 1)] = b; }
        return;
    }
    PROF_ADD(PR_TOTAL);
    QPT<TEAM>::epilogue(b, status, total_iters);
    PROF_ADD(PR_EPILOGUE);
    if ((A.flags & FLAG_KEEP_STATE) && A.state) {
        double* st = A.state + (size_t)b * A.state_doubles;
        for (int i = lane; i < A.oP; i += TEAM) st[i] = slice[i];
        const int nFR = hdr[0], nAC = hdr[1], nZ = nFR - nAC;
        double *Qp = st + A.oP, *Rp = Qp + nFR * nFR, *Tp = Rp + nZ * nZ;
        for (int k = lane; k < nFR * nFR; k += TEAM) Qp[k] = Q[(k / nFR) * ld + (k % nFR)];
        for (int k = lane; k < nZ * nZ; k += TEAM) Rp[k] = R_(k / nZ, k % nZ);
        for (int k = lane; k < nAC * nFR; k += TEAM) Tp[k] = T_(k / nFR, k % nFR);
    }
}

// -------------------------------------------------------------------------------------------
// kernel: one QP per CTA (large QPs: factors do not fit in shared memory)
// -------------------------------------------------------------------------------------------
// The slice of instance b (vectors, index lists and the nV x nV factors Q, R/T) lives in global memory at
// gwork[b][slice_doubles] and persists between launches, so a hot start needs no save/restore; the CTA streams it through
// L1/L2.  Same solver code as the warp kernel (QPT<TEAM>), the team barrier being __syncthreads(); the O(n^3) refactorisation
// runs as TMA-staged FP64 DMMA tiles shared by the CTAs of a thread-block cluster (see the block comment in QPT).
template <int CTA_THREADS>
__global__ void __launch_bounds__(CTA_THREADS, 1) qp_solve_large_kernel(const __grid_constant__ QPKernelArgs A) {
    typedef QPT<CTA_THREADS> S;
    const int tid = threadIdx.x;
    unsigned cs = 1, rank = 0;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(cs));
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    const int b = blockIdx.x / cs;  // the CTAs of a cluster share one QP: rank 0 solves, the others help with refactorisations
    {
        const int* src = reinterpret_cast<const int*>(&A);
        int* dst = reinterpret_cast<int*>(&sA);
        for (int i = tid; i < (int)(sizeof(QPKernelArgs) / 4); i += CTA_THREADS) dst[i] = src[i];
        if (tid == 0) {
            sSlice = A.gwork + (size_t)b * A.slice_doubles;
            sClusterSize = (int)cs;
            sPhase = 0u;
            for (int s = 0; s < 3; s++) mbar_init(&sFull[s], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
    }
    __syncthreads();
    if (tid == 0 && rank != 0) sA.prof = nullptr;  // phase timers: the leader's clock only
    if (A.mask && !A.mask[b]) return;  // uniform over the cluster
    const int nV = A.nV, nC = A.nC;
    double* slice = A.gwork + (size_t)b * A.slice_doubles;
    int* hdr = reinterpret_cast<int*>(slice);
    if (rank != 0) { S::helper_loop((int)rank, (int)cs); return; }

    int mode = A.mode;
    if (A.inst_state) {
        int oms, nms;
        mode = qp_instance_mode(A.inst_state + 8 * (size_t)b, false, oms, nms);
        __syncthreads();  // every thread of the CTA has read the state
        if (tid == 0) qp_instance_store(A.inst_state + 8 * (size_t)b, mode, oms, nms);
    }
    if (mode != MODE_COLD && !hdr[3]) mode = MODE_COLD;  // previous solve did not end optimal: plain re-init (handle_error)
    __syncthreads();
    if (mode != MODE_HOT_FIXED) {
        const double* av = A.Aval + (size_t)b * A.zA;
        for (int i = tid; i < A.zA; i += CTA_THREADS) slice[A.oAv + i] = av[i];
        if (A.has_H && !A.is_lp) {
            const double* hv = A.Hval + (size_t)b * A.zH;
            for (int i = tid; i < A.zH; i += CTA_THREADS) slice[A.oHv + i] = hv[i];
        }
    }
    {
        const double *gN = A.gN + (size_t)b * nV, *lbN = A.lbN + (size_t)b * nV, *ubN = A.ubN + (size_t)b * nV;
        const double *lbAN = A.lbAN + (size_t)b * nC, *ubAN = A.ubAN + (size_t)b * nC;
        for (int i = tid; i < nV; i += CTA_THREADS) {
            slice[A.ogN + i] = gN[i];
            slice[A.olbN + i] = fmin(fmax(lbN[i], -QP_INFTY), QP_INFTY);
            slice[A.oubN + i] = fmin(fmax(ubN[i], -QP_INFTY), QP_INFTY);
        }
        for (int i = tid; i < nC; i += CTA_THREADS) {
            slice[A.olbAN + i] = fmin(fmax(lbAN[i], -QP_INFTY), QP_INFTY);
            slice[A.oubAN + i] = fmin(fmax(ubAN[i], -QP_INFTY), QP_INFTY);
        }
    }
    __syncthreads();

    int iters = 0, total_iters = 0, status;
    const int lane = tid;
    PROF_T0
    bool fell_back = false;
    if (mode == MODE_HOT_VARIED) {
        if (S::refactorise()) { mode = MODE_COLD; fell_back = true; }
        else S::drift_correction();
    } else if (mode == MODE_REINIT) {
        if (S::reinit_start_state()) { mode = MODE_COLD; fell_back = true; }
    }
    if (mode == MODE_COLD) S::cold_start_state();
    status = S::homotopy(A.max_iter, iters);
    total_iters += iters;
    if ((status != ST_OPTIMAL && !fell_back) || (A.flags & FLAG_FORCE_GUESS))
        status = S::handle_error(status, mode == MODE_COLD, A.max_iter, iters, total_iters);
    PROF_ADD(PR_TOTAL);
    S::epilogue(b, status, total_iters);
    PROF_ADD(PR_EPILOGUE);
    if (tid == 0) hdr[4] = S::OP_EXIT;
    __syncthreads();
    S::large_sync();
}

#endif  // __CUDACC__

}  // namespace sqpb200
