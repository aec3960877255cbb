// capi.cu -- the C ABI of libsqpb200.so (include/sqpb200.h): handle management, host<->device
// plumbing and kernel launches.  No CPU compute path exists in this library: every numerical
// entry point launches the sm_100a kernels of qp_kernel.cuh / l0_kernels.cuh.
#include "../../include/sqpb200.h"
#include "l0_kernels.cuh"
#include "qp_kernel.cuh"

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <string>
#include <vector>

using namespace sqpb200;

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            char buf_[512];                                                                        \
            snprintf(buf_, sizeof buf_, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            h->err = buf_;                                                                         \
            return SQPB200_ERR_CUDA;                                                               \
        }                                                                                          \
    } while (0)

enum { MS_UNDEFINED = -1, MS_FIXED = 0, MS_VARIED = 1 };

struct SolveCfg { int cap = 0, teams = 0, smem = 0, slice_doubles = 0, state_doubles = 0, resident = 0, lanes = 32; };

struct sqpb200_handle_s {
    int batch = 0, nV = 0, nC = 0, qptype = SQPB200_QP, device = 0;
    sqpb200_options opt;
    cudaStream_t stream = nullptr;
    std::string err;
    // structure
    bool A_set = false, H_set = false;
    int zA = 0, zJ = 0, zH = 0, zHt = 0;  // zH: CSC entries of H; zHt: triplet count
    std::vector<int> Ap, Ai, Aorder, Asrc, Hp, Hi, Horder, Hsrc;
    std::vector<double> A_init;
    int *dAp = nullptr, *dAi = nullptr, *dArp = nullptr, *dAci = nullptr, *dAperm = nullptr, *dAsrc = nullptr;
    int *dHp = nullptr, *dHi = nullptr, *dHsrc = nullptr;
    // QORE layout (compressed-row view given by the caller, sqpb200_set_structure_*_csr): row pointers, column indices, triplet ->
    // storage position, and the position maps between the two storage orders (q2c[compressed-row position] = compressed-column
    // position, c2q its inverse), resident for the device-side value moves
    struct CsrView { bool set = false; std::vector<int> rp, ci, order, q2c, c2q; int *dq2c = nullptr, *dc2q = nullptr; } qA, qH;
    void* qscratch = nullptr;  // [batch][nC] doubles (A x) + [batch][nV+nC] int32 (working set) of sqpb200_get_solution_stacked
    size_t qscratch_bytes = 0;
    // data
    double *dAval = nullptr, *dHval = nullptr;
    double *dg = nullptr, *dlb = nullptr, *dub = nullptr, *dlbA = nullptr, *dubA = nullptr;
    // results
    double *dx = nullptr, *dy = nullptr, *dobj = nullptr, *dkkt = nullptr;
    int *dstatus = nullptr, *diters = nullptr, *dWB = nullptr, *dWC = nullptr;
    signed char *dwsB = nullptr, *dwsC = nullptr;
    unsigned char* dmask = nullptr;
    void* arena = nullptr;  // one allocation behind dg .. dmask
    size_t in_off[5] = {0, 0, 0, 0, 0}, in_bytes = 0, out_base = 0, out_off[6] = {0, 0, 0, 0, 0, 0}, out_bytes = 0;  // sqpb200_io_layout
    // hot-start state
    double* dstate = nullptr;
    int slice_doubles = 0, ld = 0;
    // change flags (src/qpOASESInterface.cpp:361-496, 817-833)
    bool first_solved = false, upd_A = false, upd_H = false, upd_g = false, upd_bounds = false;
    int old_ms = MS_UNDEFINED, new_ms = MS_UNDEFINED;
    // staging + stats
    void* stage = nullptr;
    size_t stage_bytes = 0;
    long long launches = 0;
    // learned factor capacity: the solve kernels keep a running maximum of the free variables any instance needed (device
    // int, read back asynchronously after every solve); later solves size the shared-memory factors by it
    int* dmaxfr = nullptr;
    int* dncap = nullptr;       // [1 + batch]: count and list of the instances the main launch hands to the rescue launch
    int* maxfr_host = nullptr;  // pinned
    cudaEvent_t ev_maxfr = nullptr;
    bool maxfr_pending = false, maxfr_valid = false;
    int maxfr_seen = 0, cfg_cap_key = -1;
    long long* dprof = nullptr;  // [16] phase cycle counters (written by -DQP_PROFILE builds of the solve kernels only)
    float last_ms = 0.f;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    int team = 0, teams_per_cta = 0, smem_cta = 0;
    SolveCfg cfg_main, cfg_rescue;
    bool have_rescue = false;
    // one-QP-per-CTA path (QPs whose slice does not fit in shared memory): slices and 32-bit pattern in global memory
    bool large = false;
    int* dgpat = nullptr;
    double* dgwork = nullptr;
    int large_slice_doubles = 0;
};

static int grid_for(long long total, int block) {
    long long g = (total + block - 1) / block;
    long long cap = 148LL * 16;  // 148 SMs x resident CTAs; grid-stride loops cover the rest
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

template <typename T>
static int dev_alloc(sqpb200_handle h, T** p, size_t n) {
    if (n == 0) n = 1;
    CK(cudaMalloc((void**)p, n * sizeof(T)));
    CK(cudaMemsetAsync(*p, 0, n * sizeof(T), h->stream));
    return 0;
}

static int ensure_stage(sqpb200_handle h, size_t bytes) {
    if (bytes <= h->stage_bytes) return 0;
    if (h->stage) { CK(cudaStreamSynchronize(h->stream)); CK(cudaFree(h->stage)); h->stage = nullptr; h->stage_bytes = 0; }
    CK(cudaMalloc(&h->stage, bytes));
    h->stage_bytes = bytes;
    return 0;
}

// returns a device pointer for `src` (copying through the staging buffer when it is host memory)
static int to_device(sqpb200_handle h, const void* src, size_t bytes, int loc, size_t stage_off, const void** out) {
    if (loc == SQPB200_LOC_DEVICE) { *out = src; return 0; }
    CK(cudaMemcpyAsync((char*)h->stage + stage_off, src, bytes, cudaMemcpyHostToDevice, h->stream));
    *out = (char*)h->stage + stage_off;
    return 0;
}

__global__ void widen_ws_kernel(long long total, const signed char* __restrict__ in, int* __restrict__ out) {
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long stride = (long long)gridDim.x * blockDim.x;
    for (; t < total; t += stride) out[t] = (int)in[t];
}

// All sqpb200_* functions below were declared extern "C" by include/sqpb200.h and keep that linkage.

void sqpb200_default_options(sqpb200_options* o) {
    o->qp_maxiter = 1000;
    o->lp_maxiter = 100;
    o->enable_flipping = 1;
    o->enable_ramping = 1;
    o->enable_drift = 1;
    o->team_size = 0;
    o->keep_state = 1;
    o->factor_cap = 0;
    o->debug_force_error_branch = 0;
    o->refactorise_every = 0;
}

const char* sqpb200_version(void) { return "sqpb200 0.1 (sm_100a)"; }

int sqpb200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return SQPB200_ERR_CUDA;
    return n;
}

const char* sqpb200_last_error(sqpb200_handle h) { return h ? h->err.c_str() : "null handle"; }

int sqpb200_create(int batch, int nV, int nC, int qptype, int device, const sqpb200_options* opts,
                   sqpb200_handle* out) {
    if (!out || batch <= 0 || nV <= 0 || nC < 0 || (qptype != SQPB200_QP && qptype != SQPB200_LP)) return SQPB200_ERR_INVALID;
    if (nV >= (1 << 15) || nC >= (1 << 15)) return SQPB200_ERR_TOO_LARGE;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return SQPB200_ERR_CUDA;  // no CPU fallback
    if (device < 0 || device >= ndev) return SQPB200_ERR_INVALID;
    sqpb200_handle h = new sqpb200_handle_s();
    h->batch = batch; h->nV = nV; h->nC = nC; h->qptype = qptype; h->device = device;
    if (opts) h->opt = *opts; else sqpb200_default_options(&h->opt);
    if (cudaSetDevice(device) != cudaSuccess) { delete h; return SQPB200_ERR_CUDA; }
    h->ld = (nV % 2 == 0) ? nV + 1 : nV;  // odd leading dimension: conflict-free row and column walks
    size_t B = (size_t)batch;
    int rc = 0;
    {
        // the 17 per-instance vectors and result arrays come out of ONE allocation (one cudaMalloc + one memset instead of 17:
        // handle creation is on the critical path of short batched SQP runs); every sub-array starts 256-byte aligned
        size_t off = 0;
        auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
        const size_t o_g = take(B * nV * 8), o_lb = take(B * nV * 8), o_ub = take(B * nV * 8), o_lbA = take(B * nC * 8), o_ubA = take(B * nC * 8);
        const size_t o_x = take(B * nV * 8), o_y = take(B * (nV + nC) * 8), o_obj = take(B * 8), o_kkt = take(B * 5 * 8);
        const size_t o_st = take(B * 4), o_it = take(B * 4), o_WB = take(B * nV * 4), o_WC = take(B * nC * 4);
        const size_t o_wsB = take(B * nV + 32), o_wsC = take(B * nC + 32);  // +32: kkt_tma_kernel reads 16-byte windows
        const size_t o_mask = take(B);
        if (cudaMalloc(&h->arena, off) != cudaSuccess) { h->arena = nullptr; rc = 1; }
        else {
            if (cudaMemsetAsync(h->arena, 0, off, h->stream) != cudaSuccess) rc = 1;
            char* a = (char*)h->arena;
            // the vectors (g .. ubA) and the results (x .. iters) are two contiguous blocks: one copy each way per solve
            h->in_off[0] = o_g; h->in_off[1] = o_lb; h->in_off[2] = o_ub; h->in_off[3] = o_lbA; h->in_off[4] = o_ubA; h->in_bytes = o_x;
            h->out_base = o_x;
            h->out_off[0] = 0; h->out_off[1] = o_y - o_x; h->out_off[2] = o_obj - o_x; h->out_off[3] = o_kkt - o_x; h->out_off[4] = o_st - o_x;
            h->out_off[5] = o_it - o_x; h->out_bytes = o_WB - o_x;
            h->dg = (double*)(a + o_g); h->dlb = (double*)(a + o_lb); h->dub = (double*)(a + o_ub); h->dlbA = (double*)(a + o_lbA); h->dubA = (double*)(a + o_ubA);
            h->dx = (double*)(a + o_x); h->dy = (double*)(a + o_y); h->dobj = (double*)(a + o_obj); h->dkkt = (double*)(a + o_kkt);
            h->dstatus = (int*)(a + o_st); h->diters = (int*)(a + o_it); h->dWB = (int*)(a + o_WB); h->dWC = (int*)(a + o_WC);
            h->dwsB = (signed char*)(a + o_wsB); h->dwsC = (signed char*)(a + o_wsC); h->dmask = (unsigned char*)(a + o_mask);
        }
    }
    if (rc) { h->err = "allocation of the vector arena failed"; *out = h; return SQPB200_ERR_CUDA; }
    if (cudaEventCreate(&h->ev0) != cudaSuccess || cudaEventCreate(&h->ev1) != cudaSuccess) { h->err = "cudaEventCreate failed"; *out = h; return SQPB200_ERR_CUDA; }
    if (cudaMalloc((void**)&h->dmaxfr, sizeof(int)) == cudaSuccess && cudaMallocHost((void**)&h->maxfr_host, sizeof(int)) == cudaSuccess &&
        cudaEventCreateWithFlags(&h->ev_maxfr, cudaEventDisableTiming) == cudaSuccess) {
        *h->maxfr_host = 0;
        if (cudaMemset(h->dmaxfr, 0, sizeof(int)) != cudaSuccess || cudaMalloc((void**)&h->dncap, (size_t)(batch + 1) * sizeof(int)) != cudaSuccess ||
            cudaMemset(h->dncap, 0, (size_t)(batch + 1) * sizeof(int)) != cudaSuccess) { h->err = "allocation failed"; *out = h; return SQPB200_ERR_CUDA; }
    } else { h->err = "allocation of the capacity counter failed"; *out = h; return SQPB200_ERR_CUDA; }
    if (cudaMalloc((void**)&h->dprof, 16 * sizeof(long long)) == cudaSuccess) cudaMemset(h->dprof, 0, 16 * sizeof(long long));
    else h->dprof = nullptr;
    // status = NOTINITIALISED until the first solve
    std::vector<int> st(batch, SQPB200_QPERROR_NOTINITIALISED);
    if (cudaMemcpy(h->dstatus, st.data(), B * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) { h->err = "initialising the status array failed"; *out = h; return SQPB200_ERR_CUDA; }
    *out = h;
    return 0;
}

int sqpb200_destroy(sqpb200_handle h) {
    if (!h) return SQPB200_ERR_INVALID;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    void* ptrs[] = {h->dAp, h->dAi, h->dArp, h->dAci, h->dAperm, h->dAsrc, h->dHp, h->dHi, h->dHsrc, h->dAval, h->dHval,
                    h->arena, h->dstate, h->stage, h->dgpat, h->dgwork, h->dprof, h->dmaxfr, h->dncap};
    for (void* p : ptrs) if (p) cudaFree(p);
    void* qptrs[] = {h->qA.dq2c, h->qA.dc2q, h->qH.dq2c, h->qH.dc2q, h->qscratch};
    for (void* p : qptrs) if (p) cudaFree(p);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->ev_maxfr) cudaEventDestroy(h->ev_maxfr);
    if (h->maxfr_host) cudaFreeHost(h->maxfr_host);
    delete h;
    return 0;
}

int sqpb200_set_stream(sqpb200_handle h, void* s) {
    if (!h) return SQPB200_ERR_INVALID;
    if ((cudaStream_t)s == h->stream) return 0;
    // work already queued on the old stream (arena memset, uploads, an in-flight solve) is ordered before anything the new
    // stream will run: the new stream waits on an event recorded at the tail of the old one (no host synchronisation)
    CK(cudaSetDevice(h->device));
    cudaEvent_t ev;
    CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CK(cudaEventRecord(ev, h->stream));
    CK(cudaStreamWaitEvent((cudaStream_t)s, ev, 0));
    CK(cudaEventDestroy(ev));
    h->stream = (cudaStream_t)s;
    return 0;
}

int sqpb200_reset(sqpb200_handle h) {
    if (!h) return SQPB200_ERR_INVALID;
    h->first_solved = false;
    h->upd_A = h->upd_H = h->upd_g = h->upd_bounds = false;
    h->old_ms = h->new_ms = MS_UNDEFINED;
    // invalidate every instance's hot-start image (its header says "not initialised"): an instance that is first solved later
    // through a hot-start call then starts cold, exactly as on a fresh handle
    CK(cudaSetDevice(h->device));
    if (h->dstate && h->cfg_main.state_doubles > 0)
        CK(cudaMemset2DAsync(h->dstate, (size_t)h->cfg_main.state_doubles * 8, 0, 32, h->batch, h->stream));
    if (h->dgwork && h->large_slice_doubles > 0)
        CK(cudaMemset2DAsync(h->dgwork, (size_t)h->large_slice_doubles * 8, 0, 32, h->batch, h->stream));
    return 0;
}

int sqpb200_synchronize(sqpb200_handle h) {
    if (!h) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// ------------------------------------------------------------------------------ assembly
// Runs csc_assemble_kernel over nmat segments whose triplets are already on the host.
static int run_assembly(sqpb200_handle h, cudaStream_t stream, int nmat, const int* seg, const int* ncol,
                        const int* row1, const int* col1, int* colptr, int* rowidx, int* order, float* ms,
                        std::string* err) {
    (void)h;
    int ztot = seg[nmat];
    std::vector<int> cp_off(nmat + 1, 0), pad_off(nmat + 1, 0);
    for (int m = 0; m < nmat; m++) {
        int z = seg[m + 1] - seg[m];
        int P = 1;
        while (P < z) P <<= 1;
        if (z >= (1 << 21) || ncol[m] >= (1 << 21)) { *err = "matrix too large for packed keys"; return SQPB200_ERR_TOO_LARGE; }
        pad_off[m + 1] = pad_off[m] + P;
        cp_off[m + 1] = cp_off[m] + ncol[m] + 1;
    }
    // one checked allocation behind every scratch array (each sub-array 256-byte aligned), freed on every exit path
    int *dseg, *dncol, *dcpoff, *drow, *dcol, *dpad, *dcolptr, *drowidx, *dorder;
    uint64_t* dscr;
    char* pool = nullptr;
    cudaError_t e = cudaSuccess;
    {
        size_t off = 0;
        auto take = [&](size_t bytes) { size_t o = off; off += ((bytes ? bytes : 4) + 255) / 256 * 256; return o; };
        const size_t o_seg = take((size_t)(nmat + 1) * 4), o_ncol = take((size_t)nmat * 4), o_cp = take((size_t)(nmat + 1) * 4),
                     o_pad = take((size_t)(nmat + 1) * 4), o_row = take((size_t)ztot * 4), o_col = take((size_t)ztot * 4),
                     o_colptr = take((size_t)cp_off[nmat] * 4), o_rowidx = take((size_t)ztot * 4), o_order = take((size_t)ztot * 4),
                     o_scr = take((size_t)pad_off[nmat] * 8);
        e = cudaMalloc((void**)&pool, off);
        if (e != cudaSuccess) { *err = cudaGetErrorString(e); return SQPB200_ERR_NOMEM; }
        dseg = (int*)(pool + o_seg); dncol = (int*)(pool + o_ncol); dcpoff = (int*)(pool + o_cp); dpad = (int*)(pool + o_pad);
        drow = (int*)(pool + o_row); dcol = (int*)(pool + o_col); dcolptr = (int*)(pool + o_colptr); drowidx = (int*)(pool + o_rowidx);
        dorder = (int*)(pool + o_order); dscr = (uint64_t*)(pool + o_scr);
    }
    cudaMemcpyAsync(dseg, seg, (nmat + 1) * 4, cudaMemcpyHostToDevice, stream);
    cudaMemcpyAsync(dncol, ncol, nmat * 4, cudaMemcpyHostToDevice, stream);
    cudaMemcpyAsync(dcpoff, cp_off.data(), (nmat + 1) * 4, cudaMemcpyHostToDevice, stream);
    cudaMemcpyAsync(dpad, pad_off.data(), (nmat + 1) * 4, cudaMemcpyHostToDevice, stream);
    cudaMemcpyAsync(drow, row1, (size_t)ztot * 4, cudaMemcpyHostToDevice, stream);
    cudaMemcpyAsync(dcol, col1, (size_t)ztot * 4, cudaMemcpyHostToDevice, stream);
    {
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0); cudaEventCreate(&e1);
        cudaEventRecord(e0, stream);
        int Pmax = 1;
        for (int m = 0; m < nmat; m++) Pmax = std::max(Pmax, pad_off[m + 1] - pad_off[m]);
        if (Pmax <= 256 && nmat >= 8) {  // many small matrices: one warp each, keys in registers (shuffle network)
            const int grid = (nmat + 7) / 8;
            if (Pmax <= 32) csc_assemble_reg_kernel<1><<<grid, 256, 0, stream>>>(nmat, dseg, dncol, dcpoff, drow, dcol, dcolptr, drowidx, dorder);
            else if (Pmax <= 64) csc_assemble_reg_kernel<2><<<grid, 256, 0, stream>>>(nmat, dseg, dncol, dcpoff, drow, dcol, dcolptr, drowidx, dorder);
            else if (Pmax <= 128) csc_assemble_reg_kernel<4><<<grid, 256, 0, stream>>>(nmat, dseg, dncol, dcpoff, drow, dcol, dcolptr, drowidx, dorder);
            else csc_assemble_reg_kernel<8><<<grid, 256, 0, stream>>>(nmat, dseg, dncol, dcpoff, drow, dcol, dcolptr, drowidx, dorder);
        } else if (Pmax <= ASM_WARP_KEYS && nmat >= 8)  // up to 512 keys: the network in the warp's shared-memory slice
            csc_assemble_warp_kernel<<<(nmat + 7) / 8, 256, (size_t)8 * Pmax * 8, stream>>>(nmat, Pmax, dseg, dncol, dcpoff, drow, dcol, dpad, dcolptr, drowidx, dorder);
        else
            csc_assemble_kernel<<<nmat, 256, 0, stream>>>(nmat, dseg, dncol, dcpoff, drow, dcol, dpad, dscr, dcolptr, drowidx, dorder);
        cudaEventRecord(e1, stream);
        cudaMemcpyAsync(colptr, dcolptr, (size_t)cp_off[nmat] * 4, cudaMemcpyDeviceToHost, stream);
        cudaMemcpyAsync(rowidx, drowidx, (size_t)ztot * 4, cudaMemcpyDeviceToHost, stream);
        cudaMemcpyAsync(order, dorder, (size_t)ztot * 4, cudaMemcpyDeviceToHost, stream);
        e = cudaStreamSynchronize(stream);
        float t = 0.f;
        cudaEventElapsedTime(&t, e0, e1);
        if (ms) *ms = t;
        cudaEventDestroy(e0); cudaEventDestroy(e1);
    }
    cudaFree(pool);
    if (e != cudaSuccess) { *err = cudaGetErrorString(e); return SQPB200_ERR_CUDA; }
    return 0;
}

int sqpb200_assemble_csc_batched(int device, int nmat, const int* seg, const int* ncol, const int* row1,
                                 const int* col1, int* colptr, int* rowidx, int* order, float* kernel_ms) {
    if (nmat <= 0 || !seg || !ncol) return SQPB200_ERR_INVALID;
    if (cudaSetDevice(device) != cudaSuccess) return SQPB200_ERR_CUDA;
    std::string err;
    return run_assembly(nullptr, nullptr, nmat, seg, ncol, row1, col1, colptr, rowidx, order, kernel_ms, &err);
}

template <typename T>
static int upload_vec(sqpb200_handle h, T** d, const std::vector<T>& v) {
    if (*d) { CK(cudaFree(*d)); *d = nullptr; }
    CK(cudaMalloc((void**)d, std::max<size_t>(v.size(), 1) * sizeof(T)));
    if (!v.empty()) CK(cudaMemcpyAsync(*d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

static int finish_structure_A(sqpb200_handle h) {
    const int nV = h->nV, nC = h->nC, zA = h->zA;
    // CSR view of the CSC pattern: entries of each row in column order (the CSC storage order)
    std::vector<int> Arp(nC + 1, 0), Aci(zA), Aperm(zA);
    for (int e = 0; e < zA; e++) Arp[h->Ai[e] + 1]++;
    for (int r = 0; r < nC; r++) Arp[r + 1] += Arp[r];
    std::vector<int> fill(Arp.begin(), Arp.end() - 1);
    for (int c = 0; c < nV; c++)
        for (int e = h->Ap[c]; e < h->Ap[c + 1]; e++) { int r = h->Ai[e]; Aci[fill[r]] = c; Aperm[fill[r]] = e; fill[r]++; }
    int rc = 0;
    rc |= upload_vec(h, &h->dAp, h->Ap); rc |= upload_vec(h, &h->dAi, h->Ai);
    rc |= upload_vec(h, &h->dArp, Arp); rc |= upload_vec(h, &h->dAci, Aci); rc |= upload_vec(h, &h->dAperm, Aperm);
    rc |= upload_vec(h, &h->dAsrc, h->Asrc);
    if (rc) return SQPB200_ERR_CUDA;
    if (h->dAval) { CK(cudaFree(h->dAval)); h->dAval = nullptr; }
    if (dev_alloc(h, &h->dAval, (size_t)h->batch * zA)) return SQPB200_ERR_CUDA;
    if (!h->A_init.empty() && zA > 0) {  // identity entries (and zeros) in every instance
        if (ensure_stage(h, (size_t)zA * 8)) return SQPB200_ERR_CUDA;
        CK(cudaMemcpyAsync(h->stage, h->A_init.data(), (size_t)zA * 8, cudaMemcpyHostToDevice, h->stream));
        long long total = (long long)h->batch * zA;
        broadcast_rows_kernel<<<grid_for(total, 256), 256, 0, h->stream>>>(total, zA, 0, zA, (const double*)h->stage, h->dAval);
        h->launches++;
        CK(cudaGetLastError());
    }
    h->A_set = true;
    h->cfg_cap_key = -1;  // slice layout depends on zA
    if (h->dgpat) { cudaFree(h->dgpat); h->dgpat = nullptr; }
    return 0;
}

int sqpb200_set_structure_A(sqpb200_handle h, int zJ, const int* row1, const int* col1, int I_len,
                            const int* I_irow, const int* I_jcol, const int* I_size, const double* I_value) {
    if (!h || zJ < 0) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    // entry list of SpHbMat::setStructure(rhs, I_info), src/SpHbMat.cpp:203-227
    std::vector<int> er, ec;
    std::vector<double> ev;
    for (int i = 0; i < zJ; i++) { er.push_back(row1[i]); ec.push_back(col1[i]); ev.push_back(0.0); }
    for (int b = 0; b < I_len; b++)
        for (int j = 0; j < I_size[b]; j++) { er.push_back(I_irow[b] + j); ec.push_back(I_jcol[b] + j); ev.push_back(I_value[b]); }
    int z = (int)er.size();
    for (int i = 0; i < z; i++)
        if (er[i] < 1 || er[i] > h->nC || ec[i] < 1 || ec[i] > h->nV) { h->err = "triplet index out of range"; return SQPB200_ERR_INVALID; }
    h->zA = z; h->zJ = zJ;
    h->qA.set = false;  // a compressed-row view of an earlier structure no longer applies
    h->Ap.assign(h->nV + 1, 0); h->Ai.assign(z, 0); h->Aorder.assign(z, 0);
    int seg[2] = {0, z}, ncol[1] = {h->nV};
    if (z > 0) {
        int rc = run_assembly(h, h->stream, 1, seg, ncol, er.data(), ec.data(), h->Ap.data(), h->Ai.data(), h->Aorder.data(), nullptr, &h->err);
        h->launches++;
        if (rc) return rc;
    }
    h->Asrc.assign(z, -1);
    h->A_init.assign(z, 0.0);
    for (int i = 0; i < z; i++) {
        if (i < zJ) h->Asrc[h->Aorder[i]] = i;
        else h->A_init[h->Aorder[i]] = ev[i];
    }
    int rc = finish_structure_A(h);
    return rc ? rc : z;
}

int sqpb200_set_structure_H(sqpb200_handle h, int zH, const int* row1, const int* col1, int is_symmetric) {
    if (!h || zH < 0) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    // entry list of SpHbMat::setStructure(rhs), src/SpHbMat.cpp:296-309
    std::vector<int> er, ec, srct;
    for (int i = 0; i < zH; i++) {
        er.push_back(row1[i]); ec.push_back(col1[i]); srct.push_back(i);
        if (is_symmetric && row1[i] != col1[i]) { er.push_back(col1[i]); ec.push_back(row1[i]); srct.push_back(i); }
    }
    int z = (int)er.size();
    for (int i = 0; i < z; i++)
        if (er[i] < 1 || er[i] > h->nV || ec[i] < 1 || ec[i] > h->nV) { h->err = "triplet index out of range"; return SQPB200_ERR_INVALID; }
    h->zH = z; h->zHt = zH;
    h->qH.set = false;
    h->Hp.assign(h->nV + 1, 0); h->Hi.assign(z, 0); h->Horder.assign(z, 0);
    int seg[2] = {0, z}, ncol[1] = {h->nV};
    if (z > 0) {
        int rc = run_assembly(h, h->stream, 1, seg, ncol, er.data(), ec.data(), h->Hp.data(), h->Hi.data(), h->Horder.data(), nullptr, &h->err);
        h->launches++;
        if (rc) return rc;
    }
    h->Hsrc.assign(z, -1);
    for (int i = 0; i < z; i++) h->Hsrc[h->Horder[i]] = srct[i];
    int rc = 0;
    rc |= upload_vec(h, &h->dHp, h->Hp); rc |= upload_vec(h, &h->dHi, h->Hi); rc |= upload_vec(h, &h->dHsrc, h->Hsrc);
    if (rc) return SQPB200_ERR_CUDA;
    if (h->dHval) { CK(cudaFree(h->dHval)); h->dHval = nullptr; }
    if (dev_alloc(h, &h->dHval, (size_t)h->batch * z)) return SQPB200_ERR_CUDA;
    h->H_set = true;
    h->cfg_cap_key = -1;
    return z;
}

int sqpb200_set_structure_csc(sqpb200_handle h, int which, int nnz, const int* colptr, const int* rowidx) {
    if (!h || nnz < 0 || !colptr) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    if (colptr[h->nV] != nnz) { h->err = "colptr[ncol] != nnz"; return SQPB200_ERR_INVALID; }
    if (which == SQPB200_MAT_A) {
        h->zA = nnz; h->zJ = nnz;
        h->qA.set = false;
        h->Ap.assign(colptr, colptr + h->nV + 1); h->Ai.assign(rowidx, rowidx + nnz);
        h->Aorder.resize(nnz); h->Asrc.resize(nnz);
        for (int i = 0; i < nnz; i++) { h->Aorder[i] = i; h->Asrc[i] = i; }
        h->A_init.clear();
        int rc = finish_structure_A(h);
        return rc ? rc : nnz;
    } else if (which == SQPB200_MAT_H) {
        h->zH = nnz; h->zHt = nnz;
        h->qH.set = false;
        h->Hp.assign(colptr, colptr + h->nV + 1); h->Hi.assign(rowidx, rowidx + nnz);
        h->Horder.resize(nnz); h->Hsrc.resize(nnz);
        for (int i = 0; i < nnz; i++) { h->Horder[i] = i; h->Hsrc[i] = i; }
        int rc = 0;
        rc |= upload_vec(h, &h->dHp, h->Hp); rc |= upload_vec(h, &h->dHi, h->Hi); rc |= upload_vec(h, &h->dHsrc, h->Hsrc);
        if (rc) return SQPB200_ERR_CUDA;
        if (h->dHval) { CK(cudaFree(h->dHval)); h->dHval = nullptr; }
        if (dev_alloc(h, &h->dHval, (size_t)h->batch * nnz)) return SQPB200_ERR_CUDA;
        h->H_set = true;
        h->cfg_cap_key = -1;
        return nnz;
    }
    return SQPB200_ERR_INVALID;
}

int sqpb200_get_structure(sqpb200_handle h, int which, int* colptr, int* rowidx, int* order) {
    if (!h) return SQPB200_ERR_INVALID;
    const std::vector<int>& P = which == SQPB200_MAT_A ? h->Ap : h->Hp;
    const std::vector<int>& I = which == SQPB200_MAT_A ? h->Ai : h->Hi;
    const std::vector<int>& O = which == SQPB200_MAT_A ? h->Aorder : h->Horder;
    if (P.empty()) return SQPB200_ERR_STATE;
    if (colptr) std::copy(P.begin(), P.end(), colptr);
    if (rowidx) std::copy(I.begin(), I.end(), rowidx);
    if (order) std::copy(O.begin(), O.end(), order);
    return 0;
}

int sqpb200_get_nnz(sqpb200_handle h, int which) {
    if (!h) return SQPB200_ERR_INVALID;
    return which == SQPB200_MAT_A ? h->zA : h->zH;
}

// ------------------------------------------------------------------------------ batched Vector operations (row A2)
int sqpb200_vector_reduce(int device, int op, long long batch, int n, const double* x, const double* y, double* out, int loc, void* stream_) {
    if (batch <= 0 || n < 0 || !x || !out || op < 0 || op > 2 || (op == 2 && !y)) return SQPB200_ERR_INVALID;
    if (cudaSetDevice(device) != cudaSuccess) return SQPB200_ERR_CUDA;
    cudaStream_t stream = (cudaStream_t)stream_;
    const double *dx = x, *dy = y;
    double *dout = out, *tmp = nullptr;
    const size_t bytes = (size_t)batch * (size_t)(n > 0 ? n : 1) * 8;
    if (loc == SQPB200_LOC_HOST) {
        if (cudaMalloc((void**)&tmp, bytes * (op == 2 ? 2 : 1) + (size_t)batch * 8) != cudaSuccess) return SQPB200_ERR_NOMEM;
        double* p = tmp;
        if (n > 0) cudaMemcpyAsync(p, x, bytes, cudaMemcpyHostToDevice, stream);
        dx = p; p += (size_t)batch * (n > 0 ? n : 1);
        if (op == 2) { if (n > 0) cudaMemcpyAsync(p, y, bytes, cudaMemcpyHostToDevice, stream); dy = p; p += (size_t)batch * (n > 0 ? n : 1); }
        dout = p;
    }
    long long g = (batch + 63) / 64;
    if (g > 148LL * 32) g = 148LL * 32;
    vector_reduce_kernel<<<(int)g, 64, 0, stream>>>(batch, n, op, dx, dy, dout);
    cudaError_t e = cudaGetLastError();
    if (loc == SQPB200_LOC_HOST) {
        if (e == cudaSuccess) e = cudaMemcpyAsync(out, dout, (size_t)batch * 8, cudaMemcpyDeviceToHost, stream);
        cudaError_t e2 = cudaStreamSynchronize(stream);
        if (e == cudaSuccess) e = e2;
        cudaFree(tmp);
    }
    return e == cudaSuccess ? 0 : SQPB200_ERR_CUDA;
}

int sqpb200_vector_elementwise(int device, int op, long long batch, int n, double* x, const double* y, double alpha, int loc, void* stream_) {
    if (batch <= 0 || n < 0 || !x || op < 0 || op > 5 || ((op <= 2 || op == 4) && !y)) return SQPB200_ERR_INVALID;
    if (n == 0) return 0;
    if (cudaSetDevice(device) != cudaSuccess) return SQPB200_ERR_CUDA;
    cudaStream_t stream = (cudaStream_t)stream_;
    const long long total = batch * n;
    double *dx = x, *tmp = nullptr;
    const double* dy = y;
    if (loc == SQPB200_LOC_HOST) {
        if (cudaMalloc((void**)&tmp, (size_t)total * 16) != cudaSuccess) return SQPB200_ERR_NOMEM;
        cudaMemcpyAsync(tmp, x, (size_t)total * 8, cudaMemcpyHostToDevice, stream);
        dx = tmp;
        if (y) { cudaMemcpyAsync(tmp + total, y, (size_t)total * 8, cudaMemcpyHostToDevice, stream); dy = tmp + total; }
    }
    vector_elementwise_kernel<<<grid_for(total, 256), 256, 0, stream>>>(total, op, dx, dy, alpha);
    cudaError_t e = cudaGetLastError();
    if (loc == SQPB200_LOC_HOST) {
        if (e == cudaSuccess) e = cudaMemcpyAsync(x, dx, (size_t)total * 8, cudaMemcpyDeviceToHost, stream);
        cudaError_t e2 = cudaStreamSynchronize(stream);
        if (e == cudaSuccess) e = e2;
        cudaFree(tmp);
    }
    return e == cudaSuccess ? 0 : SQPB200_ERR_CUDA;
}

// ------------------------------------------------------------------------------ values
static int set_values(sqpb200_handle h, int which, const double* vals, int loc, int broadcast, bool csc_order) {
    if (!h || !vals) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    bool isA = which == SQPB200_MAT_A;
    if (isA ? !h->A_set : !h->H_set) { h->err = "structure not set"; return SQPB200_ERR_STATE; }
    int z_out = isA ? h->zA : h->zH;
    int z_in = csc_order ? z_out : (isA ? h->zJ : h->zHt);
    if (z_out == 0 || z_in == 0) {  // empty matrix: nothing to copy, but the call still raises Update_A / Update_H (:407-409, 427-429)
        if (h->first_solved) { if (isA) h->upd_A = true; else h->upd_H = true; }
        return 0;
    }
    size_t bytes = (size_t)(broadcast ? 1 : h->batch) * z_in * 8;
    double* dout = isA ? h->dAval : h->dHval;
    long long total = (long long)h->batch * z_out;
    if (csc_order && !broadcast) {
        // one DMA copy straight into place (no staging, no SM-side copy: it must not queue behind resident solve CTAs)
        CK(cudaMemcpyAsync(dout, vals, bytes, loc == SQPB200_LOC_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, h->stream));
        if (h->first_solved) { if (isA) h->upd_A = true; else h->upd_H = true; }
        return 0;
    }
    if (loc == SQPB200_LOC_HOST && ensure_stage(h, bytes)) return SQPB200_ERR_CUDA;
    const void* din;
    if (to_device(h, vals, bytes, loc, 0, &din)) return SQPB200_ERR_CUDA;
    if (csc_order) {
        broadcast_rows_kernel<<<grid_for(total, 256), 256, 0, h->stream>>>(total, z_out, 0, z_out, (const double*)din, dout);
        h->launches++;
    } else {
        scatter_values_kernel<<<grid_for(total, 256), 256, 0, h->stream>>>(total, z_in, z_out, isA ? h->dAsrc : h->dHsrc,
                                                                           (const double*)din, broadcast, dout);
        h->launches++;
    }
    CK(cudaGetLastError());
    // change flags: src/qpOASESInterface.cpp:407-409, 427-429
    if (h->first_solved) { if (isA) h->upd_A = true; else h->upd_H = true; }
    return 0;
}

int sqpb200_set_values_A(sqpb200_handle h, const double* vals, int loc, int broadcast) { return set_values(h, SQPB200_MAT_A, vals, loc, broadcast, false); }
int sqpb200_set_values_H(sqpb200_handle h, const double* vals, int loc, int broadcast) { return set_values(h, SQPB200_MAT_H, vals, loc, broadcast, false); }
int sqpb200_set_values_csc(sqpb200_handle h, int which, const double* vals, int loc, int broadcast) { return set_values(h, which, vals, loc, broadcast, true); }

int sqpb200_get_values_csc(sqpb200_handle h, int which, double* vals, int loc) {
    if (!h || !vals) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    bool isA = which == SQPB200_MAT_A;
    size_t bytes = (size_t)h->batch * (isA ? h->zA : h->zH) * 8;
    CK(cudaMemcpyAsync(vals, isA ? h->dAval : h->dHval, bytes, loc == SQPB200_LOC_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// ------------------------------------------------------------------------------ vectors
static double* vec_ptr(sqpb200_handle h, int which, int* len) {
    switch (which) {
    case SQPB200_VEC_G: *len = h->nV; return h->dg;
    case SQPB200_VEC_LB: *len = h->nV; return h->dlb;
    case SQPB200_VEC_UB: *len = h->nV; return h->dub;
    case SQPB200_VEC_LBA: *len = h->nC; return h->dlbA;
    case SQPB200_VEC_UBA: *len = h->nC; return h->dubA;
    }
    *len = 0;
    return nullptr;
}

int sqpb200_set_vectors(sqpb200_handle h, int which, const double* vals, int offset, int count, int loc, int broadcast) {
    if (!h || !vals) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    int len;
    double* d = vec_ptr(h, which, &len);
    if (!d && len == 0 && count == 0) return 0;
    if (!d || offset < 0 || count < 0 || offset + count > len) return SQPB200_ERR_INVALID;
    if (count == 0) return 0;
    if (!broadcast) {
        const cudaMemcpyKind kind = loc == SQPB200_LOC_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
        if (offset == 0 && count == len) CK(cudaMemcpyAsync(d, vals, (size_t)h->batch * len * 8, kind, h->stream));  // whole vectors: one linear DMA copy
        else CK(cudaMemcpy2DAsync(d + offset, (size_t)len * 8, vals, (size_t)count * 8, (size_t)count * 8, h->batch, kind, h->stream));
    } else {
        if (loc == SQPB200_LOC_HOST && ensure_stage(h, (size_t)count * 8)) return SQPB200_ERR_CUDA;
        const void* din;
        if (to_device(h, vals, (size_t)count * 8, loc, 0, &din)) return SQPB200_ERR_CUDA;
        long long total = (long long)h->batch * count;
        broadcast_rows_kernel<<<grid_for(total, 256), 256, 0, h->stream>>>(total, len, offset, count, (const double*)din, d);
        h->launches++;
        CK(cudaGetLastError());
    }
    // change flags: src/qpOASESInterface.cpp:361-395
    if (h->first_solved) { if (which == SQPB200_VEC_G) h->upd_g = true; else h->upd_bounds = true; }
    return 0;
}

int sqpb200_get_vectors(sqpb200_handle h, int which, double* vals, int loc) {
    if (!h || !vals) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    int len;
    double* d = vec_ptr(h, which, &len);
    if (!d) return SQPB200_ERR_INVALID;
    CK(cudaMemcpyAsync(vals, d, (size_t)h->batch * len * 8, loc == SQPB200_LOC_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int sqpb200_qphandler_bounds(sqpb200_handle h, int mode, int n, int m, const double* delta, const double* x_l,
                             const double* x_u, const double* x_k, const double* c_l, const double* c_u,
                             const double* c_k, int loc) {
    if (!h || n + 2 * m != h->nV || m != h->nC || mode < 0 || mode > 3) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    size_t B = h->batch, bn = B * n * 8, bm = B * m * 8;
    const void *dd, *dxl, *dxu, *dxk, *dcl = nullptr, *dcu = nullptr, *dck = nullptr;
    if (loc == SQPB200_LOC_HOST && ensure_stage(h, B * 8 + 3 * bn + 3 * bm)) return SQPB200_ERR_CUDA;
    size_t off = 0;
    if (to_device(h, delta, B * 8, loc, off, &dd)) return SQPB200_ERR_CUDA; off += B * 8;
    if (to_device(h, x_l, bn, loc, off, &dxl)) return SQPB200_ERR_CUDA; off += bn;
    if (to_device(h, x_u, bn, loc, off, &dxu)) return SQPB200_ERR_CUDA; off += bn;
    if (to_device(h, x_k, bn, loc, off, &dxk)) return SQPB200_ERR_CUDA; off += bn;
    if (mode != 2 && m > 0) {
        if (to_device(h, c_l, bm, loc, off, &dcl)) return SQPB200_ERR_CUDA; off += bm;
        if (to_device(h, c_u, bm, loc, off, &dcu)) return SQPB200_ERR_CUDA; off += bm;
        if (to_device(h, c_k, bm, loc, off, &dck)) return SQPB200_ERR_CUDA; off += bm;
    }
    long long total = (long long)B * h->nV;
    qphandler_bounds_kernel<<<grid_for(total, 256), 256, 0, h->stream>>>(h->batch, (mode != 2 && m > 0) ? mode : 2, n, m, 1.0e18,
        (const double*)dd, (const double*)dxl, (const double*)dxu, (const double*)dxk, (const double*)dcl,
        (const double*)dcu, (const double*)dck, h->dlb, h->dub, h->dlbA, h->dubA);
    h->launches++;
    CK(cudaGetLastError());
    if (mode == 0 && m == 0) { /* nothing else */ }
    if (h->first_solved) h->upd_bounds = true;
    return 0;
}

int sqpb200_qphandler_g(sqpb200_handle h, int n, int m, const double* grad, const double* rho, int loc) {
    if (!h || n + 2 * m != h->nV) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    size_t B = h->batch;
    const void *dgr = nullptr, *drho = nullptr;
    if (loc == SQPB200_LOC_HOST && ensure_stage(h, B * n * 8 + B * 8)) return SQPB200_ERR_CUDA;
    if (grad && to_device(h, grad, B * n * 8, loc, 0, &dgr)) return SQPB200_ERR_CUDA;
    if (rho && to_device(h, rho, B * 8, loc, B * n * 8, &drho)) return SQPB200_ERR_CUDA;
    long long total = (long long)B * h->nV;
    qphandler_g_kernel<<<grid_for(total, 256), 256, 0, h->stream>>>(h->batch, n, m, (const double*)dgr, (const double*)drho, h->dg);
    h->launches++;
    CK(cudaGetLastError());
    if (h->first_solved) h->upd_g = true;
    return 0;
}

// ------------------------------------------------------------------------------ solve
static void fill_dims(sqpb200_handle h, QPKernelArgs& a, int cap) {
    memset(&a, 0, sizeof a);
    a.batch = h->batch; a.nV = h->nV; a.nC = h->nC; a.cap = cap; a.large = h->large ? 1 : 0;
    a.is_lp = (h->qptype == SQPB200_LP); a.has_H = !a.is_lp;
    a.zA = h->zA; a.zH = a.is_lp ? 0 : h->zH;  // an LP handle never holds H (src/qpOASESInterface.cpp:122-124)
    qp_fill_layout(a);
}

// QPs (warps) per CTA in {4, 2, 1} for a given factor capacity: the one that keeps the most QPs resident per SM.
// allow_subwarp: QPs with nV <= 16 / <= 8 run on teams of 16 / 8 lanes (2 / 4 QPs per warp, 8 / 16 QPs per 128-thread CTA).
static bool config_for_cap(sqpb200_handle h, int cap, SolveCfg& cfg, bool allow_subwarp = false) {
    QPKernelArgs a;
    fill_dims(h, a, cap);
    const size_t slice_bytes = (size_t)a.slice_doubles * 8, pat_bytes = (size_t)a.pat_shorts * 2;
    const size_t SMEM_MAX = 227 * 1024, SMEM_SM = 228 * 1024;
    cfg.lanes = 32;
    if (allow_subwarp && h->nV <= 16) {
        const int lanes = h->nV <= 8 ? 8 : 16, teams = 128 / lanes;
        const size_t smem = (size_t)teams * slice_bytes + pat_bytes;
        if (smem <= SMEM_MAX) {
            size_t ctas = SMEM_SM / (smem + 1024 + 512);
            if (ctas > 4) ctas = 4;  // 16 warps per SM (the 128-register build)
            if (ctas >= 1) {
                cfg.cap = a.cap; cfg.teams = teams; cfg.smem = (int)smem; cfg.lanes = lanes;
                cfg.slice_doubles = a.slice_doubles; cfg.state_doubles = a.state_doubles; cfg.resident = (int)(ctas * 4);
                return true;
            }
        }
    }
    int best_teams = 0;
    size_t best_res = 0;
    for (int teams = 4; teams >= 1; teams >>= 1) {
        size_t smem = (size_t)teams * slice_bytes + pat_bytes;
        if (smem > SMEM_MAX) continue;
        size_t ctas = SMEM_SM / (smem + 1024 + 512);  // 1 KiB per CTA reserved by the driver + the static argument copy
        if (ctas > 32) ctas = 32;
        size_t res = ctas * teams;
        if (res > 64) res = 64;  // 64 warps per SM
        if (res > best_res) { best_res = res; best_teams = teams; }
    }
    cfg.cap = a.cap; cfg.teams = best_teams; cfg.smem = (int)((size_t)best_teams * slice_bytes + pat_bytes);
    cfg.slice_doubles = a.slice_doubles; cfg.state_doubles = a.state_doubles; cfg.resident = (int)best_res;
    return best_teams > 0;
}

static int choose_config(sqpb200_handle h) {
    // One warp per QP: the only shared-memory resident team size shipped this round (see the note in qp_kernel.cuh).
    if (h->opt.team_size != 0 && h->opt.team_size != 32 && h->opt.team_size != 1024) { h->err = "team_size must be 0 (auto), 32 (warp per QP) or 1024 (CTA per QP)"; return SQPB200_ERR_INVALID; }
    const int nV = h->nV, nC = h->nC;
    // Factor capacity.  On the l1-penalty QPs of RestartSQP (x = [p; u; v], nV = n + 2m) the number of simultaneously free
    // variables stays near n: slacks are free only on violated rows.  auto: n + ceil(m/2) + 2; instances that need more are
    // re-solved by the rescue launch with the full capacity nV, so the choice only affects speed, never results.
    int cap = h->opt.factor_cap;
    if (cap == 0) {
        if (h->maxfr_pending && cudaEventQuery(h->ev_maxfr) == cudaSuccess) {
            if (*h->maxfr_host > h->maxfr_seen) h->maxfr_seen = *h->maxfr_host;
            h->maxfr_valid = true; h->maxfr_pending = false;
        }
        int n_est = (nV >= 2 * nC) ? nV - 2 * nC : nV;
        // learned: what this handle's QPs needed so far (+2); before the first read-back: n + ceil(m/2) + 2
        cap = h->maxfr_valid ? h->maxfr_seen + 2 : n_est + (nC + 1) / 2 + 2;
    }
    if (cap < 0 || cap > nV) cap = nV;
    if (cap == h->cfg_cap_key && h->team != 0) return 0;  // configuration already chosen for this capacity
    h->cfg_cap_key = cap;
    const bool fits16 = h->zA < 32768 && h->zH < 32768;
    h->large = (h->opt.team_size == 1024);
    if (!h->large) {
        h->have_rescue = fits16 && config_for_cap(h, nV, h->cfg_rescue);
        // without a rescue configuration the main launch must hold every QP: full capacity
        if (!fits16 || !h->have_rescue || !config_for_cap(h, cap, h->cfg_main, h->opt.team_size == 0)) {
            if (h->opt.team_size == 32) {
                h->err = "QP too large for the shared-memory resident kernel (nV=" + std::to_string(nV) + ", capacity " + std::to_string(cap) + ")";
                return SQPB200_ERR_TOO_LARGE;
            }
            h->large = true;
        }
    }
    if (h->large) {
        QPKernelArgs a;
        fill_dims(h, a, nV);
        h->large_slice_doubles = a.slice_doubles;
        h->team = 1024; h->teams_per_cta = 1; h->smem_cta = 0;
        h->slice_doubles = a.slice_doubles;
        return 0;
    }
    h->team = h->cfg_main.lanes; h->teams_per_cta = h->cfg_main.teams; h->smem_cta = h->cfg_main.smem;
    h->slice_doubles = h->cfg_main.slice_doubles;
    return 0;
}

// one object file per CTA size (qp_solve_inst.cu)
namespace sqpb200 {
cudaError_t launch_qp_solve_32_128_w16(const QPKernelArgs&, int, cudaStream_t);
cudaError_t launch_qp_solve_32_128_w32(const QPKernelArgs&, int, cudaStream_t);
cudaError_t launch_qp_solve_32_64_w16(const QPKernelArgs&, int, cudaStream_t);
cudaError_t launch_qp_solve_32_32_w16(const QPKernelArgs&, int, cudaStream_t);
cudaError_t launch_qp_solve_16_128_w16(const QPKernelArgs&, int, cudaStream_t);
cudaError_t launch_qp_solve_8_128_w16(const QPKernelArgs&, int, cudaStream_t);
cudaError_t launch_qp_solve_large(const QPKernelArgs&, cudaStream_t);
}

// global-memory slices and the 32-bit pattern of the one-QP-per-CTA kernel
static int prepare_large(sqpb200_handle h, const QPKernelArgs& a) {
    if (!h->dgwork) {
        if (dev_alloc(h, &h->dgwork, (size_t)h->batch * a.slice_doubles)) return SQPB200_ERR_CUDA;  // zeroed: "not initialised"
    }
    if (!h->dgpat) {
        std::vector<int> pat((size_t)a.pat_shorts + 4, 0);
        std::vector<int> Arp(h->nC + 1, 0), Aci(h->zA), Aperm(h->zA);
        for (int e = 0; e < h->zA; e++) Arp[h->Ai[e] + 1]++;
        for (int r = 0; r < h->nC; r++) Arp[r + 1] += Arp[r];
        std::vector<int> fill(Arp.begin(), Arp.end() - 1);
        for (int c = 0; c < h->nV; c++)
            for (int e = h->Ap[c]; e < h->Ap[c + 1]; e++) { int r = h->Ai[e]; Aci[fill[r]] = c; Aperm[fill[r]] = e; fill[r]++; }
        std::copy(h->Ap.begin(), h->Ap.end(), pat.begin() + a.pAp);
        std::copy(h->Ai.begin(), h->Ai.end(), pat.begin() + a.pAi);
        std::copy(Arp.begin(), Arp.end(), pat.begin() + a.pArp);
        std::copy(Aci.begin(), Aci.end(), pat.begin() + a.pAci);
        std::copy(Aperm.begin(), Aperm.end(), pat.begin() + a.pAperm);
        if (a.zH > 0) {
            std::copy(h->Hp.begin(), h->Hp.end(), pat.begin() + a.pHp);
            std::copy(h->Hi.begin(), h->Hi.end(), pat.begin() + a.pHi);
        }
        if (upload_vec(h, &h->dgpat, pat)) return SQPB200_ERR_CUDA;
    }
    return 0;
}
static cudaError_t launch_cfg(const SolveCfg& cfg, const QPKernelArgs& a, cudaStream_t stream) {
    if (cfg.lanes == 16) return launch_qp_solve_16_128_w16(a, cfg.smem, stream);
    if (cfg.lanes == 8) return launch_qp_solve_8_128_w16(a, cfg.smem, stream);
    switch (cfg.teams) {
    // 4 QPs per CTA and shared memory allows >= 32 resident warps: the 64-register build (see qp_kernel.cuh)
    case 4: return cfg.resident >= 32 ? launch_qp_solve_32_128_w32(a, cfg.smem, stream) : launch_qp_solve_32_128_w16(a, cfg.smem, stream);
    case 2: return launch_qp_solve_32_64_w16(a, cfg.smem, stream);
    default: return launch_qp_solve_32_32_w16(a, cfg.smem, stream);
    }
}

static int solve_impl(sqpb200_handle h, int mode_qp, int maxiter, const unsigned char* active_mask, bool mask_on_device, signed char* inst_state);
int sqpb200_solve(sqpb200_handle h, int mode_qp, int maxiter, const unsigned char* active_mask) {
    return solve_impl(h, mode_qp, maxiter, active_mask, false, nullptr);
}
int sqpb200_solve_device_mask(sqpb200_handle h, int mode_qp, int maxiter, const unsigned char* device_mask) {
    return solve_impl(h, mode_qp, maxiter, device_mask, true, nullptr);
}
int sqpb200_solve_per_instance(sqpb200_handle h, int mode_qp, int maxiter, const unsigned char* device_mask, signed char* device_inst_state) {
    if (!h || !device_inst_state || !h->opt.keep_state) return SQPB200_ERR_INVALID;
    return solve_impl(h, mode_qp, maxiter, device_mask, true, device_inst_state);
}
int sqpb200_device_buffers(sqpb200_handle h, void** out) {
    if (!h || !out) return SQPB200_ERR_INVALID;
    out[0] = h->dx; out[1] = h->dy; out[2] = h->dobj; out[3] = h->dstatus; out[4] = h->diters; out[5] = h->dkkt;
    return 0;
}
// What the first solve of a handle allocates -- the launch configuration, the hot-start images of the warp kernel, the global-memory
// slices and pattern of the one-QP-per-cluster kernel -- made without solving.  sqpb200_sqp_graph_create calls it before it records
// solves into a CUDA graph, where an allocation and the memset that zeroes it must not happen.  (Not part of the public header.)
int sqpb200_solve_prepare(sqpb200_handle h) {
    if (!h) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    if (!h->A_set) { h->err = "set_structure_A has not been called"; return SQPB200_ERR_STATE; }
    if (h->qptype == SQPB200_QP && !h->H_set) { h->err = "set_structure_H has not been called"; return SQPB200_ERR_STATE; }
    int rc = choose_config(h);
    if (rc) return rc;
    if (!h->large && h->opt.keep_state && !h->dstate) {
        if (dev_alloc(h, &h->dstate, (size_t)h->batch * h->cfg_main.state_doubles)) return SQPB200_ERR_CUDA;
    }
    if (h->large) {
        QPKernelArgs a;
        fill_dims(h, a, h->nV);
        return prepare_large(h, a);
    }
    return 0;
}

static int solve_impl(sqpb200_handle h, int mode_qp, int maxiter, const unsigned char* active_mask, bool mask_on_device, signed char* inst_state) {
    if (!h) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    bool is_lp = (mode_qp == SQPB200_LP);
    if (mode_qp != h->qptype) { h->err = "solve mode differs from the handle's QPType (the reference keeps one backend per type)"; return SQPB200_ERR_INVALID; }
    int rc = sqpb200_solve_prepare(h);
    if (rc) return rc;
    // a solve recorded into a CUDA graph (sqpb200_sqp_graph_create) reads nothing back and records no timing events: the capacity
    // frozen in the graph affects speed, never results (the rescue launch)
    cudaStreamCaptureStatus capture = cudaStreamCaptureStatusNone;
    CK(cudaStreamIsCapturing(h->stream, &capture));
    const bool recording = capture != cudaStreamCaptureStatusNone;
    // init / hotstart decision: src/qpOASESInterface.cpp:141-211 with get_Matrix_change_status :817-833
    int mode = MODE_COLD;
    if (h->first_solved && h->opt.keep_state) {
        bool varied = h->upd_A || h->upd_H;
        if (h->old_ms == MS_UNDEFINED) h->old_ms = varied ? MS_VARIED : MS_FIXED;
        else { if (h->new_ms != MS_UNDEFINED) h->old_ms = h->new_ms; h->new_ms = varied ? MS_VARIED : MS_FIXED; }
        if (h->new_ms == MS_UNDEFINED) mode = (h->old_ms == MS_FIXED) ? MODE_HOT_FIXED : MODE_HOT_VARIED;
        else if (h->new_ms == MS_FIXED && h->old_ms == MS_FIXED) mode = MODE_HOT_FIXED;
        else if (h->new_ms == MS_VARIED && h->old_ms == MS_VARIED) mode = MODE_HOT_VARIED;
        else {  // status flip: init(..., x_qp, y_qp, &bounds) :202-207, a fresh init from the previous solution
            mode = MODE_REINIT;
            h->new_ms = h->old_ms = MS_UNDEFINED;
        }
    }
    QPKernelArgs a;
    fill_dims(h, a, h->large ? h->nV : h->cfg_main.cap);
    a.max_iter = maxiter > 0 ? maxiter : (is_lp ? h->opt.lp_maxiter : h->opt.qp_maxiter);
    a.flags = (h->opt.enable_flipping ? FLAG_FLIPPING : 0) | (h->opt.enable_ramping ? FLAG_RAMPING : 0) |
              (h->opt.enable_drift ? FLAG_DRIFT : 0) | (h->opt.keep_state ? FLAG_KEEP_STATE : 0) |
              (h->opt.debug_force_error_branch ? FLAG_FORCE_GUESS : 0) | (h->opt.refactorise_every == 1 ? FLAG_NO_CARRY : 0);
    a.mode = mode;
    a.Ap = h->dAp; a.Ai = h->dAi; a.Arp = h->dArp; a.Aci = h->dAci; a.Aperm = h->dAperm;
    a.Hp = h->dHp; a.Hi = h->dHi;
    a.Aval = h->dAval; a.Hval = h->dHval;
    a.gN = h->dg; a.lbN = h->dlb; a.ubN = h->dub; a.lbAN = h->dlbA; a.ubAN = h->dubA;
    if (active_mask && mask_on_device) a.mask = active_mask;
    else if (active_mask) {
        CK(cudaMemcpyAsync(h->dmask, active_mask, h->batch, cudaMemcpyHostToDevice, h->stream));
        a.mask = h->dmask;
    }
    a.x = h->dx; a.y = h->dy; a.obj = h->dobj; a.kkt = h->dkkt; a.status = h->dstatus; a.iters = h->diters;
    a.wsB = h->dwsB; a.wsC = h->dwsC; a.WB = h->dWB; a.WC = h->dWC;
    a.state = h->dstate;
    a.maxfr = h->dmaxfr;
    a.ncap = h->dncap; a.caplist = h->dncap + 1;
    a.prof = h->dprof;
    a.inst_state = inst_state;  // per-instance init/hotstart decisions (made in the kernel) replace the handle-level `mode`
    if (h->large) {
        a.gpat = h->dgpat; a.gwork = h->dgwork;
        if (!recording) CK(cudaEventRecord(h->ev0, h->stream));
        cudaError_t el = launch_qp_solve_large(a, h->stream);
        if (el != cudaSuccess) { h->err = std::string("qp_solve_large_kernel launch: ") + cudaGetErrorString(el); return SQPB200_ERR_CUDA; }
        if (!recording) CK(cudaEventRecord(h->ev1, h->stream));
        h->launches++;
        h->upd_A = h->upd_H = h->upd_g = h->upd_bounds = false;
        h->first_solved = true;
        return 0;
    }
    if (!recording) CK(cudaEventRecord(h->ev0, h->stream));
    if (h->cfg_main.cap < h->nV) CK(cudaMemsetAsync(h->dncap, 0, sizeof(int), h->stream));
    cudaError_t e = launch_cfg(h->cfg_main, a, h->stream);
    if (e != cudaSuccess) { h->err = std::string("qp_solve_kernel launch: ") + cudaGetErrorString(e); return SQPB200_ERR_CUDA; }
    if (h->cfg_main.cap < h->nV) {
        // rescue launch: instances that needed more free variables than the capacity are re-solved from their pre-solve
        // state with the full-size factors; every other warp exits at once.  No host synchronisation in between.
        QPKernelArgs r = a;
        r.cap = h->nV; r.rescue = 1;
        qp_fill_layout(r);
        if (h->have_rescue) {
            e = launch_cfg(h->cfg_rescue, r, h->stream);
            if (e != cudaSuccess) { h->err = std::string("qp_solve_kernel rescue launch: ") + cudaGetErrorString(e); return SQPB200_ERR_CUDA; }
            h->launches++;
        }
    }
    if (!recording) CK(cudaEventRecord(h->ev1, h->stream));
    h->launches++;
    if (h->opt.factor_cap == 0 && !recording) {  // learn the capacity for later solves (asynchronous: never waited for)
        CK(cudaMemcpyAsync(h->maxfr_host, h->dmaxfr, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaEventRecord(h->ev_maxfr, h->stream));
        h->maxfr_pending = true;
    }
    // reset_flags(): src/qpOASESInterface.cpp:488-496
    h->upd_A = h->upd_H = h->upd_g = h->upd_bounds = false;
    h->first_solved = true;
    return 0;
}

int sqpb200_io_layout(sqpb200_handle h, size_t* in_off5, size_t* in_bytes, size_t* out_off6, size_t* out_bytes) {
    if (!h) return SQPB200_ERR_INVALID;
    if (in_off5) for (int i = 0; i < 5; i++) in_off5[i] = h->in_off[i];
    if (in_bytes) *in_bytes = h->in_bytes;
    if (out_off6) for (int i = 0; i < 6; i++) out_off6[i] = h->out_off[i];
    if (out_bytes) *out_bytes = h->out_bytes;
    return 0;
}

int sqpb200_solve_host(sqpb200_handle h, int mode, int maxiter, const void* in_block, const double* Aval_csc, const double* Hval_csc,
                       void* out_block) {
    if (!h) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    if (in_block) {
        CK(cudaMemcpyAsync(h->arena, in_block, h->in_bytes, cudaMemcpyHostToDevice, h->stream));
        if (h->first_solved) { h->upd_g = true; h->upd_bounds = true; }
    }
    if (Aval_csc) {
        if (!h->A_set) { h->err = "structure not set"; return SQPB200_ERR_STATE; }
        if (h->zA > 0) CK(cudaMemcpyAsync(h->dAval, Aval_csc, (size_t)h->batch * h->zA * 8, cudaMemcpyHostToDevice, h->stream));
        if (h->first_solved) h->upd_A = true;
    }
    if (Hval_csc) {
        if (!h->H_set) { h->err = "structure not set"; return SQPB200_ERR_STATE; }
        if (h->zH > 0) CK(cudaMemcpyAsync(h->dHval, Hval_csc, (size_t)h->batch * h->zH * 8, cudaMemcpyHostToDevice, h->stream));
        if (h->first_solved) h->upd_H = true;
    }
    int rc = solve_impl(h, mode, maxiter, nullptr, false, nullptr);
    if (rc) return rc;
    if (out_block) CK(cudaMemcpyAsync(out_block, (char*)h->arena + h->out_base, h->out_bytes, cudaMemcpyDeviceToHost, h->stream));
    return 0;
}

float sqpb200_last_solve_ms(sqpb200_handle h) {
    if (!h || !h->ev1) return -1.f;
    if (cudaEventSynchronize(h->ev1) != cudaSuccess) return -1.f;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, h->ev0, h->ev1);
    h->last_ms = ms;
    return ms;
}

int sqpb200_solve_config(sqpb200_handle h, int* team_size, int* qps_per_cta, int* smem_per_cta) {
    if (!h) return SQPB200_ERR_INVALID;
    if (h->team == 0) { int rc = choose_config(h); if (rc) return rc; }
    if (team_size) *team_size = h->team;
    if (qps_per_cta) *qps_per_cta = h->teams_per_cta;
    if (smem_per_cta) *smem_per_cta = h->smem_cta;
    return 0;
}

long long sqpb200_launch_count(sqpb200_handle h) { return h ? h->launches : 0; }

int sqpb200_get_profile(sqpb200_handle h, long long* out16, int reset) {
    if (!h || !out16 || !h->dprof) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(out16, h->dprof, 16 * sizeof(long long), cudaMemcpyDeviceToHost));
    if (reset) CK(cudaMemset(h->dprof, 0, 16 * sizeof(long long)));
    return 0;
}

// ------------------------------------------------------------------------------ results
static int copy_out(sqpb200_handle h, void* dst, const void* src, size_t bytes, int loc) {
    if (!dst) return 0;
    CK(cudaMemcpyAsync(dst, src, bytes, loc == SQPB200_LOC_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, h->stream));
    return 0;
}

int sqpb200_get_solution(sqpb200_handle h, double* x, double* y, double* obj, int* status, int* iters, int loc) {
    if (!h) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    size_t B = h->batch;
    if (copy_out(h, x, h->dx, B * h->nV * 8, loc) || copy_out(h, y, h->dy, B * (h->nV + h->nC) * 8, loc) ||
        copy_out(h, obj, h->dobj, B * 8, loc) || copy_out(h, status, h->dstatus, B * 4, loc) ||
        copy_out(h, iters, h->diters, B * 4, loc))
        return SQPB200_ERR_CUDA;
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int sqpb200_get_working_set(sqpb200_handle h, int* wb, int* wc, int translated, int loc) {
    if (!h) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    size_t B = h->batch;
    if (translated) {
        if (copy_out(h, wb, h->dWB, B * h->nV * 4, loc) || copy_out(h, wc, h->dWC, B * h->nC * 4, loc)) return SQPB200_ERR_CUDA;
    } else {
        size_t nb = B * h->nV, nc = B * h->nC;
        if (ensure_stage(h, (nb + nc) * 4 + 16)) return SQPB200_ERR_CUDA;
        int* sb = (int*)h->stage;
        int* sc = sb + nb;
        widen_ws_kernel<<<grid_for((long long)nb, 256), 256, 0, h->stream>>>((long long)nb, h->dwsB, sb);
        if (nc) widen_ws_kernel<<<grid_for((long long)nc, 256), 256, 0, h->stream>>>((long long)nc, h->dwsC, sc);
        h->launches += nc ? 2 : 1;
        CK(cudaGetLastError());
        if (copy_out(h, wb, sb, nb * 4, loc) || copy_out(h, wc, sc, nc * 4, loc)) return SQPB200_ERR_CUDA;
    }
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int sqpb200_kkt_residuals(sqpb200_handle h, double* out, int loc) {
    if (!h || !out) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    if (copy_out(h, out, h->dkkt, (size_t)h->batch * 5 * 8, loc)) return SQPB200_ERR_CUDA;
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int sqpb200_kkt_residuals_recompute(sqpb200_handle h, double* out, int loc) {
    if (!h || !out) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    if (!h->A_set) return SQPB200_ERR_STATE;
    KKTArgs a;
    memset(&a, 0, sizeof a);
    a.batch = h->batch; a.nV = h->nV; a.nC = h->nC; a.zA = h->zA; a.zH = h->zH;
    a.has_H = (h->qptype == SQPB200_QP && h->H_set) ? 1 : 0;
    a.Ap = h->dAp; a.Ai = h->dAi; a.Arp = h->dArp; a.Aci = h->dAci; a.Aperm = h->dAperm; a.Hp = h->dHp; a.Hi = h->dHi;
    a.Aval = h->dAval; a.Hval = h->dHval; a.g = h->dg; a.lb = h->dlb; a.ub = h->dub; a.lbA = h->dlbA; a.ubA = h->dubA;
    a.x = h->dx; a.y = h->dy; a.wsB = h->dwsB; a.wsC = h->dwsC; a.WB = h->dWB; a.WC = h->dWC;
    if (ensure_stage(h, (size_t)h->batch * 5 * 8)) return SQPB200_ERR_CUDA;
    a.out = (loc == SQPB200_LOC_DEVICE) ? out : (double*)h->stage;
    // TMA-staged kernel: G instances (warps) per CTA, two stages; largest G in {8, 4, 2} that keeps two CTAs per SM
    // (or fits at all); the plain warp-per-instance kernel remains for instances too large for that
    {
        const bool aligned = (((uintptr_t)a.Aval | (uintptr_t)a.Hval | (uintptr_t)a.x | (uintptr_t)a.y | (uintptr_t)a.g | (uintptr_t)a.lb |
                               (uintptr_t)a.ub | (uintptr_t)a.lbA | (uintptr_t)a.ubA) & 15) == 0;
        // (G warps per CTA, stages) that keeps the most warps resident per SM; ties go to two stages
        const int zHk = a.has_H ? h->zH : 0;
        int G = 0, stages = 0, best_warps = 0;
        size_t smem_t = 0;
        for (int st = 2; st >= 1 && aligned; st--)
            for (int g = 8; g >= 2; g >>= 1) {
                KKTLayout Lg = kkt_layout(g, st, h->nV, h->nC, h->zA, zHk);
                size_t sm = kkt_smem_bytes(Lg);
                if (sm > 227 * 1024) continue;
                int ctas = (int)((228 * 1024) / (sm + 1024));
                int warps = ctas * g;
                if (warps > 64) warps = 64;
                if (warps > best_warps) { best_warps = warps; G = g; stages = st; smem_t = sm; }
            }
        if (G) {
            KKTArgs at = a;
            if (!at.has_H) at.zH = 0;
            KKTLayout Lg = kkt_layout(G, stages, h->nV, h->nC, h->zA, at.zH);
            if (smem_t > 48 * 1024) CK(cudaFuncSetAttribute(kkt_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_t));
            long long ngroups = ((long long)h->batch + G - 1) / G;
            int per_sm = (int)((228 * 1024) / (smem_t + 1024));
            if (per_sm < 1) per_sm = 1;
            if (per_sm * G > 64) per_sm = 64 / G;
            long long grid = ngroups < 148LL * per_sm ? ngroups : 148LL * per_sm;
            kkt_tma_kernel<<<(int)grid, G * 32, smem_t, h->stream>>>(at, Lg);
            h->launches++;
            CK(cudaGetLastError());
            if (loc == SQPB200_LOC_HOST) CK(cudaMemcpyAsync(out, h->stage, (size_t)h->batch * 5 * 8, cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            return 0;
        }
    }
    const size_t per_warp = kkt_warp_doubles(h->nV, h->nC, h->zA, h->zH) * 8;
    int warps = 4;
    while (warps > 1 && (size_t)warps * per_warp > 24 * 1024) warps >>= 1;
    size_t smem = (size_t)warps * per_warp;
    if (smem > 227 * 1024) { h->err = "KKT kernel: instance too large for shared-memory staging"; return SQPB200_ERR_TOO_LARGE; }
    if (smem > 48 * 1024) CK(cudaFuncSetAttribute(kkt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kkt_kernel<<<(h->batch + warps - 1) / warps, warps * 32, smem, h->stream>>>(a);
    h->launches++;
    CK(cudaGetLastError());
    if (loc == SQPB200_LOC_HOST) CK(cudaMemcpyAsync(out, h->stage, (size_t)h->batch * 5 * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int sqpb200_spmv(sqpb200_handle h, int which, int transpose, const double* x, double* y, int loc) {
    if (!h || !x || !y) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    bool isA = which == SQPB200_MAT_A;
    if (isA ? !h->A_set : !h->H_set) return SQPB200_ERR_STATE;
    int nin, nout, nnz;
    const int *ptr, *idx, *perm;
    const double* val;
    if (isA && !transpose) { nin = h->nV; nout = h->nC; nnz = h->zA; ptr = h->dArp; idx = h->dAci; perm = h->dAperm; val = h->dAval; }
    else if (isA) { nin = h->nC; nout = h->nV; nnz = h->zA; ptr = h->dAp; idx = h->dAi; perm = nullptr; val = h->dAval; }
    else { nin = h->nV; nout = h->nV; nnz = h->zH; ptr = h->dHp; idx = h->dHi; perm = nullptr; val = h->dHval; }
    size_t B = h->batch, bin = B * nin * 8, bout = B * nout * 8;
    if (nout == 0) return 0;
    const void* dxv = x;
    double* dyv = y;
    if (loc == SQPB200_LOC_HOST) {
        if (ensure_stage(h, bin + bout + 16)) return SQPB200_ERR_CUDA;
        if (to_device(h, x, bin, loc, 0, &dxv)) return SQPB200_ERR_CUDA;
        dyv = (double*)((char*)h->stage + ((bin + 15) / 16) * 16);
    }
    long long total = (long long)B * nout;
    {
        // TMA-staged kernel: groups of G instances (G even), two shared-memory stages of ~20 KB each filled by bulk
        // asynchronous copies; the one-thread-per-output kernel remains for instances too large for a stage
        const size_t pat_bytes = ((size_t)nout + 1 + 2 * (size_t)nnz) * 4 + 16;
        const size_t per_inst = ((size_t)nnz + nin) * 8;
        const size_t budget = 44 * 1024;
        int G = (int)((budget > pat_bytes ? (budget - pat_bytes) / 2 : 0) / (per_inst ? per_inst : 1));
        G &= ~1;
        const bool aligned = (((uintptr_t)val | (uintptr_t)dxv) & 15) == 0;
        if (G >= 2 && aligned) {
            if ((long long)G > (long long)B) G = (int)((B + 1) & ~1ull);
            const size_t smem = 2 * (size_t)G * per_inst + pat_bytes;
            long long ngroups = ((long long)B + G - 1) / G;
            long long grid = ngroups < 148LL * 5 ? ngroups : 148LL * 5;
            spmv_tma_kernel<<<(int)grid, 256, smem, h->stream>>>((long long)B, G, nout, nin, nnz, ptr, idx, perm, val, (const double*)dxv, dyv);
        } else {
            spmv_kernel<<<grid_for(total, 256), 256, 0, h->stream>>>(total, nout, nin, nnz, ptr, idx, perm, val, (const double*)dxv, dyv);
        }
    }
    h->launches++;
    CK(cudaGetLastError());
    if (loc == SQPB200_LOC_HOST) {
        CK(cudaMemcpyAsync(y, dyv, bout, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }  // device pointers: asynchronous on the handle's stream
    return 0;
}

// ------------------------------------------------------------------------------ QORE layout (compressed-row matrices, stacked bounds)
// The reference's QORE backend keeps A and H row-compressed and one lb / ub pair of length nV + nC (src/QOREInterface.cpp:89-102,
// 191-219).  These entry points accept and return that layout; the solve kernels keep working on the column-compressed pattern,
// which is derived here once per structure (host, O(nnz)), and values move between the two storage orders through position
// maps on the device (scatter_values_kernel in its gather form).
__global__ void qore_workingset_kernel(long long total, int nV, int nC, const signed char* __restrict__ wsB,
                                       const signed char* __restrict__ wsC, int* __restrict__ out) {
    // QORE's sign is the opposite of qpOASES's: src/QOREInterface.cpp:445-458 reads -1 as "at the upper bound" where
    // src/qpOASESInterface.cpp:848-861 reads +1
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const int ld = nV + nC;
    for (; t < total; t += stride) {
        const long long b = t / ld;
        const int i = (int)(t - b * ld);
        const int w = i < nV ? (int)wsB[b * nV + i] : (int)wsC[b * nC + (i - nV)];
        out[t] = -w;
    }
}

// compressed-row (rp, ci) -> compressed-column (cp, ri) plus the position map q2c; entries with equal keys keep their order
static void csr_to_csc(int nrow, int ncol, const std::vector<int>& rp, const std::vector<int>& ci, std::vector<int>& cp,
                       std::vector<int>& ri, std::vector<int>& q2c) {
    const int z = (int)ci.size();
    cp.assign(ncol + 1, 0); ri.assign(z, 0); q2c.assign(z, 0);
    for (int e = 0; e < z; e++) cp[ci[e] + 1]++;
    for (int c = 0; c < ncol; c++) cp[c + 1] += cp[c];
    std::vector<int> fill(cp.begin(), cp.end() - 1);
    for (int r = 0; r < nrow; r++)
        for (int e = rp[r]; e < rp[r + 1]; e++) { const int pos = fill[ci[e]]++; ri[pos] = r; q2c[e] = pos; }
}

static int finish_csr_view(sqpb200_handle h, sqpb200_handle_s::CsrView& q) {
    const int z = (int)q.ci.size();
    q.c2q.assign(z, 0);
    for (int e = 0; e < z; e++) q.c2q[q.q2c[e]] = e;
    if (upload_vec(h, &q.dq2c, q.q2c) || upload_vec(h, &q.dc2q, q.c2q)) return SQPB200_ERR_CUDA;
    q.set = true;
    return 0;
}

static int finish_structure_H(sqpb200_handle h) {
    int rc = 0;
    rc |= upload_vec(h, &h->dHp, h->Hp); rc |= upload_vec(h, &h->dHi, h->Hi); rc |= upload_vec(h, &h->dHsrc, h->Hsrc);
    if (rc) return SQPB200_ERR_CUDA;
    if (h->dHval) { CK(cudaFree(h->dHval)); h->dHval = nullptr; }
    if (dev_alloc(h, &h->dHval, (size_t)h->batch * h->zH)) return SQPB200_ERR_CUDA;
    h->H_set = true;
    h->cfg_cap_key = -1;
    return 0;
}

int sqpb200_set_structure_A_csr(sqpb200_handle h, int zJ, const int* row1, const int* col1, int I_len, const int* I_irow,
                                const int* I_jcol, const int* I_size, const double* I_value) {
    if (!h || zJ < 0) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    // entry list of SpHbMat::setStructure(rhs, I_info), src/SpHbMat.cpp:203-227
    std::vector<int> er, ec;
    std::vector<double> ev;
    for (int i = 0; i < zJ; i++) { er.push_back(row1[i]); ec.push_back(col1[i]); ev.push_back(0.0); }
    for (int b = 0; b < I_len; b++)
        for (int j = 0; j < I_size[b]; j++) { er.push_back(I_irow[b] + j); ec.push_back(I_jcol[b] + j); ev.push_back(I_value[b]); }
    const int z = (int)er.size();
    for (int i = 0; i < z; i++)
        if (er[i] < 1 || er[i] > h->nC || ec[i] < 1 || ec[i] > h->nV) { h->err = "triplet index out of range"; return SQPB200_ERR_INVALID; }
    if (h->nV >= (1 << 21)) { h->err = "matrix too large for packed keys"; return SQPB200_ERR_TOO_LARGE; }
    // compressed-row branch (:238-250): the device sort with the roles of row and column exchanged, key (row, column, counter)
    auto& q = h->qA;
    q.rp.assign(h->nC + 1, 0); q.ci.assign(z, 0); q.order.assign(z, 0);
    int seg[2] = {0, z}, nrow[1] = {h->nC};
    if (z > 0) {
        int rc = run_assembly(h, h->stream, 1, seg, nrow, ec.data(), er.data(), q.rp.data(), q.ci.data(), q.order.data(), nullptr, &h->err);
        h->launches++;
        if (rc) return rc;
    }
    h->zA = z; h->zJ = zJ;
    csr_to_csc(h->nC, h->nV, q.rp, q.ci, h->Ap, h->Ai, q.q2c);
    h->Aorder.assign(z, 0); h->Asrc.assign(z, -1); h->A_init.assign(z, 0.0);
    for (int i = 0; i < z; i++) {
        h->Aorder[i] = q.q2c[q.order[i]];
        if (i < zJ) h->Asrc[h->Aorder[i]] = i;
        else h->A_init[h->Aorder[i]] = ev[i];
    }
    int rc = finish_structure_A(h);
    if (!rc) rc = finish_csr_view(h, q);
    return rc ? rc : z;
}

int sqpb200_set_structure_H_csr(sqpb200_handle h, int zH, const int* row1, const int* col1, int is_symmetric) {
    if (!h || zH < 0) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    // entry list of SpHbMat::setStructure(rhs), src/SpHbMat.cpp:296-309
    std::vector<int> er, ec, srct;
    for (int i = 0; i < zH; i++) {
        er.push_back(row1[i]); ec.push_back(col1[i]); srct.push_back(i);
        if (is_symmetric && row1[i] != col1[i]) { er.push_back(col1[i]); ec.push_back(row1[i]); srct.push_back(i); }
    }
    const int z = (int)er.size();
    for (int i = 0; i < z; i++)
        if (er[i] < 1 || er[i] > h->nV || ec[i] < 1 || ec[i] > h->nV) { h->err = "triplet index out of range"; return SQPB200_ERR_INVALID; }
    if (h->nV >= (1 << 21)) { h->err = "matrix too large for packed keys"; return SQPB200_ERR_TOO_LARGE; }
    auto& q = h->qH;
    q.rp.assign(h->nV + 1, 0); q.ci.assign(z, 0); q.order.assign(z, 0);
    int seg[2] = {0, z}, nrow[1] = {h->nV};
    if (z > 0) {  // compressed-row branch (:324-337)
        int rc = run_assembly(h, h->stream, 1, seg, nrow, ec.data(), er.data(), q.rp.data(), q.ci.data(), q.order.data(), nullptr, &h->err);
        h->launches++;
        if (rc) return rc;
    }
    h->zH = z; h->zHt = zH;
    csr_to_csc(h->nV, h->nV, q.rp, q.ci, h->Hp, h->Hi, q.q2c);
    h->Horder.assign(z, 0); h->Hsrc.assign(z, -1);
    for (int i = 0; i < z; i++) { h->Horder[i] = q.q2c[q.order[i]]; h->Hsrc[h->Horder[i]] = srct[i]; }
    int rc = finish_structure_H(h);
    if (!rc) rc = finish_csr_view(h, q);
    return rc ? rc : z;
}

int sqpb200_set_structure_csr(sqpb200_handle h, int which, int nnz, const int* rowptr, const int* colidx) {
    if (!h || nnz < 0 || !rowptr || (nnz > 0 && !colidx) || (which != SQPB200_MAT_A && which != SQPB200_MAT_H)) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    const bool isA = which == SQPB200_MAT_A;
    const int nrow = isA ? h->nC : h->nV;
    if (rowptr[0] != 0 || rowptr[nrow] != nnz) { h->err = "rowptr[0] != 0 or rowptr[nrow] != nnz"; return SQPB200_ERR_INVALID; }
    for (int r = 0; r < nrow; r++)
        if (rowptr[r + 1] < rowptr[r]) { h->err = "rowptr not monotone"; return SQPB200_ERR_INVALID; }
    for (int e = 0; e < nnz; e++)
        if (colidx[e] < 0 || colidx[e] >= h->nV) { h->err = "column index out of range"; return SQPB200_ERR_INVALID; }
    auto& q = isA ? h->qA : h->qH;
    q.rp.assign(rowptr, rowptr + nrow + 1); q.ci.assign(colidx, colidx + nnz); q.order.resize(nnz);
    for (int e = 0; e < nnz; e++) q.order[e] = e;
    int rc;
    if (isA) {
        h->zA = nnz; h->zJ = nnz;
        csr_to_csc(nrow, h->nV, q.rp, q.ci, h->Ap, h->Ai, q.q2c);
        h->Aorder = q.q2c; h->Asrc.assign(nnz, 0); h->A_init.clear();
        for (int e = 0; e < nnz; e++) h->Asrc[q.q2c[e]] = e;
        rc = finish_structure_A(h);
    } else {
        h->zH = nnz; h->zHt = nnz;
        csr_to_csc(nrow, h->nV, q.rp, q.ci, h->Hp, h->Hi, q.q2c);
        h->Horder = q.q2c; h->Hsrc.assign(nnz, 0);
        for (int e = 0; e < nnz; e++) h->Hsrc[q.q2c[e]] = e;
        rc = finish_structure_H(h);
    }
    if (!rc) rc = finish_csr_view(h, q);
    return rc ? rc : nnz;
}

int sqpb200_get_structure_csr(sqpb200_handle h, int which, int* rowptr, int* colidx, int* order) {
    if (!h) return SQPB200_ERR_INVALID;
    const auto& q = which == SQPB200_MAT_A ? h->qA : h->qH;
    if (!q.set) { h->err = "structure was not given in compressed-row form"; return SQPB200_ERR_STATE; }
    if (rowptr) std::copy(q.rp.begin(), q.rp.end(), rowptr);
    if (colidx) std::copy(q.ci.begin(), q.ci.end(), colidx);
    if (order) std::copy(q.order.begin(), q.order.end(), order);
    return 0;
}

int sqpb200_set_values_csr(sqpb200_handle h, int which, const double* vals, int loc, int broadcast) {
    if (!h || !vals) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    const bool isA = which == SQPB200_MAT_A;
    const auto& q = isA ? h->qA : h->qH;
    if (!q.set || (isA ? !h->A_set : !h->H_set)) { h->err = "structure was not given in compressed-row form"; return SQPB200_ERR_STATE; }
    const int z = isA ? h->zA : h->zH;
    if (z > 0) {
        const size_t bytes = (size_t)(broadcast ? 1 : h->batch) * z * 8;
        if (loc == SQPB200_LOC_HOST && ensure_stage(h, bytes)) return SQPB200_ERR_CUDA;
        const void* din;
        if (to_device(h, vals, bytes, loc, 0, &din)) return SQPB200_ERR_CUDA;
        const long long total = (long long)h->batch * z;
        // out[b][compressed-column position] = in[b][c2q[position]]
        scatter_values_kernel<<<grid_for(total, 256), 256, 0, h->stream>>>(total, z, z, q.dc2q, (const double*)din, broadcast,
                                                                           isA ? h->dAval : h->dHval);
        h->launches++;
        CK(cudaGetLastError());
    }
    if (h->first_solved) { if (isA) h->upd_A = true; else h->upd_H = true; }
    return 0;
}

int sqpb200_get_values_csr(sqpb200_handle h, int which, double* vals, int loc) {
    if (!h || !vals) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    const bool isA = which == SQPB200_MAT_A;
    const auto& q = isA ? h->qA : h->qH;
    if (!q.set) { h->err = "structure was not given in compressed-row form"; return SQPB200_ERR_STATE; }
    const int z = isA ? h->zA : h->zH;
    if (z == 0) return 0;
    const size_t bytes = (size_t)h->batch * z * 8;
    double* dout = vals;
    if (loc == SQPB200_LOC_HOST) { if (ensure_stage(h, bytes)) return SQPB200_ERR_CUDA; dout = (double*)h->stage; }
    const long long total = (long long)h->batch * z;
    scatter_values_kernel<<<grid_for(total, 256), 256, 0, h->stream>>>(total, z, z, q.dq2c, isA ? h->dAval : h->dHval, 0, dout);
    h->launches++;
    CK(cudaGetLastError());
    if (loc == SQPB200_LOC_HOST) CK(cudaMemcpyAsync(vals, dout, bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int sqpb200_set_bounds_stacked(sqpb200_handle h, const double* lb, const double* ub, int loc, int broadcast) {
    if (!h) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    const int nV = h->nV, nC = h->nC;
    const size_t ld = (size_t)(nV + nC) * 8;
    const cudaMemcpyKind kind = loc == SQPB200_LOC_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    const double* src[2] = {lb, ub};
    double* dx[2] = {h->dlb, h->dub};
    double* dc[2] = {h->dlbA, h->dubA};
    const int wx[2] = {SQPB200_VEC_LB, SQPB200_VEC_UB}, wc[2] = {SQPB200_VEC_LBA, SQPB200_VEC_UBA};
    for (int k = 0; k < 2; k++) {
        if (!src[k]) continue;
        if (broadcast) {  // one row for every instance: the broadcast path of the split setters
            int rc = sqpb200_set_vectors(h, wx[k], src[k], 0, nV, loc, 1);
            if (!rc && nC > 0) rc = sqpb200_set_vectors(h, wc[k], src[k] + nV, 0, nC, loc, 1);
            if (rc) return rc;
        } else {  // two strided DMA copies per vector: rows of nV + nC doubles split at nV
            CK(cudaMemcpy2DAsync(dx[k], (size_t)nV * 8, src[k], ld, (size_t)nV * 8, h->batch, kind, h->stream));
            if (nC > 0) CK(cudaMemcpy2DAsync(dc[k], (size_t)nC * 8, src[k] + nV, ld, (size_t)nC * 8, h->batch, kind, h->stream));
        }
    }
    if (h->first_solved && (lb || ub)) h->upd_bounds = true;  // Update_bounds, as the per-entry setters raise it
    return 0;
}

int sqpb200_get_bounds_stacked(sqpb200_handle h, double* lb, double* ub, int loc) {
    if (!h) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    const int nV = h->nV, nC = h->nC;
    const size_t ld = (size_t)(nV + nC) * 8;
    const cudaMemcpyKind kind = loc == SQPB200_LOC_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    double* dst[2] = {lb, ub};
    const double* dx[2] = {h->dlb, h->dub};
    const double* dc[2] = {h->dlbA, h->dubA};
    for (int k = 0; k < 2; k++) {
        if (!dst[k]) continue;
        CK(cudaMemcpy2DAsync(dst[k], ld, dx[k], (size_t)nV * 8, (size_t)nV * 8, h->batch, kind, h->stream));
        if (nC > 0) CK(cudaMemcpy2DAsync(dst[k] + nV, ld, dc[k], (size_t)nC * 8, (size_t)nC * 8, h->batch, kind, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int sqpb200_get_solution_stacked(sqpb200_handle h, double* primal, double* dual, int* workingset, int loc) {
    if (!h) return SQPB200_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    const int nV = h->nV, nC = h->nC;
    const size_t B = h->batch, ld = (size_t)(nV + nC);
    const cudaMemcpyKind kind = loc == SQPB200_LOC_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    const size_t ax_bytes = ((B * nC * 8 + 255) / 256) * 256, need = ax_bytes + B * ld * 4 + 256;
    if (need > h->qscratch_bytes) {
        if (h->qscratch) { CK(cudaStreamSynchronize(h->stream)); CK(cudaFree(h->qscratch)); h->qscratch = nullptr; h->qscratch_bytes = 0; }
        CK(cudaMalloc(&h->qscratch, need));
        h->qscratch_bytes = need;
    }
    double* dAx = (double*)h->qscratch;
    int* dws = (int*)((char*)h->qscratch + ax_bytes);
    if (primal) {  // "primalsol" = [x ; A x] (src/QOREInterface.cpp:120; its test_optimality reads x_qp_(nV + i) as the activity)
        CK(cudaMemcpy2DAsync(primal, ld * 8, h->dx, (size_t)nV * 8, (size_t)nV * 8, B, kind, h->stream));
        if (nC > 0) {
            if (!h->A_set) { h->err = "structure of A not set"; return SQPB200_ERR_STATE; }
            int rc = sqpb200_spmv(h, SQPB200_MAT_A, 0, h->dx, dAx, SQPB200_LOC_DEVICE);
            if (rc) return rc;
            CK(cudaMemcpy2DAsync(primal + nV, ld * 8, dAx, (size_t)nC * 8, (size_t)nC * 8, B, kind, h->stream));
        }
    }
    if (copy_out(h, dual, h->dy, B * ld * 8, loc)) return SQPB200_ERR_CUDA;  // "dualsol": already stacked (:303-305 of the qpOASES twin)
    if (workingset) {
        const long long total = (long long)(B * ld);
        qore_workingset_kernel<<<grid_for(total, 256), 256, 0, h->stream>>>(total, nV, nC, h->dwsB, h->dwsC, dws);
        h->launches++;
        CK(cudaGetLastError());
        if (copy_out(h, workingset, dws, B * ld * 4, loc)) return SQPB200_ERR_CUDA;
    }
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}
