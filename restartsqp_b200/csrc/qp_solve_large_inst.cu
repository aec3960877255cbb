// qp_solve_large_inst.cu -- instantiation of qp_solve_large_kernel<CTA_THREADS>: one QP per CTA (or per thread-block cluster), the
// slice (vectors and the nV x nV factors) in global memory.  Used when a QP does not fit the shared-memory resident warp kernel.
#include "qp_kernel.cuh"

namespace sqpb200 {
constexpr int CTA_THREADS = 512;  // threads per CTA: the DMMA tile mapping (QPT::mma_tile) assumes 16 warps

// CTAs per QP: the largest power of two <= 16 that keeps batch * cluster <= SM count, so that a batch smaller than the GPU still
// fills it (16 is a non-portable cluster size: opt-in attribute, and a fall-back to 8 if the launch is refused).
static int cluster_for_batch(int batch, int nV) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // Every shared primitive costs two cluster barriers, and since R is carried through additions the refactorisation (the
    // one phase that scales with the CTA count) is rare.  Measured (ms; CTAs per QP in brackets): nV = 128 x 8: 8.5 [1], 8.5 [2],
    // 9.7 [4]; nV = 512 x 16: 92 [1], 91 [2], 87 [4], 161 [8]; nV = 1024 x 16: 371 [2], 326 [4], 546 [8]; nV = 2048 x 16:
    // 2854 [2], 2330 [4], 3263 [8]; nV = 4096 x 4: 13312 [4], 11548 [8], 10817 [16] (non-portable size).
    const int cap = nV < 64 ? 1 : (nV <= 256 ? 2 : (nV <= 2048 ? 4 : (nV <= 3072 ? 8 : 16)));
    int cs = 1;
    while (cs < cap && (long long)batch * cs * 2 <= sms) cs *= 2;  // 16 = non-portable cluster size (opt-in below), batch <= 9
    return cs;
}

cudaError_t launch_qp_solve_large(const QPKernelArgs& a, cudaStream_t stream) {
    int cs = cluster_for_batch(a.batch, a.nV);
    const size_t smem = (size_t)QPT<CTA_THREADS>::LS_TOTAL * sizeof(double);
    cudaError_t e = cudaFuncSetAttribute(qp_solve_large_kernel<CTA_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    if (cs > 8) {
        e = cudaFuncSetAttribute(qp_solve_large_kernel<CTA_THREADS>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        if (e != cudaSuccess) return e;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)a.batch * cs);
    cfg.blockDim = dim3(CTA_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cs; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, qp_solve_large_kernel<CTA_THREADS>, a);
    if (e != cudaSuccess && cs > 8) {  // non-portable size refused on this device / partition: portable maximum
        (void)cudaGetLastError();
        cs = 8;
        cfg.gridDim = dim3((unsigned)a.batch * cs);
        attr[0].val.clusterDim.x = cs;
        e = cudaLaunchKernelEx(&cfg, qp_solve_large_kernel<CTA_THREADS>, a);
    }
    return e;
}
}  // namespace sqpb200
