// mega_decode.cu -- instantiation, launch and load-time stream builder of the persistent decode kernel.
#include "mega_decode.cuh"

namespace blk {

size_t mega_smem_bytes(const MegaParams& P) {
    size_t b = (size_t)MG_WARPS * MG_SLOTS * P.slot_bytes;
    b += MG_WARPS * MG_SLOTS * 8;
    b += 2 * sizeof(MegaPhase);
    b += 2 * (size_t)P.n_layer * sizeof(void*);
    b += (size_t)P.max_items * MG_WARPS * sizeof(float2);
    b += (size_t)(P.d_head / 2) * sizeof(float2);
    b += 8 * MG_WARPS * sizeof(double);
    b += 32 * sizeof(float);
    b += 32 * sizeof(int);
    b += (size_t)P.act_bytes;
    return b;
}

cudaError_t mega_setup(size_t smem, int* limit) {
    int dev = 0, lim = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&lim, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) return e;
    if (limit) *limit = lim;
    if (smem > (size_t)lim) return cudaErrorInvalidValue;
    e = cudaFuncSetAttribute(mega_decode_kernel<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(mega_decode_kernel<8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(mega_decode_kernel<4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(mega_decode_kernel<8, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}

cudaError_t mega_launch(const MegaParams& P, size_t smem, cudaStream_t st) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)P.n_cta); cfg.blockDim = dim3(MG_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    // GQ = compile-time bound on the query heads per KV head (attention register arrays)
    const bool g4 = P.n_head / P.n_head_kv <= 4;
    if (P.trace) return g4 ? cudaLaunchKernelEx(&cfg, mega_decode_kernel<4, true>, P) : cudaLaunchKernelEx(&cfg, mega_decode_kernel<8, true>, P);
    return g4 ? cudaLaunchKernelEx(&cfg, mega_decode_kernel<4, false>, P) : cudaLaunchKernelEx(&cfg, mega_decode_kernel<8, false>, P);
}

cudaError_t mega_chunk_lists(const MegaPhase* d_phases, int n_phases, int n_cta, uint4* list, int list_stride, int* counts, cudaStream_t st) {
    const int total = n_cta * MG_WARPS;
    mg_chunk_list_kernel<<<(total + 127) / 128, 128, 0, st>>>(d_phases, n_phases, n_cta, list, list_stride, counts);
    return cudaGetLastError();
}

// one thread per (row, super-block)
__global__ void mg_build_stream_kernel(const uint8_t* __restrict__ raw, uint8_t* __restrict__ base, int type, int N, int nsb, int W, int sbs,
                                       int slice_bytes, int rowmap, int d_head, int ab_fixed) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)N * nsb) return;
    const int r = (int)(idx / nsb), s = (int)(idx % nsb);
    int p, ab;
    if (rowmap == 2) { p = r; ab = ab_fixed; }
    else if (rowmap == 1) { const int hd = d_head >> 1, head = r / d_head, i = r % d_head; ab = i / hd; p = head * hd + (i % hd); }
    else { p = r >> 1; ab = r & 1; }
    const int ws = s / sbs, si = s % sbs;
    uint8_t* dst = base + (((size_t)p * W + ws) * 2 + ab) * (size_t)slice_bytes;
    if (type == QT_Q4_K || type == QT_Q5_K) {
        const int bb = type == QT_Q4_K ? 144 : 176;
        const uint8_t* src = raw + idx * bb;
        uint8_t* d = dst + (size_t)si * bb;
        for (int i = 0; i < bb; i++) d[i] = src[i];
    } else if (type == QT_Q6_K) {
        const uint8_t* src = raw + idx * 210;
        uint8_t* d = dst + (size_t)si * 208;
        for (int i = 0; i < 208; i++) d[i] = src[i];
        uint8_t* dd = dst + (size_t)sbs * 208 + si * 2;
        dd[0] = src[208]; dd[1] = src[209];
    } else if (type == QT_Q8_0) {
        const uint8_t* src = raw + idx * (8 * 34);
        uint8_t* d = dst + (size_t)si * 272;
        for (int b = 0; b < 8; b++) {
            d[256 + 2 * b] = src[b * 34]; d[256 + 2 * b + 1] = src[b * 34 + 1];
            for (int i = 0; i < 32; i++) d[b * 32 + i] = src[b * 34 + 2 + i];
        }
    }
}

cudaError_t mega_build_stream(const uint8_t* raw, uint8_t* base, int type, int N, int K, int W, int sbs, int slice_bytes,
                              int rowmap, int d_head, int ab, cudaStream_t st) {
    const int nsb = K / 256;
    const int64_t total = (int64_t)N * nsb;
    const int threads = 128;
    mg_build_stream_kernel<<<(unsigned)((total + threads - 1) / threads), threads, 0, st>>>(raw, base, type, N, nsb, W, sbs, slice_bytes, rowmap, d_head, ab);
    return cudaGetLastError();
}

} // namespace blk
