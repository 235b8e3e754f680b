// clipk - C ABI implementation (see include/clipk.h).  sm_100a only; no CPU path, no other backend.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <atomic>
#include <mutex>
#include <type_traits>
#include <vector>

#include "../../include/clipk.h"
#include "gemm_core.cuh"

namespace clipk {

// ------------------------------------------------------------------------------------------------ errors
static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};   // kernels launched by this library (clipk_launch_count)

// Optional per-kernel timing (clipk_profile_begin / clipk_profile_end, used by bench.py for the roofline of the dominant
// kernel): while it is on, every launch of this library is followed by an event on its stream; the time between two
// consecutive events is attributed to the kernel launched in between.  One stream, one thread at a time.
struct ProfEntry { const char* name; cudaEvent_t ev; };
static std::vector<ProfEntry> g_prof;
static std::atomic<int> g_prof_on{0};
static void count_launch(const char* name, cudaStream_t st) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (g_prof_on.load(std::memory_order_relaxed)) {
        cudaEvent_t ev;
        if (cudaEventCreate(&ev) == cudaSuccess) {
            cudaEventRecord(ev, st);
            g_prof.push_back(ProfEntry{name, ev});
        }
    }
}

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CK_CUDA(expr)                                                                             \
    do {                                                                                          \
        cudaError_t e__ = (expr);                                                                 \
        if (e__ != cudaSuccess) return fail(int(e__), "%s: %s", #expr, cudaGetErrorString(e__));  \
    } while (0)

// ------------------------------------------------------------------------------------------------ device info
struct DevInfo {
    int ok = 0;       // 1 = CC 10.x
    int sms = 0;
    int queried = 0;
};
static DevInfo g_dev[64];
static std::mutex g_dev_mu;

static int device_info(DevInfo* out) {
    int dev = 0;
    CK_CUDA(cudaGetDevice(&dev));
    // The driver-API tensor-map encoder needs the device's primary context CURRENT on the calling thread.  PyTorch's
    // autograd worker threads only have the device selected: until the first runtime call that touches the context
    // (a launch, a memset) cuTensorMapEncodeTiled fails there with CUDA_ERROR_INVALID_CONTEXT.  Bind it once per thread
    // and device.
    static thread_local int bound_dev = -1;
    if (bound_dev != dev) {
        CK_CUDA(cudaFree(nullptr));
        bound_dev = dev;
    }
    if (dev < 0 || dev >= 64) return fail(CLIPK_EINVAL, "device index %d out of range", dev);
    std::lock_guard<std::mutex> lk(g_dev_mu);
    if (!g_dev[dev].queried) {
        int major = 0, sms = 0;
        CK_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
        CK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        g_dev[dev].ok = (major == 10);
        g_dev[dev].sms = sms;
        g_dev[dev].queried = 1;
    }
    *out = g_dev[dev];
    if (!out->ok) return fail(CLIPK_EARCH, "device %d is not compute capability 10.x (B200 / sm_100a required)", dev);
    return CLIPK_OK;
}

// ------------------------------------------------------------------------------------------------ TMA descriptors
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static std::once_flag g_encode_once;

static EncodeTiledFn encode_fn() {
    std::call_once(g_encode_once, [] {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            g_encode = reinterpret_cast<EncodeTiledFn>(fn);
    });
    return g_encode;
}

// 2D tensor map, SWIZZLE_128B, zero fill out of bounds.  inner = contiguous extent (elements of esize bytes).
static int make_tmap(CUtensorMap* m, const void* base, long long inner, long long outer, long long ld_elems,
                     int box_inner, int box_outer, int esize, int swizzle_bytes = 128) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return fail(CLIPK_EDRIVER, "cuTensorMapEncodeTiled entry point not available");
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return fail(CLIPK_EINVAL, "operand pointer not 16-byte aligned");
    if ((ld_elems * esize) % 16 != 0) return fail(CLIPK_EINVAL, "leading dimension %lld is not a multiple of 16 bytes", ld_elems);
    cuuint64_t dims[2] = {cuuint64_t(inner), cuuint64_t(outer)};
    cuuint64_t strides[1] = {cuuint64_t(ld_elems) * esize};
    cuuint32_t box[2] = {cuuint32_t(box_inner), cuuint32_t(box_outer)};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(m, esize == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                    const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(CLIPK_EDRIVER, "cuTensorMapEncodeTiled failed with CUresult %d", int(r));
    return CLIPK_OK;
}
static int make_tmap_bf16(CUtensorMap* m, const void* base, long long inner, long long outer, long long ld_elems,
                          int box_inner, int box_outer) {
    return make_tmap(m, base, inner, outer, ld_elems, box_inner, box_outer, 2);
}
// epilogue stores: fp32 output tile pieces of 32 columns x 32 rows, fp16 G tile pieces of 64 columns x 32 rows
static int tmap_out_f32(CUtensorMap* m, const float* base, long long rows, long long cols, long long ld) {
    return make_tmap(m, base, cols, rows, ld, 32, 32, 4);
}
static int tmap_g_store(CUtensorMap* m, const void* base, long long rows, long long cols, long long ld) {
    return make_tmap(m, base, cols, rows, ld, 64, 32, 2);
}
// the A-resident recompute kernel stores 32 columns x 32 rows from 64-byte rows in SWIZZLE_64B order (conflict-free
// 16-byte stores of one row per lane; plain 64-byte rows put 32 lanes on 8 banks: 78 % of that kernel's shared-memory
// wavefronts were bank-conflict replays, profiles/r02b)
static int tmap_g_store_dense32(CUtensorMap* m, const void* base, long long rows, long long cols, long long ld) {
    return make_tmap(m, base, cols, rows, ld, 32, 32, 2, 64);
}
// operand [rows, K] row-major, consumed K-major: box = 64 (K) x box_rows
static int tmap_kmajor(CUtensorMap* m, const void* base, long long rows, long long K, long long ld, int box_rows) {
    return make_tmap_bf16(m, base, K, rows, ld, BK, box_rows);
}
// operand stored [K, mn] row-major (mn contiguous), consumed MN-major: box = 64 (mn) x 64 (K)
static int tmap_mnmajor(CUtensorMap* m, const void* base, long long mn, long long K, long long ld) {
    return make_tmap_bf16(m, base, mn, K, ld, 64, BK);
}

// ------------------------------------------------------------------------------------------------ small kernels
// merge the per-unit partial row statistics (log2-scaled domain) into natural-log (max, sum, dot):
//   row_max = max_j S_ij,  row_sum = sum_j exp(S_ij - row_max),  row_dot = sum_j exp(S_ij - row_max) * S_ij
__global__ void merge_row_parts_kernel(const float* __restrict__ part_max, const float* __restrict__ part_sum,
                                       const float* __restrict__ part_dot, int nparts, int rows,
                                       float* __restrict__ row_max, float* __restrict__ row_sum,
                                       float* __restrict__ row_dot) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows) return;
    float m = -CUDART_INF_F;
    for (int p = 0; p < nparts; ++p) m = fmaxf(m, part_max[(size_t)p * rows + i]);
    float l = 0.f, t = 0.f;
    for (int p = 0; p < nparts; ++p) {
        const float pm = part_max[(size_t)p * rows + i];
        if (pm > -CUDART_INF_F) {
            const float w = exp2f(pm - m);
            l += part_sum[(size_t)p * rows + i] * w;
            t += part_dot[(size_t)p * rows + i] * w;
        }
    }
    row_max[i] = m * LN2;
    row_sum[i] = l;
    row_dot[i] = t * LN2;
}

// column j: merge nparts (max, sum, dot) triples -> (lse, expected logit under the column softmax)
__device__ __forceinline__ void merge_col(const float* __restrict__ cmax, const float* __restrict__ csum,
                                          const float* __restrict__ cdot, int nparts, long long stride, long long j,
                                          float* lse, float* expect) {
    float m = -CUDART_INF_F;
    for (int p = 0; p < nparts; ++p) m = fmaxf(m, cmax[(size_t)p * stride + j]);
    float l = 0.f, t = 0.f;
    for (int p = 0; p < nparts; ++p) {
        const float pm = cmax[(size_t)p * stride + j];
        if (pm > -CUDART_INF_F) {
            const float w = expf(pm - m);
            l += csum[(size_t)p * stride + j] * w;
            t += cdot[(size_t)p * stride + j] * w;
        }
    }
    *lse = m + logf(l);
    *expect = t / l;
}

// sums[0] = sum_i (lse_row_i - pos_i)          sums[1] = sum_i (lse_col_{off+i} - pos_i)        (cross-entropy sums)
// sums[2] = sum_i (E_row_i - pos_i)            sums[3] = sum_i (E_col_{off+i} - pos_i)          (s * dloss/ds sums)
// with E = expected logit under the row / column softmax.
__global__ void finalize_kernel(const float* __restrict__ row_max, const float* __restrict__ row_sum,
                                const float* __restrict__ row_dot, const float* __restrict__ pos, int rows,
                                const float* __restrict__ cmax, const float* __restrict__ csum,
                                const float* __restrict__ cdot, int nparts, long long stride, int cols,
                                long long diag_offset, float* __restrict__ lse_row, float* __restrict__ lse_col,
                                float* __restrict__ sums, int* __restrict__ mm, float loss_div) {
    // mm != null (clipk_step_forward): sums is the step's scalar block - [0..3] the sums, [4..5] receive (CE sums) /
    // loss_div and (dscale sums) / loss_div from the last block to finish, [6] is its ticket, mm = ints [8..9].
    // (one block preparing the recompute's per-row / per-column factors here as well was measured: +37 us for 40K
    //  entries - they stay with grad_prep_kernel in the backward)
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    int lo = 0x7fffffff, hi = int(0x80000000);       // min / max LSE of this thread (ordered ints), for grad_prep_kernel
    if (i < cols) {
        float lse, e;
        merge_col(cmax, csum, cdot, nparts, stride, i, &lse, &e);
        lse_col[i] = lse;
        lo = hi = float_to_ordered(lse);
    }
    if (i < rows) {
        const float rs = row_sum[i];
        const float lr = row_max[i] + logf(rs);
        lse_row[i] = lr;
        lo = min(lo, float_to_ordered(lr));
        hi = max(hi, float_to_ordered(lr));
        const float p = pos[i];
        v[0] = lr - p;
        v[2] = row_dot[i] / rs - p;
        const long long j = diag_offset + i;
        if (j >= 0 && j < cols) {
            float lse, e;
            merge_col(cmax, csum, cdot, nparts, stride, j, &lse, &e);
            v[1] = lse - p;
            v[3] = e - p;
        }
    }
    __shared__ float sh[4][32];
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (mm) {
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, off));
            hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, off));
        }
        if (l == 0) {
            if (lo < __ldcg(mm)) atomicMin(mm, lo);
            if (hi > __ldcg(mm + 1)) atomicMax(mm + 1, hi);
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], off);
        if (l == 0) sh[k][w] = v[k];
    }
    __syncthreads();
    if (w == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float x = (l < (blockDim.x >> 5)) ? sh[k][l] : 0.f;
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
            if (l == 0) atomicAdd(sums + k, x);
        }
    }
    if (!mm) return;
    __shared__ int last_block;
    __syncthreads();                                  // every warp's lse stores and atomics are issued
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned int ticket = atomicAdd(reinterpret_cast<unsigned int*>(sums) + 6, 1u);
        last_block = (ticket == gridDim.x - 1);
        if (last_block) {
            __threadfence();
            sums[4] = (__ldcg(sums) + __ldcg(sums + 1)) / loss_div;
            sums[5] = (__ldcg(sums + 2) + __ldcg(sums + 3)) / loss_div;
        }
    }
    __syncthreads();
}

// ---- backward preparation: one reference for every exponential of this backward (see grad_chunk PATH 0)

// mm[0] = min, mm[1] = max (ordered-int encoding) over both LSE vectors
__global__ void lse_minmax_kernel(const float* __restrict__ a, int na, const float* __restrict__ b, int nb, int* mm) {
    int lo = 0x7fffffff, hi = int(0x80000000);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < na + nb; i += gridDim.x * blockDim.x) {
        const int v = float_to_ordered(i < na ? a[i] : b[i - na]);
        lo = min(lo, v);
        hi = max(hi, v);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, off));
        hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, off));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin(mm, lo);
        atomicMax(mm + 1, hi);
    }
}

// c = min LSE (log2 units); avec[i] = 2^(c - Lr_i), bvec[j] = 2^(c - Lc_j); gref = {c, fast flag}
__global__ void grad_prep_kernel(const float* __restrict__ lse_row, int rows, const float* __restrict__ lse_col, int cols,
                                 const int* __restrict__ mm, float* __restrict__ avec, float* __restrict__ bvec,
                                 float* __restrict__ gref) {
    const float lo = ordered_to_float(mm[0]) * LOG2E, hi = ordered_to_float(mm[1]) * LOG2E;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {
        gref[0] = lo;
        gref[1] = (hi - lo <= 100.f && lo > -CUDART_INF_F && hi < CUDART_INF_F) ? 1.f : 0.f;
    }
    if (i < rows) avec[i] = exp2f(lo - lse_row[i] * LOG2E);
    if (i < cols) bvec[i] = exp2f(lo - lse_col[i] * LOG2E);
}

__global__ void cast_kernel(const float* __restrict__ src, void* __restrict__ dst, long long n, int dtype) {
    const long long i = (long long)(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long base = i * 4;
    if (base >= n) return;
    if (base + 4 <= n && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
        const float4 v = *reinterpret_cast<const float4*>(src + base);
        if (dtype == CLIPK_BF16) {
            uint2 o = make_uint2(ptx::pack_bf16x2(v.x, v.y), ptx::pack_bf16x2(v.z, v.w));
            *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(dst) + base) = o;
        } else {
            *reinterpret_cast<float4*>(reinterpret_cast<float*>(dst) + base) = v;
        }
    } else {
        for (long long k = base; k < n && k < base + 4; ++k) {
            if (dtype == CLIPK_BF16) reinterpret_cast<__nv_bfloat16*>(dst)[k] = __float2bfloat16(src[k]);
            else reinterpret_cast<float*>(dst)[k] = src[k];
        }
    }
}

// |x| maximum of a [rows, d] matrix as the bit pattern of a non-negative float (monotonic under integer max).
// One thread handles 8 consecutive elements of a row (d % 8 == 0): 16-byte loads for bf16, 2 x 16 bytes for fp32.
template <typename T>
__device__ __forceinline__ void load8(const T* p, float (&v)[8]);
template <>
__device__ __forceinline__ void load8<__nv_bfloat16>(const __nv_bfloat16* p, float (&v)[8]) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        v[2 * i] = __uint_as_float(w[i] << 16);
        v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
}
template <>
__device__ __forceinline__ void load8<float>(const float* p, float (&v)[8]) {
    const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

template <typename T>
__global__ void amax_kernel(const T* __restrict__ src, long long rows, long long d8, long long ld,
                            unsigned int* __restrict__ amax_bits) {
    float m = 0.f;
    const long long n = rows * d8;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / d8, k = (i - r * d8) * 8;
        float v[8];
        load8(src + r * ld + k, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float a = fabsf(v[j]);
            if (a < CUDART_INF_F) m = fmaxf(m, a);
        }
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
    if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(amax_bits, __float_as_uint(m));
}

// [rows, d] bf16 / fp32  ->  scaled fp16 planes laid side by side (plane width dpad, zero padded):
//   planes = 1:  dst = fp16(x * 2^e)                      exact for bf16 sources (8 significant bits fit in 11)
//   planes = 2:  dst = [hi | lo], hi + lo = x * 2^e to 22 bits
// 2^e maps the largest |x| into [2^13, 2^14), so entries down to 2^-28 of the maximum stay normal fp16 numbers.
// scale_io[0] holds the amax bits on entry; scale_io[1] receives 2^-e (true value = stored * scale_io[1]).
// One thread converts 8 consecutive elements (16-byte stores).
template <typename T>
__global__ void to_f16_kernel(const T* __restrict__ src, __half* __restrict__ dst, long long rows, long long d,
                              long long ld_src, long long dpad, int planes, float* __restrict__ scale_io) {
    const float amax = scale_io[0];
    int ex = 0;
    float scale = 1.f;
    if (amax > 0.f && amax < CUDART_INF_F) {
        frexpf(amax, &ex);                 // amax = m * 2^ex, m in [0.5, 1)
        int e = 14 - ex;
        e = e > 120 ? 120 : (e < -120 ? -120 : e);
        scale = ldexpf(1.f, e);
    }
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx == 0) scale_io[1] = 1.f / scale;
    const long long dp8 = dpad / 8;
    if (idx >= rows * dp8) return;
    const long long r = idx / dp8, k = (idx - r * dp8) * 8;
    float v[8];
    if (k < d) {
        load8(src + r * ld_src + k, v);     // d % 8 == 0, so a group of 8 is either all inside or all padding
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = 0.f;
    }
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float x0 = v[2 * j] * scale, x1 = v[2 * j + 1] * scale;
        hi[j] = ptx::pack_f16x2(x0, x1);
        if (planes == 2) {
            const float h0 = __half2float(__ushort_as_half((unsigned short)(hi[j] & 0xffffu)));
            const float h1 = __half2float(__ushort_as_half((unsigned short)(hi[j] >> 16)));
            lo[j] = ptx::pack_f16x2(x0 - h0, x1 - h1);
        }
    }
    __half* o = dst + r * (planes * dpad) + k;
    *reinterpret_cast<uint4*>(o) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    if (planes == 2) *reinterpret_cast<uint4*>(o + dpad) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}

// ---- L2 normalisation of the embeddings (the F.normalize calls that feed the loss: open_clip/model.py:216,231)
template <typename T>
__device__ __forceinline__ void store8(T* p, const float (&v)[8]);
template <>
__device__ __forceinline__ void store8<__nv_bfloat16>(__nv_bfloat16* p, const float (&v)[8]) {
    *reinterpret_cast<uint4*>(p) = make_uint4(ptx::pack_bf16x2(v[0], v[1]), ptx::pack_bf16x2(v[2], v[3]),
                                              ptx::pack_bf16x2(v[4], v[5]), ptx::pack_bf16x2(v[6], v[7]));
}
template <>
__device__ __forceinline__ void store8<float>(float* p, const float (&v)[8]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}

// y = x / max(|x|, eps) per row, inv[row] = 1 / max(|x|, eps).  One warp per row, 8 elements per lane and step.
template <typename T>
__global__ void normalize_fwd_kernel(const T* __restrict__ x, long long rows, int d8, long long ldx, T* __restrict__ y,
                                     long long ldy, float* __restrict__ inv, float eps) {
    const int lane = threadIdx.x & 31;
    const long long r = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= rows) return;
    float ss = 0.f;
    for (int k = lane; k < d8; k += 32) {
        float v[8];
        load8(x + r * ldx + (long long)k * 8, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) ss = fmaf(v[j], v[j], ss);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
    const float scale = 1.f / fmaxf(sqrtf(ss), eps);
    if (lane == 0) inv[r] = scale;
    for (int k = lane; k < d8; k += 32) {
        float v[8];
        load8(x + r * ldx + (long long)k * 8, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] *= scale;
        store8(y + r * ldy + (long long)k * 8, v);
    }
}

// dx = (g - y * (y . g)) * inv for rows with |x| >= eps (y = x * inv is then a unit vector), dx = g * inv otherwise
template <typename T>
__global__ void normalize_bwd_kernel(const T* __restrict__ g, long long ldg, const T* __restrict__ y, long long ldy,
                                     const float* __restrict__ inv, long long rows, int d8, T* __restrict__ dx,
                                     long long ldd, float eps) {
    const int lane = threadIdx.x & 31;
    const long long r = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= rows) return;
    float dot = 0.f;
    for (int k = lane; k < d8; k += 32) {
        float a[8], b[8];
        load8(g + r * ldg + (long long)k * 8, a);
        load8(y + r * ldy + (long long)k * 8, b);
#pragma unroll
        for (int j = 0; j < 8; ++j) dot = fmaf(a[j], b[j], dot);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, off);
    const float scale = inv[r];
    if (scale >= 1.f / eps * 0.999999f) dot = 0.f;      // |x| < eps: y = x / eps, a plain scaling
    for (int k = lane; k < d8; k += 32) {
        float a[8], b[8];
        load8(g + r * ldg + (long long)k * 8, a);
        load8(y + r * ldy + (long long)k * 8, b);
#pragma unroll
        for (int j = 0; j < 8; ++j) a[j] = (a[j] - b[j] * dot) * scale;
        store8(dx + r * ldd + (long long)k * 8, a);
    }
}

// ---- forward sweep helpers
// Operand preparation: ONE pass over the rows of both feature matrices (open_clip/model.py:216,231 + the casts that
// precede loss.py:112-119) that leaves
//   * the statistics the kernels steer by (OperandStats, gemm_core.cuh): max |x_i|^2 and max |y_j|^2 (bound of the single
//     sweep), max |element| of both (scale of the fp16 copies the gradient GEMMs read), min_i x_i . y_i over the positive
//     pairs (keeps the single sweep at large logit scales);
//   * optionally the bf16 operands themselves: L2-normalised rows (NORMALIZE, with 1 / max(|row|, eps) per row for the
//     Jacobian in the backward) and / or the cast of fp32 inputs, the text rows going straight into the buffer the
//     all-gather reads.  Statistics are those of the values the tensor cores will see (after rounding to bf16).
// One warp per row pair (x_i, y_i); the partner of x_i in the dot product is y row pair_off + i.
struct PrepArgs {
    const void* x; const void* y;
    long long rows_x, rows_y, ldx, ldy;
    int d8;                        // d / 8
    long long pair_off;
    __nv_bfloat16* x_out; __nv_bfloat16* y_out;    // null = operand not written (bf16 input used in place)
    long long ldxo, ldyo;
    float* inv_x; float* inv_y;    // NORMALIZE
    float eps;
    float* stats;                  // this rank's row of the statistics
    // How the blocks' partial results meet.  ticket == null: atomics on `stats`, which the launcher zeroes first
    // (cudaMemsetAsync: a separate operation on the stream, ~10-30 us of engine switching around a 5 us kernel).
    // ticket != null (the fused step, whose scratch lives across calls): every block leaves its five values in
    // partials[block], takes a ticket, and the LAST block reduces them, writes `stats` and puts the ticket back to 0 -
    // no memset, no atomics on the statistics.  *ticket must be 0 when the scratch is created.
    unsigned int* ticket;
    float* partials;               // [gridDim.x][8]
    float* reset;                  // 8 floats + 2 ints of accumulators of LATER kernels of the step, reset here (null = none)
};

template <typename T>
__device__ __forceinline__ void load8_as_bf16(const T* p, float scale, float (&v)[8]) {
    load8(p, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __bfloat162float(__float2bfloat16_rn(v[j] * scale));
}

template <typename T, bool NORMALIZE>
__global__ void prep_kernel(const PrepArgs a) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    const T* X = static_cast<const T*>(a.x);
    const T* Y = static_cast<const T*>(a.y);
    const long long nmax = a.rows_x > a.rows_y ? a.rows_x : a.rows_y;
    // bf16 inputs used as they are need no rounding; everything else is rounded to the bf16 value the MMA will read
    constexpr bool ROUND = NORMALIZE || !std::is_same<T, __nv_bfloat16>::value;
    if (blockIdx.x == 0 && threadIdx.x == 0 && a.reset) {
#pragma unroll
        for (int k = 0; k < 8; ++k) a.reset[k] = 0.f;
        reinterpret_cast<int*>(a.reset)[8] = 0x7f7f7f7f;          // min LSE (ordered int), see finalize_kernel
        reinterpret_cast<int*>(a.reset)[9] = int(0x80808080);     // max LSE
    }
    float best_x = 0.f, best_y = 0.f, am_x = 0.f, am_y = 0.f, min_pos = CUDART_INF_F;
    bool bad = false;
    for (long long i = (long long)blockIdx.x * wpb + warp; i < nmax; i += (long long)gridDim.x * wpb) {
        const bool hx = i < a.rows_x, hy = i < a.rows_y;
        const long long j = a.pair_off + i;
        const bool hp = hx && j >= 0 && j < a.rows_y;
        const T* xr = X + i * a.ldx;
        const T* yr = Y + i * a.ldy;
        const T* pr = Y + j * a.ldy;
        float sx = 1.f, sy = 1.f;
        if (NORMALIZE) {
            float ssx = 0.f, ssy = 0.f;
            for (int k = lane; k < a.d8; k += 32) {
                float v[8];
                if (hx) { load8(xr + (long long)k * 8, v);
#pragma unroll
                    for (int q = 0; q < 8; ++q) ssx = fmaf(v[q], v[q], ssx); }
                if (hy) { load8(yr + (long long)k * 8, v);
#pragma unroll
                    for (int q = 0; q < 8; ++q) ssy = fmaf(v[q], v[q], ssy); }
            }
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) {
                ssx += __shfl_xor_sync(0xffffffffu, ssx, off);
                ssy += __shfl_xor_sync(0xffffffffu, ssy, off);
            }
            sx = 1.f / fmaxf(sqrtf(ssx), a.eps);
            sy = 1.f / fmaxf(sqrtf(ssy), a.eps);
            if (lane == 0) {
                if (hx) a.inv_x[i] = sx;
                if (hy) a.inv_y[i] = sy;
            }
        }
        float nx = 0.f, ny = 0.f, dot = 0.f;
#pragma unroll 2
        for (int k = lane; k < a.d8; k += 32) {          // two iterations' loads in flight (d = 512: the whole row pair)
            float vx[8], vy[8], vp[8];
            if (hx) {
                if (ROUND) load8_as_bf16(xr + (long long)k * 8, sx, vx); else load8(xr + (long long)k * 8, vx);
                if (a.x_out) store8(a.x_out + i * a.ldxo + (long long)k * 8, vx);
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    nx = fmaf(vx[q], vx[q], nx);
                    const float m = fabsf(vx[q]);
                    if (m < CUDART_INF_F) am_x = fmaxf(am_x, m);
                }
            }
            if (hy) {
                if (ROUND) load8_as_bf16(yr + (long long)k * 8, sy, vy); else load8(yr + (long long)k * 8, vy);
                if (a.y_out) store8(a.y_out + i * a.ldyo + (long long)k * 8, vy);
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    ny = fmaf(vy[q], vy[q], ny);
                    const float m = fabsf(vy[q]);
                    if (m < CUDART_INF_F) am_y = fmaxf(am_y, m);
                }
            }
            if (hp) {
                if (j == i) {
#pragma unroll
                    for (int q = 0; q < 8; ++q) dot = fmaf(vx[q], vy[q], dot);
                } else {            // never with NORMALIZE (the host requires pair_off == 0 there)
                    if (ROUND) load8_as_bf16(pr + (long long)k * 8, 1.f, vp); else load8(pr + (long long)k * 8, vp);
#pragma unroll
                    for (int q = 0; q < 8; ++q) dot = fmaf(vx[q], vp[q], dot);
                }
            }
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            nx += __shfl_xor_sync(0xffffffffu, nx, off);
            ny += __shfl_xor_sync(0xffffffffu, ny, off);
            dot += __shfl_xor_sync(0xffffffffu, dot, off);
        }
        // NaN / Inf propagate into the bound, which then fails its tests (exact mode)
        if (hx) { bad = bad || !(nx == nx); best_x = fmaxf(best_x, nx); }
        if (hy) { bad = bad || !(ny == ny); best_y = fmaxf(best_y, ny); }
        if (hp) min_pos = fminf(min_pos, dot);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        am_x = fmaxf(am_x, __shfl_xor_sync(0xffffffffu, am_x, off));
        am_y = fmaxf(am_y, __shfl_xor_sync(0xffffffffu, am_y, off));
    }
    __shared__ float sh[5][32];
    __shared__ int shbad;
    if (threadIdx.x == 0) shbad = 0;
    __syncthreads();
    if (lane == 0) {
        sh[0][warp] = best_x; sh[1][warp] = best_y; sh[2][warp] = am_x; sh[3][warp] = am_y; sh[4][warp] = min_pos;
        if (bad) shbad = 1;
    }
    __syncthreads();
    if (warp == 0) {
        bool last = false;
        float v[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) v[k] = lane < wpb ? sh[k][lane] : (k == 4 ? CUDART_INF_F : 0.f);
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
#pragma unroll
            for (int k = 0; k < 4; ++k) v[k] = fmaxf(v[k], __shfl_xor_sync(0xffffffffu, v[k], off));
            v[4] = fminf(v[4], __shfl_xor_sync(0xffffffffu, v[4], off));
        }
        if (lane == 0) {
            unsigned int* su = reinterpret_cast<unsigned int*>(a.stats);
            const bool isbad = shbad != 0;
            const unsigned int mine[5] = {isbad ? 0x7f800000u : __float_as_uint(v[0]), isbad ? 0x7f800000u : __float_as_uint(v[1]),
                                          __float_as_uint(v[2]), __float_as_uint(v[3]),
                                          // min over the positives as a max over an order-reversing unsigned code (0 = "no
                                          // pair seen" is its identity); decoded by stat_min_pos (gemm_core.cuh)
                                          ~unsigned(float_to_ordered(v[4]) ^ 0x80000000)};
            if (!a.ticket) {
                // hundreds of blocks hit the same five words: look first, only a block that raises a maximum pays for an atomic
#pragma unroll
                for (int k = 0; k < 5; ++k)
                    if (mine[k] > __ldcg(su + k)) atomicMax(su + k, mine[k]);
            } else {
                unsigned int* part = reinterpret_cast<unsigned int*>(a.partials) + (size_t)blockIdx.x * 8;
#pragma unroll
                for (int k = 0; k < 5; ++k) part[k] = mine[k];
                __threadfence();
                last = atomicAdd(a.ticket, 1u) == gridDim.x - 1;
            }
        }
        last = __shfl_sync(0xffffffffu, last ? 1 : 0, 0) != 0;
        if (last) {
            // the last block to finish: reduce every block's five values (all of them are maxima)
            __threadfence();
            unsigned int best[5] = {0u, 0u, 0u, 0u, 0u};
            const unsigned int* all = reinterpret_cast<const unsigned int*>(a.partials);
            for (unsigned int b = lane; b < gridDim.x; b += 32)
#pragma unroll
                for (int k = 0; k < 5; ++k) best[k] = max(best[k], __ldcg(all + (size_t)b * 8 + k));
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1)
#pragma unroll
                for (int k = 0; k < 5; ++k) best[k] = max(best[k], __shfl_xor_sync(0xffffffffu, best[k], off));
            if (lane == 0) {
                unsigned int* su = reinterpret_cast<unsigned int*>(a.stats);
#pragma unroll
                for (int k = 0; k < 5; ++k) su[k] = best[k];
                su[5] = su[6] = su[7] = 0u;
                *a.ticket = 0u;
            }
        }
    }
}

// Both fp16 copies the gradient GEMMs read, in one launch: Xg = fp16(X * 2^ex) for this rank's rows, Yg = fp16(Y * 2^ey)
// for all gathered rows; exact for bf16 sources (8 significant bits fit in 11).  The scales come from the statistics:
// max |x_ij| of this rank's row of the table, max |y_ij| over every row of it.  inv_out[0 / 1] = 2^-ex / 2^-ey.
__device__ __forceinline__ float f16_scale_of(float amax) {
    if (!(amax > 0.f && amax < CUDART_INF_F)) return 1.f;
    int ex = 0;
    frexpf(amax, &ex);                 // amax = m * 2^ex, m in [0.5, 1)
    int e = 14 - ex;
    e = e > 120 ? 120 : (e < -120 ? -120 : e);
    return ldexpf(1.f, e);
}
__global__ void to_f16_pair_kernel(const __nv_bfloat16* __restrict__ X, long long rows_x, long long ldx, __half* __restrict__ Xg,
                                   const __nv_bfloat16* __restrict__ Y, long long rows_y, long long ldy, __half* __restrict__ Yg,
                                   long long d, long long dpad, const float* __restrict__ stats, int nstat, int stats_rank,
                                   float* __restrict__ inv_out) {
    float ay = 0.f;
    for (int r = 0; r < nstat; ++r) ay = fmaxf(ay, __ldg(stats + r * STAT_WORDS + 3));
    const float sx = f16_scale_of(__ldg(stats + stats_rank * STAT_WORDS + 2)), sy = f16_scale_of(ay);
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx == 0) { inv_out[0] = 1.f / sx; inv_out[1] = 1.f / sy; }
    const long long dp8 = dpad / 8;
    if (idx >= (rows_x + rows_y) * dp8) return;
    const bool second = idx >= rows_x * dp8;
    const long long t = second ? idx - rows_x * dp8 : idx;
    const long long r = t / dp8, k = (t - r * dp8) * 8;
    const __nv_bfloat16* src = (second ? Y + r * ldy : X + r * ldx) + k;
    const float scale = second ? sy : sx;
    float v[8];
    if (k < d) {
        load8(src, v);
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = 0.f;
    }
    uint32_t hi[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) hi[j] = ptx::pack_f16x2(v[2 * j] * scale, v[2 * j + 1] * scale);
    __half* o = (second ? Yg : Xg) + r * dpad + k;
    *reinterpret_cast<uint4*>(o) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
}

// Last pass of the backward, one warp per row of either gradient: sum the per-source slots of the fused reduce-scatter
// (text gradient), apply the Jacobian of the L2 normalisation when the forward normalised (dx = (g - y (y . g)) / |x|,
// with y the operand row), cast to the dtype of the inputs.  Replaces clipk_cast and clipk_normalize_bwd of the
// unfused path and the separate slot sum of round 1.  Thread 0 also finishes dlogit_scale = go * (s dloss/ds) / s.
struct FinishArgs {
    const float* gx; long long rows_x;             // [rows_x, d] fp32 image gradient (null = skip)
    const float* gy; long long rows_y;             // [slots][rows_y, d] fp32 text gradient (null = skip)
    int slots; long long slot_stride;              // elements between slots
    int d8;
    const __nv_bfloat16* xn; const __nv_bfloat16* yn;   // operand rows for the Jacobian (null = no normalisation)
    long long ldxn, ldyn;
    const float* inv_x; const float* inv_y;
    float eps;
    void* out_x; void* out_y; int out_dtype;       // CLIPK_BF16 or CLIPK_F32, [rows, d] contiguous
    const float* pair; const float* go; const float* scale; float* dscale;   // dscale: null = skip
};
__global__ void finish_grad_kernel(const FinishArgs a) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    if (blockIdx.x == 0 && threadIdx.x == 0 && a.dscale) a.dscale[0] = a.pair[1] * a.go[0] / a.scale[0];
    const long long rx = a.gx ? a.rows_x : 0, ry = a.gy ? a.rows_y : 0;
    const long long d = (long long)a.d8 * 8;
    for (long long t = (long long)blockIdx.x * wpb + warp; t < rx + ry; t += (long long)gridDim.x * wpb) {
        const bool second = t >= rx;
        const long long r = second ? t - rx : t;
        const float* g = (second ? a.gy : a.gx) + r * d;
        const int slots = second ? a.slots : 1;
        const __nv_bfloat16* yn = second ? a.yn : a.xn;
        const long long ldn = second ? a.ldyn : a.ldxn;
        auto load_g = [&](int k, float (&v)[8]) {
            load8(g + (long long)k * 8, v);
            for (int w = 1; w < slots; ++w) {
                float u[8];
                load8(g + (long long)w * a.slot_stride + (long long)k * 8, u);
#pragma unroll
                for (int q = 0; q < 8; ++q) v[q] += u[q];
            }
        };
        float dot = 0.f, inv = 1.f;
        if (yn) {
            for (int k = lane; k < a.d8; k += 32) {
                float v[8], y[8];
                load_g(k, v);
                load8(yn + r * ldn + (long long)k * 8, y);
#pragma unroll
                for (int q = 0; q < 8; ++q) dot = fmaf(v[q], y[q], dot);
            }
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, off);
            inv = (second ? a.inv_y : a.inv_x)[r];
            if (inv >= 1.f / a.eps * 0.999999f) dot = 0.f;      // |x| < eps: y = x / eps, a plain scaling
        }
        void* out = second ? a.out_y : a.out_x;
        for (int k = lane; k < a.d8; k += 32) {
            float v[8];
            load_g(k, v);
            if (yn) {
                float y[8];
                load8(yn + r * ldn + (long long)k * 8, y);
#pragma unroll
                for (int q = 0; q < 8; ++q) v[q] = (v[q] - y[q] * dot) * inv;
            }
            if (a.out_dtype == CLIPK_BF16) store8(static_cast<__nv_bfloat16*>(out) + r * d + (long long)k * 8, v);
            else store8(static_cast<float*>(out) + r * d + (long long)k * 8, v);
        }
    }
}

// ---- data-parallel ranks of one NVLink domain: flags, barrier and all-gather over peer-mapped (symmetric) memory --------
// Every rank owns an array of MAX_PEERS flag words per purpose, mapped into all peers.  Rank r publishes epoch e to rank
// t by storing e into word [r] of t's array (release at system scope, after everything the stream did before); t waits
// until word [r] of its own array has reached e.  Epochs only grow (compared modulo 2^32), flags are never reset.
struct PeerPtrs {
    void* p[MAX_PEERS];
};
__device__ __forceinline__ void peer_signal(unsigned int* flag, unsigned int epoch) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flag), "r"(epoch) : "memory");
}
// A wait gives up after ~20 s (a peer died, or skipped the collective call) and leaves `code` in *err - a word in
// pinned host memory the host side checks before its next call - instead of hanging the GPU.
__device__ __forceinline__ bool peer_wait(const unsigned int* flag, unsigned int epoch, int* err, int code) {
    unsigned long long t0 = 0;
    unsigned int spins = 0;
    for (;;) {
        unsigned int v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if (int(v - epoch) >= 0) return true;
        if ((++spins & 0xfffu) == 0) {
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (t0 == 0) t0 = t;
            else if (t - t0 > 20000000000ull) {
                if (err) { *reinterpret_cast<volatile int*>(err) = code; __threadfence_system(); }
                return false;
            }
        }
    }
}


// rows: merge the per-item parts (max, sum, dot; log2-scaled domain) into natural-log (max, sum, dot), as
// merge_row_parts_kernel.  columns: in single-sweep mode sum the per-row-block partial (sum, dot) of the global
// reference u; in exact mode merge the parts the swapped launch wrote.  The mode is recomputed from the same scalars.
// Block = 32 indices x 8 slices: the (up to hundreds of) row-block partials of a column are summed by 8 threads.
// sig.ticket != null (fused step on several ranks): the LAST block to finish publishes the epoch flag of the statistics
// exchange to every peer - the column statistics this kernel wrote are what they pull next - and returns the ticket to 0.
struct MergeSignal {
    unsigned int* ticket;
    PeerPtrs flags;
    int rank, world;
    unsigned int epoch;
};
__global__ void fwd_merge_kernel(const FwdArgs a0, const FwdArgs a1, int m_blocks, float* __restrict__ row_out,
                                 float* __restrict__ col_out, const __grid_constant__ MergeSignal sig) {
    const int lane = threadIdx.x & 31, sl = threadIdx.x >> 5;      // blockDim.x == 256
    const int i = blockIdx.x * 32 + lane;
    const int rows = a0.M, cols = a0.N;
    __shared__ float shL[8][32], shD[8][32];
    auto merge_parts = [](const float* pmx, const float* psm, const float* pdt, int nparts, int n, int idx, float* o, int on) {
        float m = -CUDART_INF_F;
        for (int p = 0; p < nparts; ++p) m = fmaxf(m, pmx[(size_t)p * n + idx]);
        float l = 0.f, t = 0.f;
        for (int p = 0; p < nparts; ++p) {
            const float pm = pmx[(size_t)p * n + idx];
            if (pm > -CUDART_INF_F) {
                const float w = exp2f(pm - m);
                l += psm[(size_t)p * n + idx] * w;
                t += pdt[(size_t)p * n + idx] * w;
            }
        }
        o[idx] = m * LN2;
        o[on + idx] = l;
        o[2 * on + idx] = t * LN2;
    };
    // parts of a row = (clusters whose tile range touches its row pair) x 2 column halves
    auto nparts_of = [](const FwdArgs& a, int row) {
        const long long total = (long long)a.m_pairs * a.n_tiles, f = (long long)(row / (2 * BM)) * a.n_tiles;
        return PARTS_PER_UNIT * (sweep_cluster_of(total, f + a.n_tiles - 1, a.n_clusters) - sweep_cluster_of(total, f, a.n_clusters) + 1);
    };
    if (sl == 0 && i < rows) merge_parts(a0.part_max, a0.part_sum, a0.part_dot, nparts_of(a0, i), rows, i, row_out, rows);
    float u;
    const bool single = fwd_bound(a0, &u);      // uniform over the grid
    if (blockIdx.x == 0 && threadIdx.x == 0 && a0.mode_out) *a0.mode_out = single ? 1.f : 0.f;
    if (single) {
        float L = 0.f, D = 0.f;
        if (i < cols)
            for (int b = sl; b < m_blocks; b += 8) {
                L += a0.colpart_sum[(size_t)b * a0.ldc + i];
                D += a0.colpart_dot[(size_t)b * a0.ldc + i];
            }
        shL[sl][lane] = L; shD[sl][lane] = D;
        __syncthreads();
        if (sl == 0 && i < cols) {
#pragma unroll
            for (int k = 1; k < 8; ++k) { L += shL[k][lane]; D += shD[k][lane]; }
            col_out[i] = u * LN2;
            col_out[cols + i] = L;
            col_out[2 * cols + i] = fmaf(u, L, D) * LN2;
        }
    } else if (sl == 0 && i < cols) {
        merge_parts(a1.part_max, a1.part_sum, a1.part_dot, nparts_of(a1, i), cols, i, col_out, cols);
    }
    if (sig.ticket) {
        __shared__ int last_block;
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            last_block = atomicAdd(sig.ticket, 1u) == gridDim.x - 1;
        }
        __syncthreads();
        if (last_block) {
            const int t = threadIdx.x;
            if (t < sig.world && t != sig.rank) peer_signal(static_cast<unsigned int*>(sig.flags.p[t]) + sig.rank, sig.epoch);
            if (t == 0) *sig.ticket = 0u;
        }
    }
}

// Rank of the target column in every row of a materialised fp32 logits panel (evaluation side: retrieval ranks of
// training/train.py:631-648, top-k accuracy of training/zero_shot.py:36-39) without sorting the row:
//   greater[r]     = #{ j : S[r, j] >  S[r, t_r] }
//   ties_before[r] = #{ j < t_r : S[r, j] == S[r, t_r] }       (greater + ties_before = position in a stable descending sort)
// One block per row, float4 loads; HBM-bound (4 bytes per logit, read once).
__global__ void rank_count_kernel(const float* __restrict__ S, long long ld, int cols, const long long* __restrict__ target,
                                  long long diag_offset, long long row0, int* __restrict__ greater,
                                  int* __restrict__ ties_before) {
    const long long gr = row0 + blockIdx.x;
    const long long tj = target ? target[gr] : diag_offset + gr;
    const bool valid = tj >= 0 && tj < cols;
    const float* row = S + (size_t)blockIdx.x * ld;
    int g = 0, t = 0;
    if (valid) {
        const float thr = row[tj];
        const int n4 = cols >> 2;
        const float4* row4 = reinterpret_cast<const float4*>(row);
        for (int q = threadIdx.x; q < n4; q += blockDim.x) {
            const float4 v = row4[q];
            const long long j = (long long)q << 2;
            g += int(v.x > thr) + int(v.y > thr) + int(v.z > thr) + int(v.w > thr);
            t += int(v.x == thr && j < tj) + int(v.y == thr && j + 1 < tj) + int(v.z == thr && j + 2 < tj) +
                 int(v.w == thr && j + 3 < tj);
        }
        for (int j = (n4 << 2) + threadIdx.x; j < cols; j += blockDim.x) {
            const float v = row[j];
            g += int(v > thr);
            t += int(v == thr && j < tj);
        }
    }
    __shared__ int sg[32], st[32];
    for (int o = 16; o > 0; o >>= 1) {
        g += __shfl_xor_sync(0xffffffffu, g, o);
        t += __shfl_xor_sync(0xffffffffu, t, o);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    if (lane == 0) { sg[warp] = g; st[warp] = t; }
    __syncthreads();
    if (warp == 0) {
        g = lane < nwarps ? sg[lane] : 0;
        t = lane < nwarps ? st[lane] : 0;
        for (int o = 16; o > 0; o >>= 1) {
            g += __shfl_xor_sync(0xffffffffu, g, o);
            t += __shfl_xor_sync(0xffffffffu, t, o);
        }
        if (lane == 0) {
            greater[gr] = valid ? g : -1;       // -1: the target column does not exist in this row
            if (ties_before) ties_before[gr] = valid ? t : 0;
        }
    }
}

// ---- distillation term of DistillClipLoss (loss.py:187-216) over a pair of materialised fp32 logits panels ----------
// S = student, T = teacher raw dot products of the same [rows, cols] block; logits are S * (*s_mul) and T * (*t_mul).
//   -sum_j softmax(T_i)(j) * log_softmax(S_i)(j) = lse(S_i) - sum_j exp(T_ij - lse(T_i)) * S_ij: the LSEs come from the
// fused forward of each model; the cross term needs both logits of an element at once, which is what these passes read.
// HBM-bound: 8 bytes per logit and pass.
__global__ void distill_row_cross_kernel(const float* __restrict__ S, const float* __restrict__ T, long long ld, int cols,
                                         const float* __restrict__ s_mul, const float* __restrict__ t_mul,
                                         const float* __restrict__ t_lse_row, long long row0,
                                         float* __restrict__ row_cross) {
    const long long g = row0 + blockIdx.x;
    const float sm = __ldg(s_mul), tm = __ldg(t_mul) * LOG2E, L = __ldg(t_lse_row + g) * LOG2E;
    const float* srow = S + (size_t)blockIdx.x * ld;
    const float* trow = T + (size_t)blockIdx.x * ld;
    float acc = 0.f;
    for (int j = threadIdx.x; j < cols; j += blockDim.x) acc = fmaf(ptx::ex2(fmaf(trow[j], tm, -L)), srow[j] * sm, acc);
    __shared__ float red[32];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    if (lane == 0) red[warp] = acc;
    __syncthreads();
    if (warp == 0) {
        acc = lane < nwarps ? red[lane] : 0.f;
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) row_cross[g] = acc;
    }
}
// col_part[j] = sum over the panel's rows of exp(T_ij - lse_col(T)(j)) * S_ij.  Block = 32 columns x 8 row lanes: a warp
// reads 32 consecutive floats of one row.
__global__ void distill_col_cross_kernel(const float* __restrict__ S, const float* __restrict__ T, int rows, int cols,
                                         long long ld, const float* __restrict__ s_mul, const float* __restrict__ t_mul,
                                         const float* __restrict__ t_lse_col, float* __restrict__ col_part) {
    const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int j = blockIdx.x * 32 + cx;
    const float sm = __ldg(s_mul), tm = __ldg(t_mul) * LOG2E;
    float acc = 0.f;
    if (j < cols) {
        const float L = __ldg(t_lse_col + j) * LOG2E;
        for (int r = ry; r < rows; r += 8) {
            const size_t o = (size_t)r * ld + j;
            acc = fmaf(ptx::ex2(fmaf(T[o], tm, -L)), S[o] * sm, acc);
        }
    }
    __shared__ float red[8][33];
    red[ry][cx] = acc;
    __syncthreads();
    if (ry == 0 && j < cols) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += red[k][cx];
        col_part[j] = t;
    }
}
// G = 2^14 * (P_row(S) - P_row(T) + P_col(S) - P_col(T)) as fp16: the derivative of both directions' distillation terms
// with respect to the student's logits (up to the 1 / (2 n) the caller applies), in the format the gradient GEMMs take.
__global__ void distill_grad_kernel(const float* __restrict__ S, const float* __restrict__ T, int cols, long long ld,
                                    const float* __restrict__ s_mul, const float* __restrict__ t_mul,
                                    const float* __restrict__ s_lse_row, const float* __restrict__ t_lse_row, long long row0,
                                    const float* __restrict__ s_lse_col, const float* __restrict__ t_lse_col,
                                    __half* __restrict__ G, long long ldg) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= cols) return;
    const long long g = row0 + blockIdx.y;
    const size_t o = (size_t)blockIdx.y * ld + j;
    const float s = S[o] * (__ldg(s_mul) * LOG2E), t = T[o] * (__ldg(t_mul) * LOG2E);
    const float v = ptx::ex2(s - __ldg(s_lse_row + g) * LOG2E) - ptx::ex2(t - __ldg(t_lse_row + g) * LOG2E) +
                    ptx::ex2(s - __ldg(s_lse_col + j) * LOG2E) - ptx::ex2(t - __ldg(t_lse_col + j) * LOG2E);
    G[(size_t)blockIdx.y * ldg + j] = __float2half_rn(16384.f * v);
}

// ---- data-parallel ranks of one NVLink domain: barrier and all-gather over peer-mapped (symmetric) memory (flags: see above)
__global__ void peer_barrier_kernel(const __grid_constant__ PeerPtrs flags, const int rank, const int world, const unsigned int epoch, int* const err) {
    const int t = threadIdx.x;
    if (t < world && t != rank) {
        peer_signal(static_cast<unsigned int*>(flags.p[t]) + rank, epoch);
        peer_wait(static_cast<const unsigned int*>(flags.p[rank]) + t, epoch, err, 2);
    }
}

// All-gather by pulling, flags included: chunk o of dst <- rank o's source buffer, for a main buffer and an optional small
// side buffer (the operand statistics travel with the text features).  Block (0, 0) first tells every peer that this
// rank's sources are complete (they were written by earlier kernels of this stream); the blocks of column o then wait
// for rank o's flag and copy with 16-byte loads, all sources in flight together (NVSwitch gives every pair its full
// link).  Peer data is read with ld.cv: a line of the same address cached by an earlier pull must not be served.
// A source buffer may be rewritten two calls later: before its owner got there it has waited, in the call in
// between, for a flag every reader published after finishing this pull.
struct GatherArgs {
    PeerPtrs src0; long long n16_0; uint4* dst0;
    PeerPtrs src1; long long n16_1; uint4* dst1;
    PeerPtrs flags;
    int rank, world;
    unsigned int epoch;
    int* err;
    int do_signal;        // 0: the flags were already published by the kernel that wrote the sources (work was put in between)
};
__global__ void peer_allgather_kernel(const __grid_constant__ GatherArgs a) {
    const int o = blockIdx.y;
    if (a.do_signal && blockIdx.x == 0 && blockIdx.y == 0 && int(threadIdx.x) < a.world && int(threadIdx.x) != a.rank)
        peer_signal(static_cast<unsigned int*>(a.flags.p[threadIdx.x]) + a.rank, a.epoch);
    const bool remote = o != a.rank;
    if (remote) {
        if (threadIdx.x == 0) peer_wait(static_cast<const unsigned int*>(a.flags.p[a.rank]) + o, a.epoch, a.err, 1);
        __syncthreads();
    }
    const long long stride = (long long)gridDim.x * blockDim.x;
    {
        const uint4* __restrict__ from = static_cast<const uint4*>(a.src0.p[o]);
        uint4* __restrict__ to = a.dst0 + (long long)o * a.n16_0;
        long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
        for (; i + 3 * stride < a.n16_0; i += 4 * stride) {      // four loads in flight per thread
            uint4 v0, v1, v2, v3;
            if (remote) { v0 = __ldcv(from + i); v1 = __ldcv(from + i + stride); v2 = __ldcv(from + i + 2 * stride); v3 = __ldcv(from + i + 3 * stride); }
            else { v0 = from[i]; v1 = from[i + stride]; v2 = from[i + 2 * stride]; v3 = from[i + 3 * stride]; }
            to[i] = v0; to[i + stride] = v1; to[i + 2 * stride] = v2; to[i + 3 * stride] = v3;
        }
        for (; i < a.n16_0; i += stride) to[i] = remote ? __ldcv(from + i) : from[i];
    }
    if (blockIdx.x == 0 && a.n16_1 > 0) {
        const uint4* __restrict__ from = static_cast<const uint4*>(a.src1.p[o]);
        uint4* __restrict__ to = a.dst1 + (long long)o * a.n16_1;
        for (long long i = threadIdx.x; i < a.n16_1; i += blockDim.x) to[i] = remote ? __ldcv(from + i) : from[i];
    }
}

// Test hook: where does tcgen05.ld.16x256b put the accumulator elements?  Four warps fill 128 lanes x 32 columns
// with lane * 1000 + column through the 32x32b shape (thread == lane); every warp then reads the two 16-lane halves of
// its lane quarter with the 16x256b shape and dumps its registers: out[(warp * 2 + h) * 32 * 16 + thread * 16 + k].
__global__ void tmem_layout_kernel(int* out) {
    __shared__ uint32_t tmem_ptr;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0) {
        ptx::tmem_alloc(ptx::smem_u32(&tmem_ptr), 32);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t base = tmem_ptr;
    uint32_t v[32];
    for (int k = 0; k < 32; ++k) v[k] = uint32_t((warp * 32 + lane) * 1000 + k);
    ptx::tmem_st_32x32(base + (uint32_t(warp * 32) << 16), v);
    ptx::tmem_st_wait();
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    for (int h = 0; h < 2; ++h) {
        uint32_t r[16];
        ptx::tmem_ld_16x256b_x4(base + (uint32_t(warp * 32 + h * 16) << 16), r);
        ptx::tmem_ld_wait();
        for (int k = 0; k < 16; ++k) out[((warp * 2 + h) * 32 + lane) * 16 + k] = int(r[k]);
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(base, 32);
    }
}

// ------------------------------------------------------------------------------------------------ launch helpers
static inline int cdiv(long long a, long long b) { return int((a + b - 1) / b); }
static inline long long round_up(long long a, long long b) { return (a + b - 1) / b * b; }

constexpr int MAX_SPLIT = 32;
constexpr int MAX_PARTS = MAX_SPLIT * PARTS_PER_UNIT;
// Budget of the fp16 G panel (CLIPK_PANEL_MB overrides it) - the only place a piece of the softmax gradient exists in
// memory.  It is a constant, independent of the problem size; what it buys is fewer recompute / gradient-GEMM launch pairs
// (each pays a fill and a drain of the persistent pipelines).  The panel streams through HBM either way - it stopped
// fitting the 126 MB L2 at 134 MB - and the traffic (written once, read by both gradient GEMMs) does not depend on how it is
// cut.  Measured at N = 32768, d = 512 on one B200, whole step: 48 MB panels (round 1, backward only) 3.13 vs 2.82 ms at
// 134-179 MB; round 2, same call (profiles/r02z_panel_budget_ab_1gpu.log): 192 MB (12 panels) 3.87 / 3.78 ms, 384 MB (6)
// 3.77, 512 MB (4) 3.66 / 3.80, the whole block as ONE 2 GiB panel 3.56 ms (3.55 in another call).
static long long panel_bytes() {
    static long long v = [] {
        const char* e = getenv("CLIPK_PANEL_MB");
        long long mb = e ? atoll(e) : 768;
        if (mb < 8) mb = 8;
        if (mb > 4096) mb = 4096;
        return mb << 20;
    }();
    return v;
}
// A block that fits ONE panel of up to 3x the budget takes it whole: a single recompute + gradient-GEMM launch instead of
// several (backward of one rank, profiles/r02z: 8-GPU shard 4096 x 32768, 268 MB: 343 vs 358 us with two panels; 4-GPU
// shard 8192 x 32768, 537 MB: 657 vs 676 us with four; 2-GPU shard, 1 GiB: 1279 vs 1336 us with six; one GPU, 2 GiB: see
// above).  With the default budget that covers blocks up to 2.25 GiB of fp16 G - the headline problem on 1..8 GPUs;
// anything larger (N = 65536 on one GPU: 8 GiB; N = 163840 on eight: 6.25 GiB per rank) is cut into panels of the budget,
// so the memory the backward needs stays bounded whatever N is.  CLIPK_PANEL_MB=192 restores round 1's small panels.
static long long panel_budget_for(long long rows, long long cols, int gplanes) {
    const long long whole = round_up(rows, 2 * BM) * round_up(cols, BN) * 2 * gplanes;
    const long long budget = panel_bytes();
    return (whole > budget && whole <= 3 * budget) ? whole : budget;
}

// How many CTAs share the column sweep of one 128-row block: fill the SMs in as few equal waves as possible.
static int choose_split(int m_pairs, int n_tiles, int sms) {
    const int m_blocks = 2 * m_pairs;   // CTAs per unit
    int best = 1;
    double best_cost = 1e30;
    const int lim = n_tiles < MAX_SPLIT ? n_tiles : MAX_SPLIT;
    for (int s = 1; s <= lim; ++s) {
        const int per = cdiv(n_tiles, s);
        const int waves = cdiv((long long)m_blocks * s, sms);
        const double cost = waves * (per + 0.35);   // 0.35 tile-times of prologue/epilogue per CTA
        if (cost < best_cost - 1e-9) { best_cost = cost; best = s; }
    }
    return best;
}

// Panel of the backward: G[rp x cp] (rp, cp multiples of 256) is produced by one recompute launch and consumed by the
// dX jobs (rp/256 * nt tiles, K = cp) and dY jobs (cp/256 * nt tiles, K = rp) of one gradient-GEMM launch.  All even
// splits of the block whose panel fits the budget are scored with a small cost model (us; constants measured at
// N = 32768, d = 512 on B200): per launch a fixed fill / drain, the recompute at ~2.7 us per tile and CTA pair, and
// the gradient GEMMs at 0.45 us per K block with the jobs list-scheduled, in launch order, over the CTA pairs.
// The choice depends only on the shape and is cached.
struct PanelKey {
    int rows, cols, d, gplanes, sms, one_row_panel;
    long long budget;
    bool operator==(const PanelKey& o) const {
        return rows == o.rows && cols == o.cols && d == o.d && gplanes == o.gplanes && sms == o.sms && budget == o.budget &&
               one_row_panel == o.one_row_panel;
    }
};
struct PanelChoice { PanelKey key; long long rp, cp; };
static std::mutex g_panel_mu;
static std::vector<PanelChoice> g_panel_cache;

static double panel_cost_us(int rb, int cb, int nt, int s_kb, int g_nseg, int pairs) {
    // recompute: tiles cut evenly over the pairs
    const double grad = 14.0 + cdiv((long long)rb * cb, pairs) * (2.7 * s_kb / 8.0);
    // gradient GEMMs: dX jobs (K = cb * 4 blocks) and dY jobs (K = rb * 4), each to the earliest free pair
    std::vector<double> free_at(pairs, 0.0);
    auto run = [&](int jobs, double len) {
        for (int j = 0; j < jobs; ++j) {
            auto it = std::min_element(free_at.begin(), free_at.end());
            *it += len;
        }
    };
    // the launch dispatches the kind with the longer K first (gemm_pair_kernel)
    if (cb >= rb) {
        run(rb * nt, 0.45 * 4 * cb * g_nseg);
        run(cb * nt, 0.45 * 4 * rb * g_nseg);
    } else {
        run(cb * nt, 0.45 * 4 * rb * g_nseg);
        run(rb * nt, 0.45 * 4 * cb * g_nseg);
    }
    const double pair = 12.0 + *std::max_element(free_at.begin(), free_at.end());
    return grad + pair;
}

// one_row_panel: prefer splits that keep all rows in ONE panel (fused reduce-scatter: the dY tiles of the first row panel
// are plain stores into the owners' slots, those of later row panels reduce-adds, ~3x slower over NVLink)
static void choose_panel(int rows, int cols, int d, int gplanes, int sms, long long budget, long long* rp_out, long long* cp_out,
                         int one_row_panel = 0) {
    const PanelKey key{rows, cols, d, gplanes, sms, one_row_panel, budget};
    {
        std::lock_guard<std::mutex> lk(g_panel_mu);
        for (const PanelChoice& c : g_panel_cache)
            if (c.key == key) { *rp_out = c.rp; *cp_out = c.cp; return; }
    }
    const int nt = cdiv(d, BN);
    const int R = cdiv(rows, 2 * BM), C = cdiv(cols, BN);       // available 256-row / 256-col blocks
    const int pairs = std::max(1, sms / 2);
    const int s_kb = cdiv(d, BK) * (gplanes == 2 ? 3 : 1);       // K blocks of a recompute tile (three plane pairs for fp32 inputs)
    const int g_nseg = gplanes == 2 ? 3 : 1;
    double best = 1e300;
    int best_rb = 1, best_cb = 1;
    int last_rb = 0;
    // a single row panel must leave room for at least one 256-column block
    const bool single_rows = one_row_panel && (long long)R * 4 * BM * BM * 2 * gplanes <= budget;
    for (int nr = 1; nr <= (single_rows ? 1 : R); ++nr) {
        const int rb = cdiv(R, nr);
        if (rb == last_rb) continue;
        last_rb = rb;
        int last_cb = 0;
        for (int nc = 1; nc <= C; ++nc) {
            const int cb = cdiv(C, nc);
            if (cb == last_cb) continue;
            last_cb = cb;
            if ((long long)rb * cb * 4 * BM * BM * 2 * gplanes > budget && (rb > 1 || cb > 1)) continue;
            const double cost = panel_cost_us(rb, cb, nt, s_kb, g_nseg, pairs) * cdiv(R, rb) * cdiv(C, cb);
            if (cost < best) { best = cost; best_rb = rb; best_cb = cb; }
        }
    }
    // experiments: CLIPK_PANEL_RB / CLIPK_PANEL_CB force the panel extents (in 256-blocks)
    if (const char* e = getenv("CLIPK_PANEL_RB")) best_rb = std::max(1, std::min(R, atoi(e)));
    if (const char* e = getenv("CLIPK_PANEL_CB")) best_cb = std::max(1, std::min(C, atoi(e)));
    const int nrp = cdiv(R, best_rb), ncp = cdiv(C, best_cb);
    *rp_out = (long long)cdiv(R, nrp) * 2 * BM;
    *cp_out = (long long)cdiv(C, ncp) * BN;
    if (getenv("CLIPK_VERBOSE")) fprintf(stderr, "[clipk] panel %d x %d blocks of 256 for a %d x %d x %d block (%d x %d panels, model %.0f us)\n", best_rb, best_cb, rows, cols, d, nrp, ncp, best);
    std::lock_guard<std::mutex> lk(g_panel_mu);
    if (g_panel_cache.size() < 256) g_panel_cache.push_back(PanelChoice{key, *rp_out, *cp_out});
}

// Launch with a thread-block cluster of two CTAs (the tcgen05 cta_group::2 pair).
template <typename... Args>
static int launch_clustered(const char* name, void (*kfn)(Args...), dim3 grid, dim3 cluster, int smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = size_t(smem);
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cluster.x;
    attr[0].val.clusterDim.y = cluster.y;
    attr[0].val.clusterDim.z = cluster.z;
    // programmatic dependent launch: this kernel's CTAs may be scheduled (and run their prologue up to
    // griddepcontrol.wait) while the previous kernel of the stream drains
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 2;
    CK_CUDA(cudaLaunchKernelEx(&cfg, kfn, args...));
    count_launch(name, st);
    return CLIPK_OK;
}

// tc = epilogue store map (G panel for GRAD, fp32 output for OUT; unused by STATS - pass ta).
// grid = (units, m_pairs): every unit is run by a PAIR of CTAs covering 256 rows.
template <int MODE, int F16>
static int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const KArgs& a, int units,
                       int m_pairs, cudaStream_t st) {
    auto kfn = gemm_kernel<MODE, F16>;
    constexpr int smem = smem_bytes_of(MODE);
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, [&] { attr_err = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); });
    if (attr_err != cudaSuccess) return fail(int(attr_err), "cudaFuncSetAttribute: %s", cudaGetErrorString(attr_err));
    KArgs aa = a;
    aa.f16 = F16;
    return launch_clustered(MODE == MODE_STATS ? "gemm_kernel<STATS>" : MODE == MODE_GRAD ? "gemm_kernel<GRAD>" : "gemm_kernel<OUT>", kfn, dim3(2 * m_pairs, units), dim3(2, 1, 1), smem, st, ta, tb, tc, aa);
}

// jobs0 / jobs1 are counted in PAIRS (256 x 256 output tiles)
static int launch_pair(const CUtensorMap& ta0, const CUtensorMap& tb0, const CUtensorMap& tc0, const KArgs& a0, int jobs0,
                       const CUtensorMap& ta1, const CUtensorMap& tb1, const CUtensorMap& tc1, const KArgs& a1, int jobs1,
                       const PeerOut& peers, cudaStream_t st) {
    auto kfn = gemm_pair_kernel<1>;
    constexpr int smem = smem_bytes_of(MODE_OUT);
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, [&] { attr_err = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); });
    if (attr_err != cudaSuccess) return fail(int(attr_err), "cudaFuncSetAttribute: %s", cudaGetErrorString(attr_err));
    KArgs b0 = a0, b1 = a1;
    b0.f16 = b1.f16 = 1;
    // the kind with the longer K goes first (see gemm_pair_kernel)
    const int dy_first = a1.num_kb > a0.num_kb ? 1 : 0;
    return launch_clustered("gemm_pair_kernel", kfn, dim3(2 * (jobs0 + jobs1)), dim3(2, 1, 1), smem, st, ta0, tb0, tc0, b0, ta1, tb1, tc1, b1,
                            jobs0, jobs1, dy_first, peers);
}

// plane pairs of the split-precision product, SMALLEST terms first: the tensor core truncates when it adds into the
// fp32 accumulator, so the big hi.hi products go last, when only d/16 more additions can bias the sum.
static const int kPairA[3] = {1, 0, 0};
static const int kPairB[3] = {0, 1, 0};

static inline int planes_of(int dtype) { return dtype == CLIPK_F16X2 ? 2 : 1; }
static inline bool is_f16(int dtype) { return dtype == CLIPK_F16 || dtype == CLIPK_F16X2; }

// one K segment for single-plane operands; three for two-plane ones (planes `a_plane` / `b_plane` inner elements apart)
static void set_segments(KArgs& a, int planes, int k_extent, long long a_plane, long long b_plane) {
    a.kb_per_seg = cdiv(k_extent, BK);
    a.nseg = (planes == 2) ? 3 : 1;
    a.num_kb = a.nseg * a.kb_per_seg;
    for (int i = 0; i < 3; ++i) { a.a_off[i] = 0; a.b_off[i] = 0; }
    if (planes == 2)
        for (int i = 0; i < 3; ++i) {
            a.a_off[i] = int(kPairA[i] * a_plane);
            a.b_off[i] = int(kPairB[i] * b_plane);
        }
}

static int check_common(const void* X, const void* Y, int rows, int cols, int d, long long ldx, long long ldy, int dtype) {
    if (!X || !Y) return fail(CLIPK_EINVAL, "null operand pointer");
    if (rows <= 0 || cols <= 0 || d <= 0) return fail(CLIPK_EINVAL, "rows, cols and d must be positive (got %d, %d, %d)", rows, cols, d);
    if (dtype != CLIPK_BF16 && dtype != CLIPK_F16 && dtype != CLIPK_F16X2)
        return fail(CLIPK_EUNSUPPORTED, "dtype %d: operands must be CLIPK_BF16, CLIPK_F16 or CLIPK_F16X2 (fp32 inputs go through clipk_to_f16 first)", dtype);
    const long long need = (dtype == CLIPK_BF16) ? d : planes_of(dtype) * round_up(d, BK);
    if (ldx < need || ldy < need) return fail(CLIPK_EINVAL, "leading dimension smaller than the row width (%lld)", need);
    if (d % 8 != 0) return fail(CLIPK_EUNSUPPORTED, "d = %d is not a multiple of 8", d);
    return CLIPK_OK;
}

template <int F16>
static int launch_grad_sweep(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const KArgs& a,
                             const SweepGeom& g, int n_clusters, cudaStream_t st) {
    auto kfn = grad_sweep_kernel<F16>;
    constexpr int smem = smem_bytes_grad_sweep();
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, [&] { attr_err = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); });
    if (attr_err != cudaSuccess) return fail(int(attr_err), "cudaFuncSetAttribute: %s", cudaGetErrorString(attr_err));
    KArgs aa = a;
    aa.f16 = F16;
    return launch_clustered("grad_sweep_kernel", kfn, dim3(2 * n_clusters), dim3(2, 1, 1), smem, st, ta, tb, tc, aa, g);
}

// ---- host helpers of clipk_fwd_both
// upper bound of the parts (clusters) that share one row pair of a sweep, for any device with <= 256 SMs
static int sweep_parts_bound(int rows) {
    const int m_pairs = cdiv(rows, 2 * BM);
    return std::min(128, cdiv(128, m_pairs) + 1);
}
struct FwdCarve {
    size_t norm2, parts0, parts1, colparts, total;
    int ldc, m_blocks;
};
FwdCarve fwd_carve(int rows, int cols) {
    FwdCarve c;
    c.ldc = int(round_up(cols, BN));
    c.m_blocks = 2 * cdiv(rows, 2 * BM);
    size_t off = 0;
    c.norm2 = off; off += 256;
    c.parts0 = off; off += size_t(3) * sweep_parts_bound(rows) * PARTS_PER_UNIT * rows * sizeof(float);
    c.parts1 = off; off += size_t(3) * sweep_parts_bound(cols) * PARTS_PER_UNIT * cols * sizeof(float);
    off = size_t(round_up((long long)off, 256));
    c.colparts = off; off += size_t(2) * c.m_blocks * c.ldc * sizeof(float);
    c.total = off + 256;
    return c;
}
template <int F16, bool ARES>
int launch_fwd_sweep(const CUtensorMap& ta, const CUtensorMap& tb, const FwdArgs& a, int n_clusters, cudaStream_t st) {
    auto kfn = fwd_sweep_kernel<F16, ARES>;
    constexpr int smem = smem_bytes_fwd(ARES);
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, [&] { attr_err = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); });
    if (attr_err != cudaSuccess) return fail(int(attr_err), "cudaFuncSetAttribute: %s", cudaGetErrorString(attr_err));
    return launch_clustered("fwd_sweep_kernel", kfn, dim3(2 * n_clusters), dim3(2, 1, 1), smem, st, ta, tb, a);
}

// ---- SigLipLoss (clipk_siglip_forward / _backward) -------------------------------------------------------------------
enum { SIG_LOSS = 0, SIG_GMAX = 1, SIG_MAXNEG = 2, SIG_MINPOS = 3, SIG_P2E = 4, SIG_OSCALE = 5 };   // state words
// Largest G panel of the SigLIP backward: it stays L2-resident between the recompute that writes it and the two gradient
// GEMMs that read it, and the backward's extra memory stays a small fraction of the b x N logits the formula holds.
constexpr long long SIG_PANEL_BYTES = 64ll << 20;

// Per row: the partial sums of the sweep's (part, half) slots, in part order.  Forward (max_b): out_a = sum of
// softplus / ln 2, out_b = largest negative logit * log2(e).  Recompute: out_a (+)= sum g, out_b (+)= sum g x.y
// (accumulate: later column panels add to the earlier ones, in panel order).
__global__ void siglip_rows_kernel(const float* __restrict__ part_a, const float* __restrict__ part_b, int M,
                                   const SweepGeom g, int n_clusters, int max_b, int accumulate, float* __restrict__ out_a,
                                   float* __restrict__ out_b) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const long long total = (long long)g.m_pairs * g.n_tiles, f = (long long)(i / (2 * BM)) * g.n_tiles;
    const int nparts = PARTS_PER_UNIT * (sweep_cluster_of(total, f + g.n_tiles - 1, n_clusters) - sweep_cluster_of(total, f, n_clusters) + 1);
    float a = 0.f, b = max_b ? -CUDART_INF_F : 0.f;
    for (int p = 0; p < nparts; ++p) {
        a += part_a[(size_t)p * M + i];
        const float v = part_b[(size_t)p * M + i];
        b = max_b ? fmaxf(b, v) : b + v;
    }
    if (accumulate) { a += out_a[i]; b += out_b[i]; }
    out_a[i] = a;
    out_b[i] = b;
}

__device__ __forceinline__ float sig_sigmoid(float x) { return 1.f / (1.f + expf(-x)); }

// One block of 1024 threads, fixed-order sums over the rows (strided per thread, then a tree).
//   forward  (go == null): state[LOSS] = ln 2 / b * sum row_a, [MAXNEG] = max row_b * ln 2, [MINPOS] = min pos,
//                          [GMAX] = max(sigma(MAXNEG), sigma(-MINPOS)) = the largest |g| of the block
//   backward            : d_bias = go / b * sum row_a, d_scale = go / b * sum row_b  (either may be null)
__global__ void __launch_bounds__(1024) siglip_reduce_kernel(const float* __restrict__ row_a, const float* __restrict__ row_b,
                                                             const float* __restrict__ pos, int M, float* __restrict__ state,
                                                             const float* __restrict__ go, float* d_scale, float* d_bias) {
    __shared__ float sa[1024], sb[1024], sp[1024];
    const int tid = threadIdx.x;
    const bool fwd = go == nullptr;
    float a = 0.f, b = fwd ? -CUDART_INF_F : 0.f, pm = CUDART_INF_F;
    for (int i = tid; i < M; i += 1024) {
        a += row_a[i];
        if (fwd) { b = fmaxf(b, row_b[i]); pm = fminf(pm, pos[i]); }
        else b += row_b[i];
    }
    sa[tid] = a; sb[tid] = b; sp[tid] = pm;
    __syncthreads();
    for (int w = 512; w > 0; w >>= 1) {
        if (tid < w) {
            sa[tid] += sa[tid + w];
            sb[tid] = fwd ? fmaxf(sb[tid], sb[tid + w]) : sb[tid] + sb[tid + w];
            sp[tid] = fminf(sp[tid], sp[tid + w]);
        }
        __syncthreads();
    }
    if (tid != 0) return;
    if (fwd) {
        const float maxneg = sb[0] * LN2, minpos = sp[0];
        state[SIG_LOSS] = sa[0] * LN2 / float(M);
        state[SIG_MAXNEG] = maxneg;
        state[SIG_MINPOS] = minpos;
        state[SIG_GMAX] = fmaxf(maxneg > -CUDART_INF_F ? sig_sigmoid(maxneg) : 0.f, sig_sigmoid(-minpos));
    } else {
        const float k = go[0] / float(M);
        if (d_bias) d_bias[0] = sa[0] * k;
        if (d_scale) d_scale[0] = sb[0] * k;
    }
}

// The power of two of the G panel, from gmax: the largest |g| * 2^e lands in [2^13, 2^14) of fp16 (CLIP's fixed 2^14
// would leave a well-separated batch, every |g| ~ 2e-9, in fp16 subnormals).  e <= 64 keeps go * s / (b * 2^e) times the
// fp16 operand scales a normal fp32 number; gmax = 0 / NaN (a NaN feature) takes 2^14.
__global__ void siglip_bwd_prep_kernel(float* __restrict__ state, const float* __restrict__ go,
                                       const float* __restrict__ scale, int rows) {
    const float gmax = state[SIG_GMAX];
    int e = 14;
    if (gmax > 0.f && gmax <= 1.f) {
        int k = 0;
        frexpf(gmax, &k);                  // gmax = m * 2^k, m in [0.5, 1)
        e = 14 - k;
        if (e > 64) e = 64;
    }
    state[SIG_P2E] = ldexpf(1.f, e);
    state[SIG_OSCALE] = go[0] * scale[0] / float(rows) * ldexpf(1.f, -e);
}

template <bool ARES>
static int launch_sig_fwd(const CUtensorMap& ta, const CUtensorMap& tb, const SigArgs& a, const SweepGeom& g, int n_clusters,
                          cudaStream_t st) {
    auto kfn = siglip_fwd_kernel<ARES>;
    constexpr int smem = smem_bytes_sig_fwd(ARES);
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, [&] { attr_err = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); });
    if (attr_err != cudaSuccess) return fail(int(attr_err), "cudaFuncSetAttribute: %s", cudaGetErrorString(attr_err));
    return launch_clustered("siglip_fwd_kernel", kfn, dim3(2 * n_clusters), dim3(2, 1, 1), smem, st, ta, tb, a, g);
}
template <bool ARES>
static int launch_sig_grad(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const SigArgs& a,
                           const SweepGeom& g, int n_clusters, cudaStream_t st) {
    auto kfn = siglip_grad_kernel<ARES>;
    constexpr int smem = smem_bytes_sig_grad(ARES);
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, [&] { attr_err = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); });
    if (attr_err != cudaSuccess) return fail(int(attr_err), "cudaFuncSetAttribute: %s", cudaGetErrorString(attr_err));
    return launch_clustered("siglip_grad_kernel", kfn, dim3(2 * n_clusters), dim3(2, 1, 1), smem, st, ta, tb, tc, a, g);
}

}  // namespace clipk

using namespace clipk;

// ================================================================================================ C ABI
extern "C" {

int clipk_version(void) { return CLIPK_VERSION; }
long long clipk_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
const char* clipk_last_error(void) { return g_err; }

int clipk_check_device(void) {
    DevInfo di;
    return device_info(&di);
}

static int to_f16_impl(const void* src, int src_dtype, long long rows, long long d, long long ld_src, void* dst, int planes,
                       long long ld_dst, float* scale_io, const float* amax, void* stream);

int clipk_to_f16(const void* src, int src_dtype, long long rows, long long d, long long ld_src, void* dst, int planes,
                 long long ld_dst, float* scale_io, void* stream) {
    return to_f16_impl(src, src_dtype, rows, d, ld_src, dst, planes, ld_dst, scale_io, nullptr, stream);
}

int clipk_to_f16_amax(const void* src, int src_dtype, long long rows, long long d, long long ld_src, void* dst, int planes,
                      long long ld_dst, float* scale_io, const float* amax, void* stream) {
    if (!amax) return fail(CLIPK_EINVAL, "null amax");
    return to_f16_impl(src, src_dtype, rows, d, ld_src, dst, planes, ld_dst, scale_io, amax, stream);
}

static int to_f16_impl(const void* src, int src_dtype, long long rows, long long d, long long ld_src, void* dst, int planes,
                       long long ld_dst, float* scale_io, const float* amax, void* stream) {
    if (!src || !dst || !scale_io || rows <= 0 || d <= 0) return fail(CLIPK_EINVAL, "bad argument");
    if (planes != 1 && planes != 2) return fail(CLIPK_EINVAL, "planes must be 1 or 2");
    if (src_dtype != CLIPK_BF16 && src_dtype != CLIPK_F32) return fail(CLIPK_EUNSUPPORTED, "source dtype %d", src_dtype);
    const long long dpad = round_up(d, BK);
    if (ld_src < d || ld_dst != planes * dpad) return fail(CLIPK_EINVAL, "ld_dst must be planes * round_up(d, 64) = %lld", planes * dpad);
    DevInfo di;
    int rc = device_info(&di);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // scale_io[0] = max |x| (bit pattern): computed here, or handed in by the caller (clipk_fwd_both's amax_xy)
    if (amax) CK_CUDA(cudaMemcpyAsync(scale_io, amax, sizeof(float), cudaMemcpyDeviceToDevice, st));
    else CK_CUDA(cudaMemsetAsync(scale_io, 0, 2 * sizeof(float), st));
    if (d % 8 != 0) return fail(CLIPK_EUNSUPPORTED, "d = %lld is not a multiple of 8", d);
    if ((reinterpret_cast<uintptr_t>(src) & 15) != 0 || (ld_src * (src_dtype == CLIPK_BF16 ? 2 : 4)) % 16 != 0)
        return fail(CLIPK_EINVAL, "source rows must be 16-byte aligned");
    const long long n = rows * (dpad / 8);
    const long long n_src = rows * (d / 8);
    const int rblocks = int(n_src / 256 < 1 ? 1 : (n_src / 256 > 8 * di.sms ? 8 * di.sms : n_src / 256));
    unsigned int* bits = reinterpret_cast<unsigned int*>(scale_io);
    __half* out = static_cast<__half*>(dst);
    if (src_dtype == CLIPK_BF16) {
        const __nv_bfloat16* p = static_cast<const __nv_bfloat16*>(src);
        if (!amax) {
            amax_kernel<<<rblocks, 256, 0, st>>>(p, rows, d / 8, ld_src, bits);
            count_launch("amax_kernel", st);
        }
        to_f16_kernel<<<cdiv(n, 256), 256, 0, st>>>(p, out, rows, d, ld_src, dpad, planes, scale_io);
        count_launch("to_f16_kernel", st);
    } else {
        const float* p = static_cast<const float*>(src);
        if (!amax) {
            amax_kernel<<<rblocks, 256, 0, st>>>(p, rows, d / 8, ld_src, bits);
            count_launch("amax_kernel", st);
        }
        to_f16_kernel<<<cdiv(n, 256), 256, 0, st>>>(p, out, rows, d, ld_src, dpad, planes, scale_io);
        count_launch("to_f16_kernel", st);
    }
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}

size_t clipk_fwd_workspace_bytes(int rows, int cols, int d, int dtype) {
    (void)cols; (void)d; (void)dtype;
    if (rows <= 0) return 0;
    return size_t(3) * MAX_PARTS * size_t(rows) * sizeof(float) + 256;
}

int clipk_fwd_stats(const void* X, const void* Y, int rows, int cols, int d, long long ldx, long long ldy, int dtype,
                    const float* x_inv_scale, const float* y_inv_scale, const float* logit_scale,
                    long long diag_offset, float* row_max, float* row_sum, float* row_dot, float* pos_logit,
                    void* workspace, size_t workspace_bytes, void* stream) {
    int rc = check_common(X, Y, rows, cols, d, ldx, ldy, dtype);
    if (rc) return rc;
    if (!logit_scale || !row_max || !row_sum || !row_dot || !workspace) return fail(CLIPK_EINVAL, "null pointer argument");
    if (workspace_bytes < clipk_fwd_workspace_bytes(rows, cols, d, dtype)) return fail(CLIPK_EWORKSPACE, "workspace too small");
    DevInfo di;
    if ((rc = device_info(&di))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);

    const int planes = planes_of(dtype);
    const long long dpad = round_up(d, BK);
    const long long kext = (dtype == CLIPK_BF16) ? d : planes * dpad;
    CUtensorMap ta, tb;
    if ((rc = tmap_kmajor(&ta, X, rows, kext, ldx, BM))) return rc;
    if ((rc = tmap_kmajor(&tb, Y, cols, kext, ldy, BN / 2))) return rc;
    KArgs a{};
    a.M = rows; a.N = cols; a.n_tiles = cdiv(cols, BN);
    set_segments(a, planes, d, dpad, dpad);
    const int m_pairs = cdiv(rows, 2 * BM);
    const int split = choose_split(m_pairs, a.n_tiles, di.sms);
    a.tiles_per_unit = cdiv(a.n_tiles, split);
    const int units = cdiv(a.n_tiles, a.tiles_per_unit);
    a.scale = logit_scale; a.xs = x_inv_scale; a.ys = y_inv_scale; a.diag_offset = diag_offset;
    a.part_max = static_cast<float*>(workspace);
    a.part_sum = a.part_max + size_t(MAX_PARTS) * rows;
    a.part_dot = a.part_sum + size_t(MAX_PARTS) * rows;
    a.pos = pos_logit;
    if (!pos_logit) a.diag_offset = -(1LL << 40);   // no row has a positive inside [0, cols)
    if (is_f16(dtype)) {
        rc = launch_gemm<MODE_STATS, 1>(ta, tb, ta, a, units, m_pairs, st);
    } else {
        rc = launch_gemm<MODE_STATS, 0>(ta, tb, ta, a, units, m_pairs, st);
    }
    if (rc) return rc;
    merge_row_parts_kernel<<<cdiv(rows, 256), 256, 0, st>>>(a.part_max, a.part_sum, a.part_dot, units * PARTS_PER_UNIT,
                                                            rows, row_max, row_sum, row_dot);
    count_launch("merge_row_parts_kernel", st);
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}

// ---- both directions of the forward (see fwd_sweep_kernel)

size_t clipk_fwd_both_workspace_bytes(int rows, int cols, int d, int dtype) {
    if (rows <= 0 || cols <= 0) return 0;
    const size_t two = clipk_fwd_workspace_bytes(rows, cols, d, dtype) + clipk_fwd_workspace_bytes(cols, rows, d, dtype);
    const size_t one = fwd_carve(rows, cols).total;
    return one > two ? one : two;
}

// launch of prep_kernel over (X rows, Y rows); stats must be this rank's row of the table (it is reset here)
constexpr int PREP_MAX_BLOCKS = 1024;        // bound of the partials array of the ticket path
static int launch_prep(const PrepArgs& a, int src_dtype, int normalize, int sms, cudaStream_t st) {
    if (!a.ticket) CK_CUDA(cudaMemsetAsync(a.stats, 0, STAT_WORDS * sizeof(float), st));
    const long long nmax = a.rows_x > a.rows_y ? a.rows_x : a.rows_y;
    const int wpb = 8;
    const int blocks = int(std::max<long long>(1, std::min<long long>(cdiv(nmax, wpb), std::min<long long>(4LL * sms, PREP_MAX_BLOCKS))));
    if (src_dtype == CLIPK_BF16) {
        if (normalize) prep_kernel<__nv_bfloat16, true><<<blocks, wpb * 32, 0, st>>>(a);
        else prep_kernel<__nv_bfloat16, false><<<blocks, wpb * 32, 0, st>>>(a);
    } else {
        if (normalize) prep_kernel<float, true><<<blocks, wpb * 32, 0, st>>>(a);
        else prep_kernel<float, false><<<blocks, wpb * 32, 0, st>>>(a);
    }
    count_launch("prep_kernel", st);
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}

// The sweeps + merge of the forward for one-plane operands (bf16 / fp16): row statistics [3, rows], positives [rows] and
// this block's column statistics [3, cols].  stats = operand statistics table (null: no bound, exact mode).
static int fwd_sweeps(const void* X, const void* Y, int rows, int cols, int d, long long ldx, long long ldy, int dtype,
                      const float* x_inv_scale, const float* y_inv_scale, const float* logit_scale, long long diag_offset,
                      float* row_stats, float* pos_logit, float* col_stats, const float* stats, int nstat, int stats_rank,
                      int use_minpos, int exact, void* workspace, const DevInfo& di, cudaStream_t st,
                      const MergeSignal* signal = nullptr) {
    int rc;
    const long long dpad = round_up(d, BK);
    const int num_kb = cdiv(d, BK);
    const long long kext = (dtype == CLIPK_BF16) ? d : dpad;
    const int n_clusters = di.sms / 2;
    const FwdCarve cv = fwd_carve(rows, cols);
    char* ws = static_cast<char*>(workspace);
    float* parts0 = reinterpret_cast<float*>(ws + cv.parts0);
    float* parts1 = reinterpret_cast<float*>(ws + cv.parts1);
    float* colparts = reinterpret_cast<float*>(ws + cv.colparts);
    CUtensorMap tx_a, ty_b, ty_a, tx_b;
    if ((rc = tmap_kmajor(&tx_a, X, rows, kext, ldx, BM))) return rc;
    if ((rc = tmap_kmajor(&ty_b, Y, cols, kext, ldy, BN / 2))) return rc;
    if ((rc = tmap_kmajor(&ty_a, Y, cols, kext, ldy, BM))) return rc;
    if ((rc = tmap_kmajor(&tx_b, X, rows, kext, ldx, BN / 2))) return rc;

    FwdArgs a0{};
    a0.M = rows; a0.N = cols; a0.num_kb = num_kb;
    a0.n_tiles = cdiv(cols, BN); a0.m_pairs = cdiv(rows, 2 * BM);
    a0.n_clusters = int(std::min<long long>(n_clusters, (long long)a0.m_pairs * a0.n_tiles));
    a0.pass = 0; a0.force_exact = (stats && !exact) ? 0 : 1;
    a0.scale = logit_scale; a0.xs = x_inv_scale; a0.ys = y_inv_scale;
    a0.stats = stats; a0.nstat = nstat; a0.stats_rank = stats_rank; a0.use_minpos = (use_minpos && pos_logit) ? 1 : 0;
    a0.mode_out = stats ? const_cast<float*>(stats) + stats_rank * STAT_WORDS + 5 : nullptr;
    a0.diag_offset = pos_logit ? diag_offset : -(1LL << 40);
    const size_t pstride0 = size_t(sweep_parts_bound(rows)) * PARTS_PER_UNIT * rows;
    a0.part_max = parts0; a0.part_sum = parts0 + pstride0; a0.part_dot = parts0 + 2 * pstride0;
    a0.pos = pos_logit;
    a0.colpart_sum = colparts; a0.colpart_dot = colparts + size_t(cv.m_blocks) * cv.ldc; a0.ldc = cv.ldc;

    FwdArgs a1 = a0;
    a1.M = cols; a1.N = rows;
    a1.n_tiles = cdiv(rows, BN); a1.m_pairs = cdiv(cols, 2 * BM);
    a1.n_clusters = int(std::min<long long>(n_clusters, (long long)a1.m_pairs * a1.n_tiles));
    a1.pass = 1; a1.xs = y_inv_scale; a1.ys = x_inv_scale;
    a1.diag_offset = -(1LL << 40);
    const size_t pstride1 = size_t(sweep_parts_bound(cols)) * PARTS_PER_UNIT * cols;
    a1.part_max = parts1; a1.part_sum = parts1 + pstride1; a1.part_dot = parts1 + 2 * pstride1;
    a1.pos = nullptr; a1.colpart_sum = nullptr; a1.colpart_dot = nullptr;

    const int nc0 = a0.n_clusters, nc1 = a1.n_clusters;
    const bool ares = num_kb <= ARES_KB;       // rows of the left operand resident in shared memory (K <= 512)
    if (is_f16(dtype)) {
        if ((rc = ares ? launch_fwd_sweep<1, true>(tx_a, ty_b, a0, nc0, st) : launch_fwd_sweep<1, false>(tx_a, ty_b, a0, nc0, st))) return rc;
        if ((rc = ares ? launch_fwd_sweep<1, true>(ty_a, tx_b, a1, nc1, st) : launch_fwd_sweep<1, false>(ty_a, tx_b, a1, nc1, st))) return rc;
    } else {
        if ((rc = ares ? launch_fwd_sweep<0, true>(tx_a, ty_b, a0, nc0, st) : launch_fwd_sweep<0, false>(tx_a, ty_b, a0, nc0, st))) return rc;
        if ((rc = ares ? launch_fwd_sweep<0, true>(ty_a, tx_b, a1, nc1, st) : launch_fwd_sweep<0, false>(ty_a, tx_b, a1, nc1, st))) return rc;
    }
    const int n = rows > cols ? rows : cols;
    MergeSignal sig;
    memset(&sig, 0, sizeof(sig));
    if (signal) sig = *signal;
    fwd_merge_kernel<<<cdiv(n, 32), 256, 0, st>>>(a0, a1, cv.m_blocks, row_stats, col_stats, sig);
    count_launch("fwd_merge_kernel", st);
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}

int clipk_fwd_both(const void* X, const void* Y, int rows, int cols, int d, long long ldx, long long ldy, int dtype,
                   const float* x_inv_scale, const float* y_inv_scale, const float* logit_scale, long long diag_offset,
                   float* row_stats, float* pos_logit, float* col_stats, float* amax_xy, int exact, void* workspace,
                   size_t workspace_bytes, void* stream) {
    int rc = check_common(X, Y, rows, cols, d, ldx, ldy, dtype);
    if (rc) return rc;
    if (!logit_scale || !row_stats || !col_stats || !workspace) return fail(CLIPK_EINVAL, "null pointer argument");
    if (workspace_bytes < clipk_fwd_both_workspace_bytes(rows, cols, d, dtype)) return fail(CLIPK_EWORKSPACE, "workspace too small");
    if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) return fail(CLIPK_EINVAL, "workspace must be 256-byte aligned");
    DevInfo di;
    if ((rc = device_info(&di))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int planes = planes_of(dtype);
    if (amax_xy) CK_CUDA(cudaMemsetAsync(amax_xy, 0xff, 2 * sizeof(float), st));   // NaN = not computed
    if (planes != 1) {
        // split-precision operands (fp32 inputs): two streaming sweeps
        char* ws = static_cast<char*>(workspace);
        const size_t w0 = clipk_fwd_workspace_bytes(rows, cols, d, dtype);
        rc = clipk_fwd_stats(X, Y, rows, cols, d, ldx, ldy, dtype, x_inv_scale, y_inv_scale, logit_scale, diag_offset,
                             row_stats, row_stats + rows, row_stats + 2 * (size_t)rows, pos_logit, ws, w0, stream);
        if (rc) return rc;
        return clipk_fwd_stats(Y, X, cols, rows, d, ldy, ldx, dtype, y_inv_scale, x_inv_scale, logit_scale, -(1LL << 40),
                               col_stats, col_stats + cols, col_stats + 2 * (size_t)cols, nullptr, ws + round_up((long long)w0, 256),
                               workspace_bytes - size_t(round_up((long long)w0, 256)), stream);
    }
    float* stats = nullptr;
    if (dtype == CLIPK_BF16) {
        // statistics of both operands in one pass; the positives' bound only when every column's positive is one of
        // this call's rows, i.e. when the block is the whole problem (rows == cols, diagonal positives)
        stats = reinterpret_cast<float*>(static_cast<char*>(workspace) + fwd_carve(rows, cols).norm2);
        PrepArgs pa{};
        pa.x = X; pa.y = Y; pa.rows_x = rows; pa.rows_y = cols; pa.ldx = ldx; pa.ldy = ldy; pa.d8 = d / 8;
        pa.pair_off = pos_logit ? diag_offset : (1LL << 40);
        pa.stats = stats;
        if ((rc = launch_prep(pa, CLIPK_BF16, 0, di.sms, st))) return rc;
        if (amax_xy) CK_CUDA(cudaMemcpyAsync(amax_xy, stats + 2, 2 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    const int use_minpos = (pos_logit && rows == cols && diag_offset == 0) ? 1 : 0;
    return fwd_sweeps(X, Y, rows, cols, d, ldx, ldy, dtype, x_inv_scale, y_inv_scale, logit_scale, diag_offset, row_stats,
                      pos_logit, col_stats, stats, 1, 0, use_minpos, exact, workspace, di, st);
}

int clipk_finalize(const float* row_max, const float* row_sum, const float* row_dot, const float* pos_logit, int rows,
                   const float* col_max_parts, const float* col_sum_parts, const float* col_dot_parts, int nparts,
                   long long part_stride, int cols, long long diag_offset, float* lse_row, float* lse_col, float* sums,
                   void* stream) {
    if (!row_max || !row_sum || !row_dot || !pos_logit || !col_max_parts || !col_sum_parts || !col_dot_parts || !lse_row ||
        !lse_col || !sums)
        return fail(CLIPK_EINVAL, "null pointer argument");
    if (rows <= 0 || cols <= 0 || nparts <= 0) return fail(CLIPK_EINVAL, "rows, cols and nparts must be positive");
    if (part_stride < cols) return fail(CLIPK_EINVAL, "part_stride smaller than cols");
    DevInfo di;
    int rc = device_info(&di);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CK_CUDA(cudaMemsetAsync(sums, 0, 4 * sizeof(float), st));
    const int n = rows > cols ? rows : cols;
    finalize_kernel<<<cdiv(n, 256), 256, 0, st>>>(row_max, row_sum, row_dot, pos_logit, rows, col_max_parts, col_sum_parts,
                                                  col_dot_parts, nparts, part_stride, cols, diag_offset, lse_row, lse_col,
                                                  sums, nullptr, 1.f);
    count_launch("finalize_kernel", st);
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}

size_t clipk_bwd_workspace_bytes(int rows, int cols, int d, int g_dtype) {
    if (rows <= 0 || cols <= 0 || d <= 0) return 0;
    // one G panel (two planes at most), slack for its padding, and the reference vectors of the recompute
    const long long panel = std::max(panel_budget_for(rows, cols, 1), panel_budget_for(rows, cols, 2));
    return size_t(panel) + size_t(4) * 1024 * 1024 + (size_t(rows) + size_t(cols)) * sizeof(float) + 4096;
}

static int bwd_impl(const void* X, const void* Y, int rows, int cols, int d, long long ldx, long long ldy, int dtype,
                    const float* x_inv_scale, const float* y_inv_scale, const void* Xg, const void* Yg, long long ldxg,
                    long long ldyg, int g_dtype, const float* xg_inv_scale, const float* yg_inv_scale,
                    const float* logit_scale, long long diag_offset, const float* lse_row, const float* lse_col,
                    float alpha, float beta, const float* gscale, float* dX_acc, float* dY_acc, void* const* dY_peer_acc,
                    int world, int rows_per_rank, void* workspace, size_t workspace_bytes, void* stream,
                    const int* mm_ready = nullptr, float coef = 1.f, int split_row_col = 0) {
    // mm_ready: min / max of both LSE vectors (ordered ints) already computed by the forward (clipk_step_forward);
    // coef: constant factor on both gradients next to the device scalar *gscale;
    // split_row_col: dX is built from alpha (P_row - Id) only and dY from beta (P_col - Id) only - the gradients of
    // local_loss without gather_with_grad (loss.py:53-56: the gathered tensors carry no gradient) - from ONE recompute
    // that writes the two parts as two planes of the panel (one-plane fp16 operands only)
    int rc = check_common(X, Y, rows, cols, d, ldx, ldy, dtype);
    if (rc) return rc;
    PeerOut peers;
    memset(&peers, 0, sizeof(peers));
    if (dY_peer_acc) {
        // fused reduce-scatter: dY tiles are written into this rank's slot at their owners (see gemm_pair_kernel)
        if (world < 1 || world > MAX_PEERS) return fail(CLIPK_EUNSUPPORTED, "peer output supports 1..%d ranks (got %d)", MAX_PEERS, world);
        if (rows_per_rank <= 0 || rows_per_rank % BM != 0 || (long long)rows_per_rank * world != cols)
            return fail(CLIPK_EUNSUPPORTED, "peer output needs cols == world * rows_per_rank and rows_per_rank %% 128 == 0");
        if (!dX_acc || dY_acc) return fail(CLIPK_EINVAL, "peer output: dX_acc is required and dY_acc must be NULL");
        for (int o = 0; o < world; ++o) {
            if (!dY_peer_acc[o]) return fail(CLIPK_EINVAL, "null peer accumulator %d", o);
            if ((rc = tmap_out_f32(&peers.map[o], static_cast<const float*>(dY_peer_acc[o]), rows_per_rank, d, d))) return rc;
        }
        peers.world = world;
        peers.rows_per_rank = rows_per_rank;
        dY_acc = static_cast<float*>(dY_peer_acc[0]);   // only marks "dY wanted" below; job 1 never writes through it
    }
    if (g_dtype != CLIPK_F16 && g_dtype != CLIPK_F16X2) return fail(CLIPK_EUNSUPPORTED, "g_dtype must be CLIPK_F16 or CLIPK_F16X2");
    if ((rc = check_common(Xg, Yg, rows, cols, d, ldxg, ldyg, g_dtype))) return rc;
    if (!logit_scale || !lse_row || !lse_col || !gscale || !workspace) return fail(CLIPK_EINVAL, "null pointer argument");
    if (!dX_acc && !dY_acc) return fail(CLIPK_EINVAL, "nothing to compute: dX_acc and dY_acc are both NULL");
    if (workspace_bytes < clipk_bwd_workspace_bytes(rows, cols, d, g_dtype)) return fail(CLIPK_EWORKSPACE, "workspace too small");
    if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) return fail(CLIPK_EINVAL, "workspace must be 256-byte aligned");
    DevInfo di;
    if ((rc = device_info(&di))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);

    const int planes = planes_of(dtype);                // S-GEMM operand planes
    const int fplanes = planes_of(g_dtype);             // planes of the gradient-GEMM features
    if (split_row_col && fplanes != 1) return fail(CLIPK_EUNSUPPORTED, "split_row_col needs one-plane (CLIPK_F16) gradient operands");
    const int gplanes = split_row_col ? 2 : fplanes;    // planes of G: [hi | lo] with two-plane features, [row | col] when split
    const long long dpad = round_up(d, BK);
    const long long kext = (dtype == CLIPK_BF16) ? d : planes * dpad;   // inner extent of X / Y rows
    const long long gext = fplanes * dpad;                              // inner extent of Xg / Yg rows
    long long rp_max, cp_max;
    choose_panel(rows, cols, d, gplanes, di.sms, panel_budget_for(rows, cols, gplanes), &rp_max, &cp_max, peers.world > 0 ? 1 : 0);
    const int ncp = int(cp_max);                        // panel width (multiple of BN) = G plane stride
    const int ldg = gplanes * ncp;
    if ((unsigned long long)round_up(rp_max, 2 * BM) * ldg * 2 > workspace_bytes) return fail(CLIPK_EWORKSPACE, "panel does not fit the workspace");
    __half* G = static_cast<__half*>(workspace);
    // after the panel(s): avec[rows], bvec[cols], gref[2], minmax[2]
    const size_t g_bytes = size_t(round_up(round_up(rp_max, 2 * BM) * ldg * 2, 256));
    const int n_gbuf = 1;
    float* avec = reinterpret_cast<float*>(static_cast<char*>(workspace) + n_gbuf * g_bytes);
    float* bvec = avec + round_up(rows, 64);
    float* gref = bvec + round_up(cols, 64);
    int* mm = reinterpret_cast<int*>(gref + 4);
    if (n_gbuf * g_bytes + (round_up(rows, 64) + round_up(cols, 64) + 8) * sizeof(float) > workspace_bytes)
        return fail(CLIPK_EWORKSPACE, "workspace too small for the panel and the reference vectors");
    {
        const int* mm_src = mm_ready;
        if (!mm_src) {
            CK_CUDA(cudaMemsetAsync(mm, 0x7f, sizeof(int), st));
            CK_CUDA(cudaMemsetAsync(mm + 1, 0x80, sizeof(int), st));
            const int n = rows + cols;
            int blocks = cdiv(n, 256);
            if (blocks > 4 * di.sms) blocks = 4 * di.sms;
            lse_minmax_kernel<<<blocks, 256, 0, st>>>(lse_row, rows, lse_col, cols, mm);
            count_launch("lse_minmax_kernel", st);
            mm_src = mm;
        }
        const int m = rows > cols ? rows : cols;
        grad_prep_kernel<<<cdiv(m, 256), 256, 0, st>>>(lse_row, rows, lse_col, cols, mm_src, avec, bvec, gref);
        count_launch("grad_prep_kernel", st);
        CK_CUDA(cudaGetLastError());
    }
    const size_t esz = 2;
    const char* Xb = static_cast<const char*>(X);
    const char* Yb = static_cast<const char*>(Y);
    const char* Xgb = static_cast<const char*>(Xg);
    const char* Ygb = static_cast<const char*>(Yg);
    const int nt = cdiv(d, BN);

    for (long long r0 = 0; r0 < rows; r0 += rp_max) {
        const int nr = int(rows - r0 < rp_max ? rows - r0 : rp_max);
        for (long long c0 = 0; c0 < cols; c0 += cp_max) {
            const int nc = int(cols - c0 < cp_max ? cols - c0 : cp_max);
            __half* const Gp = G;
            const cudaStream_t sg = st;
            // ---- recompute S on the panel, write G (fp16, x 2^14)
            {
                CUtensorMap ta, tb, tc;
                if ((rc = tmap_kmajor(&ta, Xb + r0 * ldx * esz, nr, kext, ldx, BM))) return rc;
                if ((rc = tmap_kmajor(&tb, Yb + c0 * ldy * esz, nc, kext, ldy, BN / 2))) return rc;
                if ((rc = tmap_g_store(&tc, Gp, round_up(nr, 2 * BM), ldg, ldg))) return rc;
                KArgs a{};
                a.M = nr; a.N = nc; a.n_tiles = cdiv(nc, BN);
                set_segments(a, planes, d, dpad, dpad);
                const int m_pairs = cdiv(nr, 2 * BM);
                const int split = choose_split(m_pairs, a.n_tiles, di.sms);
                a.tiles_per_unit = cdiv(a.n_tiles, split);
                const int units = cdiv(a.n_tiles, a.tiles_per_unit);
                a.scale = logit_scale; a.xs = x_inv_scale; a.ys = y_inv_scale;
                a.diag_offset = diag_offset + r0 - c0;
                a.lse_row = lse_row + r0; a.lse_col = lse_col + c0;
                a.alpha = alpha; a.beta = beta;
                a.avec = avec + r0; a.bvec = bvec + c0; a.gref = gref;
                a.G = Gp; a.ldg = ldg; a.g_planes = gplanes; a.g_plane_stride = ncp; a.g_split = split_row_col ? 1 : 0;
                if (planes == 1 && gplanes == 1 && a.num_kb <= ARES_KB) {
                    // rows of X resident in shared memory, persistent over the panel (see grad_sweep_kernel)
                    SweepGeom g{};
                    g.num_kb = a.num_kb; g.n_tiles = a.n_tiles; g.m_pairs = m_pairs;
                    const int nc = int(std::min<long long>(di.sms / 2, (long long)m_pairs * a.n_tiles));
                    if ((rc = tmap_g_store_dense32(&tc, Gp, round_up(nr, 2 * BM), ldg, ldg))) return rc;
                    rc = is_f16(dtype) ? launch_grad_sweep<1>(ta, tb, tc, a, g, nc, sg) : launch_grad_sweep<0>(ta, tb, tc, a, g, nc, sg);
                } else if (is_f16(dtype)) {
                    rc = launch_gemm<MODE_GRAD, 1>(ta, tb, tc, a, units, m_pairs, sg);
                } else {
                    rc = launch_gemm<MODE_GRAD, 0>(ta, tb, tc, a, units, m_pairs, sg);
                }
                if (rc) return rc;
            }
            // ---- job 0: dX[r0:r0+nr, :] (+)= G[nr, nc] * Yg[c0:c0+nc, :]      (A K-major, B MN-major, fp16 x fp16)
            // ---- job 1: dY[c0:c0+nc, :] (+)= G^T[nc, nr] * Xg[r0:r0+nr, :]    (A MN-major, B MN-major, fp16 x fp16)
            CUtensorMap ta0, tb0, tc0, ta1, tb1, tc1;
            KArgs a0{}, a1{};
            int jobs0 = 0, jobs1 = 0;
            if (dX_acc) {
                // dX reads plane 0 of a split panel (the row part); [hi | lo] panels are read across both planes
                if ((rc = tmap_kmajor(&ta0, Gp, nr, fplanes == 2 ? ldg : nc, ldg, BM))) return rc;
                if ((rc = tmap_mnmajor(&tb0, Ygb + c0 * ldyg * esz, gext, nc, ldyg))) return rc;
                if ((rc = tmap_out_f32(&tc0, dX_acc + r0 * d, nr, d, d))) return rc;
                a0.M = nr; a0.N = d; a0.n_tiles = nt; a0.tiles_per_unit = 1; a0.a_mn = 0; a0.b_mn = 1;
                set_segments(a0, fplanes, nc, ncp, dpad);
                a0.out = dX_acc + r0 * d; a0.ldo = d; a0.accumulate = (c0 > 0);
                a0.oscale0 = logit_scale; a0.oscale1 = gscale; a0.oscale2 = yg_inv_scale; a0.oconst = coef / 16384.f;
                jobs0 = cdiv(nr, 2 * BM) * nt;
            }
            if (dY_acc) {
                if ((rc = tmap_mnmajor(&ta1, Gp, gplanes == 2 ? ldg : nc, nr, ldg))) return rc;
                if ((rc = tmap_mnmajor(&tb1, Xgb + r0 * ldxg * esz, gext, nr, ldxg))) return rc;
                if ((rc = tmap_out_f32(&tc1, peers.world ? dY_acc : dY_acc + c0 * d, peers.world ? peers.rows_per_rank : nc, d, d))) return rc;
                a1.M = nc; a1.N = d; a1.n_tiles = nt; a1.tiles_per_unit = 1; a1.a_mn = 1; a1.b_mn = 1;
                set_segments(a1, fplanes, nr, ncp, dpad);
                if (split_row_col) a1.a_off[0] = ncp;       // dY reads plane 1 (the column part)
                a1.out = dY_acc + c0 * d; a1.ldo = d; a1.accumulate = (r0 > 0);
                if (peers.world) a1.c_row_off = int(c0);   // global dY row of the panel (owner = row / rows_per_rank)
                a1.oscale0 = logit_scale; a1.oscale1 = gscale; a1.oscale2 = xg_inv_scale; a1.oconst = coef / 16384.f;
                jobs1 = cdiv(nc, 2 * BM) * nt;
            }
            // One job (256 x 256 output tile, full K of the panel) per CTA pair, dispatched in order by the hardware.
            // Measured alternatives, all SLOWER although they even out the MMAs per SM pair - the tensor kernels run at
            // the power limit (SM clocks 1.55-1.65 GHz under ncu even for a single launch), so idle pairs lend their
            // budget to the busy ones and extra partial tiles cost energy: a stream-K split over the 74 pairs (round 1:
            // 2.94 vs 2.73 ms per backward at N = 32768); a persistent kernel walking a longest-first schedule with the
            // epilogue of one item under the MMAs of the next, unsplit / dX in pieces of 64 or 32 K blocks / both
            // outputs in pieces (round 2, profiles/r02c_scheduled_pair_kernel_ab.log: 1.97-2.13 vs 1.81 ms per step).
            if (dX_acc && dY_acc) rc = launch_pair(ta0, tb0, tc0, a0, jobs0, ta1, tb1, tc1, a1, jobs1, peers, st);
            else if (dX_acc) rc = launch_gemm<MODE_OUT, 1>(ta0, tb0, tc0, a0, nt, cdiv(nr, 2 * BM), st);
            else rc = launch_gemm<MODE_OUT, 1>(ta1, tb1, tc1, a1, nt, cdiv(nc, 2 * BM), st);
            if (rc) return rc;
        }
    }
    return CLIPK_OK;
}

int clipk_bwd(const void* X, const void* Y, int rows, int cols, int d, long long ldx, long long ldy, int dtype,
              const float* x_inv_scale, const float* y_inv_scale, const void* Xg, const void* Yg, long long ldxg,
              long long ldyg, int g_dtype, const float* xg_inv_scale, const float* yg_inv_scale,
              const float* logit_scale, long long diag_offset, const float* lse_row, const float* lse_col,
              float alpha, float beta, int split_row_col, const float* gscale, float* dX_acc, float* dY_acc, void* workspace,
              size_t workspace_bytes, void* stream) {
    return bwd_impl(X, Y, rows, cols, d, ldx, ldy, dtype, x_inv_scale, y_inv_scale, Xg, Yg, ldxg, ldyg, g_dtype,
                    xg_inv_scale, yg_inv_scale, logit_scale, diag_offset, lse_row, lse_col, alpha, beta, gscale, dX_acc,
                    dY_acc, nullptr, 0, 0, workspace, workspace_bytes, stream, nullptr, 1.f, split_row_col);
}

static int normalize_check(const void* a, const void* b, int dtype, long long rows, long long d, long long lda, long long ldb) {
    if (!a || !b || rows <= 0 || d <= 0) return fail(CLIPK_EINVAL, "bad argument");
    if (dtype != CLIPK_BF16 && dtype != CLIPK_F32) return fail(CLIPK_EUNSUPPORTED, "dtype %d", dtype);
    if (d % 8 != 0) return fail(CLIPK_EUNSUPPORTED, "d = %lld is not a multiple of 8", d);
    const int es = dtype == CLIPK_BF16 ? 2 : 4;
    if (lda < d || ldb < d || (lda * es) % 16 != 0 || (ldb * es) % 16 != 0 || (reinterpret_cast<uintptr_t>(a) & 15) != 0 ||
        (reinterpret_cast<uintptr_t>(b) & 15) != 0)
        return fail(CLIPK_EINVAL, "rows must be 16-byte aligned and at least d wide");
    return CLIPK_OK;
}

int clipk_normalize_fwd(const void* x, int dtype, long long rows, long long d, long long ldx, void* y, long long ldy,
                        float* inv_norm, float eps, void* stream) {
    int rc = normalize_check(x, y, dtype, rows, d, ldx, ldy);
    if (rc) return rc;
    if (!inv_norm) return fail(CLIPK_EINVAL, "null inv_norm");
    DevInfo di;
    if ((rc = device_info(&di))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int wpb = 8;
    if (dtype == CLIPK_BF16)
        normalize_fwd_kernel<<<cdiv(rows, wpb), wpb * 32, 0, st>>>(static_cast<const __nv_bfloat16*>(x), rows, int(d / 8), ldx,
                                                                    static_cast<__nv_bfloat16*>(y), ldy, inv_norm, eps);
    else
        normalize_fwd_kernel<<<cdiv(rows, wpb), wpb * 32, 0, st>>>(static_cast<const float*>(x), rows, int(d / 8), ldx,
                                                                    static_cast<float*>(y), ldy, inv_norm, eps);
    count_launch("normalize_fwd_kernel", st);
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}

int clipk_normalize_bwd(const void* g, long long ldg, const void* y, long long ldy, const float* inv_norm, int dtype,
                        long long rows, long long d, void* dx, long long ldd, float eps, void* stream) {
    int rc = normalize_check(g, y, dtype, rows, d, ldg, ldy);
    if (rc) return rc;
    if ((rc = normalize_check(dx, y, dtype, rows, d, ldd, ldy))) return rc;
    if (!inv_norm) return fail(CLIPK_EINVAL, "null inv_norm");
    DevInfo di;
    if ((rc = device_info(&di))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int wpb = 8;
    if (dtype == CLIPK_BF16)
        normalize_bwd_kernel<<<cdiv(rows, wpb), wpb * 32, 0, st>>>(static_cast<const __nv_bfloat16*>(g), ldg,
                                                                    static_cast<const __nv_bfloat16*>(y), ldy, inv_norm, rows,
                                                                    int(d / 8), static_cast<__nv_bfloat16*>(dx), ldd, eps);
    else
        normalize_bwd_kernel<<<cdiv(rows, wpb), wpb * 32, 0, st>>>(static_cast<const float*>(g), ldg, static_cast<const float*>(y),
                                                                    ldy, inv_norm, rows, int(d / 8), static_cast<float*>(dx), ldd, eps);
    count_launch("normalize_bwd_kernel", st);
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}

int clipk_rank_count(const float* S, int rows, int cols, long long ld, const long long* target, long long diag_offset,
                     long long row0, int* greater, int* ties_before, void* stream) {
    if (!S || !greater || rows < 0 || cols <= 0 || row0 < 0) return fail(CLIPK_EINVAL, "bad argument");
    if (ld < cols || ld % 4 != 0 || (reinterpret_cast<uintptr_t>(S) & 15) != 0)
        return fail(CLIPK_EINVAL, "ld must be >= cols and a multiple of 4, and S 16-byte aligned");
    DevInfo di;
    int rc = device_info(&di);
    if (rc) return rc;
    if (rows == 0) return CLIPK_OK;
    rank_count_kernel<<<rows, 256, 0, static_cast<cudaStream_t>(stream)>>>(S, ld, cols, target, diag_offset, row0, greater,
                                                                           ties_before);
    count_launch("rank_count_kernel", static_cast<cudaStream_t>(stream));
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}

int clipk_distill_cross(const float* S, const float* T, int rows, int cols, long long ld, const float* s_mul,
                        const float* t_mul, const float* t_lse_row, const float* t_lse_col, long long row0,
                        float* row_cross, float* col_part, void* stream) {
    if (!S || !T || !s_mul || !t_mul || !t_lse_row || !t_lse_col || !row_cross || !col_part)
        return fail(CLIPK_EINVAL, "null pointer argument");
    if (rows < 0 || rows > 65535 || cols <= 0 || ld < cols || row0 < 0) return fail(CLIPK_EINVAL, "bad extent");
    DevInfo di;
    int rc = device_info(&di);
    if (rc) return rc;
    if (rows == 0) return CLIPK_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    distill_row_cross_kernel<<<rows, 256, 0, st>>>(S, T, ld, cols, s_mul, t_mul, t_lse_row, row0, row_cross);
    count_launch("distill_row_cross_kernel", st);
    CK_CUDA(cudaGetLastError());
    distill_col_cross_kernel<<<cdiv(cols, 32), 256, 0, st>>>(S, T, rows, cols, ld, s_mul, t_mul, t_lse_col, col_part);
    count_launch("distill_col_cross_kernel", st);
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}

int clipk_distill_grad(const float* S, const float* T, int rows, int cols, long long ld, const float* s_mul,
                       const float* t_mul, const float* s_lse_row, const float* t_lse_row, const float* s_lse_col,
                       const float* t_lse_col, long long row0, void* G, long long ldg, void* stream) {
    if (!S || !T || !s_mul || !t_mul || !s_lse_row || !t_lse_row || !s_lse_col || !t_lse_col || !G)
        return fail(CLIPK_EINVAL, "null pointer argument");
    if (rows < 0 || rows > 65535 || cols <= 0 || ld < cols || ldg < cols || row0 < 0) return fail(CLIPK_EINVAL, "bad extent");
    DevInfo di;
    int rc = device_info(&di);
    if (rc) return rc;
    if (rows == 0) return CLIPK_OK;
    distill_grad_kernel<<<dim3(cdiv(cols, 256), rows), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        S, T, cols, ld, s_mul, t_mul, s_lse_row, t_lse_row, row0, s_lse_col, t_lse_col, static_cast<__half*>(G), ldg);
    count_launch("distill_grad_kernel", static_cast<cudaStream_t>(stream));
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}

// ---- the whole step (see include/clipk.h) ----------------------------------------------------------------------------
namespace {
struct StepCarve {
    size_t ticket, partials;                                 // persistent across calls: prep's ticket (0 at creation)
    size_t fwd, row_stats, pos, col_local, col_all;          // forward phase
    size_t xg, yg, inv2, dx, dy, bwd;                        // backward phase (overlays the forward's scratch)
    size_t total;
};
StepCarve step_carve(int rows, int cols, int d, int world) {
    StepCarve c{};
    auto take = [](size_t& off, size_t bytes) { const size_t o = off; off = size_t(round_up((long long)(off + bytes), 256)); return o; };
    size_t head = 0;
    c.ticket = take(head, 256);
    c.partials = take(head, size_t(PREP_MAX_BLOCKS) * 8 * sizeof(float));
    size_t f = head;
    c.fwd = take(f, fwd_carve(rows, cols).total);
    c.row_stats = take(f, size_t(3) * rows * sizeof(float));
    c.pos = take(f, size_t(rows) * sizeof(float));
    c.col_local = take(f, size_t(3) * cols * sizeof(float));
    c.col_all = take(f, world > 1 ? size_t(world) * 3 * cols * sizeof(float) : 0);
    const size_t dpad = size_t(round_up(d, BK));
    size_t b = head;
    c.xg = take(b, (size_t(rows) + cols) * dpad * 2 + 256);      // Xg | Yg | dequant scalars, one block (step_to_f16)
    c.yg = c.inv2 = c.xg;
    c.dx = take(b, size_t(rows) * d * sizeof(float));
    c.dy = take(b, world > 1 ? 0 : size_t(cols) * d * sizeof(float));
    c.bwd = take(b, clipk_bwd_workspace_bytes(rows, cols, d, CLIPK_F16));
    c.total = (f > b ? f : b) + 256;
    return c;
}
int step_check(const clipk_step* p, int* world, int* rank) {
    if (!p) return fail(CLIPK_EINVAL, "null step");
    const int W = p->peer ? p->peer->world : 1, r = p->peer ? p->peer->rank : 0;
    if (W < 1 || W > MAX_PEERS || r < 0 || r >= W) return fail(CLIPK_EINVAL, "world %d / rank %d out of range", W, r);
    if (p->rows <= 0 || p->d <= 0 || (long long)p->rows * W != p->cols) return fail(CLIPK_EINVAL, "cols must be world * rows");
    if (p->d % BK != 0) return fail(CLIPK_EUNSUPPORTED, "d = %d is not a multiple of 64", p->d);
    if (W > 1 && p->rows % BM != 0) return fail(CLIPK_EUNSUPPORTED, "with peers the local batch must be a multiple of 128");
    if (p->src_dtype != CLIPK_BF16 && p->src_dtype != CLIPK_F32) return fail(CLIPK_EUNSUPPORTED, "src_dtype %d", p->src_dtype);
    if (!p->image || !p->text || !p->logit_scale || !p->x_op || !p->y_all || !p->stats || !p->lse_row || !p->lse_col ||
        !p->scal || !p->workspace)
        return fail(CLIPK_EINVAL, "null pointer argument");
    if (p->normalize && (!p->inv_x || !p->inv_y)) return fail(CLIPK_EINVAL, "normalize needs inv_x and inv_y");
    const bool produced = p->normalize || p->src_dtype != CLIPK_BF16;
    if (produced && (p->x_op == p->image || p->y_all == p->text)) return fail(CLIPK_EINVAL, "x_op / y_all must be separate buffers when the operands are produced");
    if (!produced && p->x_op != p->image) return fail(CLIPK_EINVAL, "x_op must alias image when nothing is produced");
    if (W == 1 && !produced && p->y_all != p->text) return fail(CLIPK_EINVAL, "y_all must alias text when nothing is produced or gathered");
    const int es = p->src_dtype == CLIPK_BF16 ? 2 : 4;
    if (p->ld_image < p->d || p->ld_text < p->d || (p->ld_image * es) % 16 != 0 || (p->ld_text * es) % 16 != 0 ||
        (reinterpret_cast<uintptr_t>(p->image) & 15) != 0 || (reinterpret_cast<uintptr_t>(p->text) & 15) != 0)
        return fail(CLIPK_EINVAL, "input rows must be 16-byte aligned and at least d wide");
    if ((reinterpret_cast<uintptr_t>(p->workspace) & 255) != 0) return fail(CLIPK_EINVAL, "workspace must be 256-byte aligned");
    if (p->workspace_bytes < step_carve(p->rows, p->cols, p->d, W).total) return fail(CLIPK_EWORKSPACE, "workspace too small");
    if (!(p->loss_div > 0.f)) return fail(CLIPK_EINVAL, "loss_div must be positive");
    *world = W; *rank = r;
    return CLIPK_OK;
}
int launch_allgather(const GatherArgs& g, int sms, cudaStream_t st) {
    // enough 16-byte loads in flight to cover the NVLink round trip at full rate: ~160 blocks of 256 threads x 4 loads
    long long bx = cdiv(g.n16_0, 256 * 4);
    const long long want = std::max(4, 160 / g.world);
    if (bx > want) bx = want;
    if (bx < 1) bx = 1;
    (void)sms;
    peer_allgather_kernel<<<dim3(unsigned(bx), unsigned(g.world)), 256, 0, st>>>(g);
    count_launch("peer_allgather_kernel", st);
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}
}  // namespace

// exact fp16 copies of both operands for the gradient GEMMs: buf = Xg [rows, d] | Yg [cols, d] | 64 floats (2 dequant scalars)
static int step_to_f16(const clipk_step* p, int W, int rank, __half* buf, cudaStream_t st) {
    const int rows = p->rows, cols = p->cols, d = p->d;
    const long long ldx = (p->x_op == p->image) ? p->ld_image : d;
    const long long ldy = (W == 1 && p->y_all == p->text) ? p->ld_text : d;
    const long long dpad = round_up(d, BK);
    __half* Xg = buf;
    __half* Yg = buf + (size_t)rows * dpad;
    float* inv2 = reinterpret_cast<float*>(Yg + (size_t)cols * dpad);
    const long long n8 = ((long long)rows + cols) * (dpad / 8);
    to_f16_pair_kernel<<<cdiv(n8, 256), 256, 0, st>>>(static_cast<const __nv_bfloat16*>(p->x_op), rows, ldx, Xg,
                                                      static_cast<const __nv_bfloat16*>(p->y_all), cols, ldy, Yg, d, dpad,
                                                      p->stats, W, rank, inv2);
    count_launch("to_f16_pair_kernel", st);
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}

size_t clipk_step_workspace_bytes(const clipk_step* p) {
    if (!p || p->rows <= 0 || p->cols <= 0 || p->d <= 0) return 0;
    return step_carve(p->rows, p->cols, p->d, p->peer ? p->peer->world : 1).total;
}

int clipk_step_forward(const clipk_step* p) {
    int W = 1, rank = 0, rc;
    if ((rc = step_check(p, &W, &rank))) return rc;
    DevInfo di;
    if ((rc = device_info(&di))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(p->stream);
    const clipk_peer* pr = p->peer;
    const int rows = p->rows, cols = p->cols, d = p->d;
    const StepCarve cv = step_carve(rows, cols, d, W);
    char* ws = static_cast<char*>(p->workspace);
    float* row_stats = reinterpret_cast<float*>(ws + cv.row_stats);
    float* pos = reinterpret_cast<float*>(ws + cv.pos);
    float* col_local = (W > 1) ? static_cast<float*>(pr->col_src[rank]) : reinterpret_cast<float*>(ws + cv.col_local);
    float* col_all = (W > 1) ? reinterpret_cast<float*>(ws + cv.col_all) : col_local;

    // 1. one pass over the local rows: operands, statistics; resets the accumulators of finalize
    float* my_stats = (W > 1) ? static_cast<float*>(pr->stats_src[rank]) : p->stats;
    PrepArgs pa{};
    pa.x = p->image; pa.y = p->text; pa.rows_x = rows; pa.rows_y = rows; pa.ldx = p->ld_image; pa.ldy = p->ld_text;
    pa.d8 = d / 8; pa.pair_off = 0;
    pa.x_out = (p->x_op != p->image) ? static_cast<__nv_bfloat16*>(p->x_op) : nullptr;
    if (W > 1) pa.y_out = static_cast<__nv_bfloat16*>(pr->text_src[rank]);
    else pa.y_out = (p->y_all != p->text) ? static_cast<__nv_bfloat16*>(p->y_all) : nullptr;
    pa.ldxo = d; pa.ldyo = d;
    pa.inv_x = p->inv_x; pa.inv_y = p->inv_y; pa.eps = p->eps;
    pa.stats = my_stats; pa.reset = p->scal;
    pa.ticket = reinterpret_cast<unsigned int*>(ws + cv.ticket);
    pa.partials = reinterpret_cast<float*>(ws + cv.partials);
    if ((rc = launch_prep(pa, p->src_dtype, p->normalize, di.sms, st))) return rc;

    // 2. all-gather of the text operand rows and of the statistics (gather_features, loss.py:20-64)
    if (W > 1) {
        GatherArgs g{};
        for (int o = 0; o < W; ++o) {
            if (!pr->text_src[o] || !pr->stats_src[o] || !pr->flags_gather[o]) return fail(CLIPK_EINVAL, "null peer pointer %d", o);
            g.src0.p[o] = pr->text_src[o]; g.src1.p[o] = pr->stats_src[o]; g.flags.p[o] = pr->flags_gather[o];
        }
        g.n16_0 = (long long)rows * d * 2 / 16; g.dst0 = static_cast<uint4*>(p->y_all);
        g.n16_1 = STAT_WORDS * sizeof(float) / 16; g.dst1 = reinterpret_cast<uint4*>(p->stats);
        g.rank = rank; g.world = W; g.epoch = pr->epoch_gather; g.err = pr->err; g.do_signal = 1;
        if ((rc = launch_allgather(g, di.sms, st))) return rc;
    }

    // 3. single-sweep forward over the [rows, cols] block + merge.  When the backward's operand conversion is to run
    //    under the statistics exchange, the merge kernel's last block already tells the peers that this rank's column
    //    statistics are complete.
    const long long off = (long long)rank * rows;
    const bool early_signal = W > 1 && p->g16;
    MergeSignal sig;
    memset(&sig, 0, sizeof(sig));
    if (early_signal) {
        for (int o = 0; o < W; ++o) {
            if (!pr->flags_stats[o]) return fail(CLIPK_EINVAL, "null peer pointer %d", o);
            sig.flags.p[o] = pr->flags_stats[o];
        }
        sig.ticket = reinterpret_cast<unsigned int*>(ws + cv.ticket) + 1;
        sig.rank = rank; sig.world = W; sig.epoch = pr->epoch_stats;
    }
    if ((rc = fwd_sweeps(p->x_op, p->y_all, rows, cols, d, p->x_op == p->image ? p->ld_image : d,
                         (W == 1 && p->y_all == p->text) ? p->ld_text : d, CLIPK_BF16, nullptr, nullptr, p->logit_scale, off,
                         row_stats, pos, col_local, p->stats, W, rank, 1, 0, ws + cv.fwd, di, st, early_signal ? &sig : nullptr)))
        return rc;

    // 4. the column statistics of every rank's block
    if (W > 1) {
        GatherArgs g{};
        for (int o = 0; o < W; ++o) {
            if (!pr->col_src[o] || !pr->flags_stats[o]) return fail(CLIPK_EINVAL, "null peer pointer %d", o);
            g.src0.p[o] = pr->col_src[o]; g.flags.p[o] = pr->flags_stats[o];
        }
        g.n16_0 = (long long)3 * cols * sizeof(float) / 16; g.dst0 = reinterpret_cast<uint4*>(col_all);
        g.n16_1 = 0;
        g.rank = rank; g.world = W; g.epoch = pr->epoch_stats; g.err = pr->err; g.do_signal = 1;
        if (early_signal) {
            // the peers were told by the merge kernel; the fp16 copies for the gradient GEMMs are made while their
            // statistics are on the way
            g.do_signal = 0;
            if ((rc = step_to_f16(p, W, rank, static_cast<__half*>(p->g16), st))) return rc;
        }
        if ((rc = launch_allgather(g, di.sms, st))) return rc;
    }

    // 5. log-sum-exps, cross-entropy sums, loss
    const int n = rows > cols ? rows : cols;
    finalize_kernel<<<cdiv(n, 256), 256, 0, st>>>(row_stats, row_stats + rows, row_stats + 2 * (size_t)rows, pos, rows, col_all,
                                                  col_all + cols, col_all + 2 * (size_t)cols, W, (long long)3 * cols, cols, off,
                                                  p->lse_row, p->lse_col, p->scal, reinterpret_cast<int*>(p->scal) + 8,
                                                  p->loss_div);
    count_launch("finalize_kernel", st);
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}

int clipk_step_backward(const clipk_step* p) {
    int W = 1, rank = 0, rc;
    if ((rc = step_check(p, &W, &rank))) return rc;
    if (!p->grad_out) return fail(CLIPK_EINVAL, "null grad_out");
    if (p->out_dtype != CLIPK_BF16 && p->out_dtype != CLIPK_F32) return fail(CLIPK_EUNSUPPORTED, "out_dtype %d", p->out_dtype);
    DevInfo di;
    if ((rc = device_info(&di))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(p->stream);
    const clipk_peer* pr = p->peer;
    const int rows = p->rows, cols = p->cols, d = p->d;
    const StepCarve cv = step_carve(rows, cols, d, W);
    char* ws = static_cast<char*>(p->workspace);
    const long long ldx = (p->x_op == p->image) ? p->ld_image : d;
    const long long ldy = (W == 1 && p->y_all == p->text) ? p->ld_text : d;
    const long long off = (long long)rank * rows;
    const bool want_feat = p->d_image || p->d_text;
    if (want_feat) {
        if (!p->d_image || !p->d_text) return fail(CLIPK_EINVAL, "d_image and d_text must be given together");
        // 1. exact fp16 copies of both operands for the gradient GEMMs (already made by the forward when it had a wait
        //    to fill, see clipk_step_forward)
        const long long dpad = round_up(d, BK);
        __half* g16 = p->g16 ? static_cast<__half*>(p->g16) : reinterpret_cast<__half*>(ws + cv.xg);
        if (!(p->g16 && W > 1) && (rc = step_to_f16(p, W, rank, g16, st))) return rc;
        __half* Xg = g16;
        __half* Yg = g16 + (size_t)rows * dpad;
        float* inv2 = reinterpret_cast<float*>(Yg + (size_t)cols * dpad);
        // 2. recompute + gradient GEMMs, panel by panel; with peers the dY tiles go straight to their owners
        float* dX = reinterpret_cast<float*>(ws + cv.dx);
        float* dY = (W > 1) ? nullptr : reinterpret_cast<float*>(ws + cv.dy);
        void* slots[MAX_PEERS];
        if (W > 1)
            for (int o = 0; o < W; ++o) {
                if (!pr->grad_slot[o] || !pr->flags_grad[o]) return fail(CLIPK_EINVAL, "null peer pointer %d", o);
                slots[o] = pr->grad_slot[o];
            }
        if ((rc = bwd_impl(p->x_op, p->y_all, rows, cols, d, ldx, ldy, CLIPK_BF16, nullptr, nullptr, Xg, Yg, dpad, dpad, CLIPK_F16,
                           inv2, inv2 + 1, p->logit_scale, off, p->lse_row, p->lse_col, 1.f, 1.f, p->grad_out, dX, dY,
                           W > 1 ? slots : nullptr, W, rows, ws + cv.bwd, clipk_bwd_workspace_bytes(rows, cols, d, CLIPK_F16),
                           p->stream, reinterpret_cast<const int*>(p->scal) + 8, p->grad_coef, p->grad_split)))
            return rc;
        // 3. every rank's tiles have landed in the slots this rank owns
        if (W > 1) {
            PeerPtrs pf;
            memset(&pf, 0, sizeof(pf));
            for (int o = 0; o < W; ++o) pf.p[o] = pr->flags_grad[o];
            peer_barrier_kernel<<<1, 32, 0, st>>>(pf, rank, W, pr->epoch_grad, pr->err);
            count_launch("peer_barrier_kernel", st);
            CK_CUDA(cudaGetLastError());
        }
        // 4. slots -> text gradient, Jacobian of the normalisation, cast, dlogit_scale
        FinishArgs fa{};
        fa.gx = dX; fa.rows_x = rows;
        fa.gy = (W > 1) ? pr->my_slots : dY; fa.rows_y = rows;
        fa.slots = W; fa.slot_stride = (long long)rows * d;
        fa.d8 = d / 8;
        if (p->normalize) {
            fa.xn = static_cast<const __nv_bfloat16*>(p->x_op); fa.ldxn = ldx;
            // this rank's own rows of the gathered text operand
            fa.yn = static_cast<const __nv_bfloat16*>(p->y_all) + off * ldy; fa.ldyn = ldy;
            fa.inv_x = p->inv_x; fa.inv_y = p->inv_y; fa.eps = p->eps;
        }
        fa.out_x = p->d_image; fa.out_y = p->d_text; fa.out_dtype = p->out_dtype;
        fa.pair = p->scal + 4; fa.go = p->grad_out; fa.scale = p->logit_scale; fa.dscale = p->d_scale;
        const int wpb = 8;
        const int blocks = int(std::max<long long>(1, std::min<long long>(cdiv(2LL * rows, wpb), 8LL * di.sms)));
        finish_grad_kernel<<<blocks, wpb * 32, 0, st>>>(fa);
        count_launch("finish_grad_kernel", st);
        CK_CUDA(cudaGetLastError());
    } else if (p->d_scale) {
        FinishArgs fa{};
        fa.pair = p->scal + 4; fa.go = p->grad_out; fa.scale = p->logit_scale; fa.dscale = p->d_scale;
        finish_grad_kernel<<<1, 32, 0, st>>>(fa);
        count_launch("finish_grad_kernel", st);
        CK_CUDA(cudaGetLastError());
    }
    return CLIPK_OK;
}

// ---- SigLipLoss (see include/clipk.h) ---------------------------------------------------------------------------------
namespace {
struct SigCarve {
    size_t part_a, part_b, pos, row_a, row_b, scale_io, xg, yg, g, total;
    long long g_bytes;
};
SigCarve sig_carve(int rows, int cols, int d) {
    SigCarve c{};
    auto take = [](size_t& off, size_t bytes) { const size_t o = off; off = size_t(round_up((long long)(off + bytes), 256)); return o; };
    // sweep_parts_bound(n) * n <= 32768 + 2n for every row count n: the slots of the forward and of any row panel
    const size_t parts = size_t(PARTS_PER_UNIT) * (32768 + 2 * size_t(rows)) * sizeof(float);
    size_t off = 0;
    c.part_a = take(off, parts);
    c.part_b = take(off, parts);
    c.pos = take(off, size_t(rows) * sizeof(float));
    c.row_a = take(off, size_t(rows) * sizeof(float));
    c.row_b = take(off, size_t(rows) * sizeof(float));
    c.scale_io = take(off, 4 * sizeof(float));
    c.xg = take(off, size_t(rows) * d * 2);
    c.yg = take(off, size_t(cols) * d * 2);
    c.g_bytes = std::min(SIG_PANEL_BYTES, round_up(rows, 2 * BM) * round_up(cols, BN) * 2);
    c.g = take(off, size_t(c.g_bytes));
    c.total = off;
    return c;
}
int sig_check(const clipk_siglip* p) {
    if (!p) return fail(CLIPK_EINVAL, "null argument");
    if (p->rows <= 0 || p->cols <= 0 || p->d <= 0) return fail(CLIPK_EINVAL, "rows, cols and d must be positive");
    if (p->d % BK != 0) return fail(CLIPK_EUNSUPPORTED, "d = %d is not a multiple of 64", p->d);
    if (p->diag_offset < 0 || p->diag_offset + p->rows > p->cols) return fail(CLIPK_EINVAL, "the positives must be columns of the block");
    if (!p->x || !p->y || !p->logit_scale || !p->state || !p->workspace) return fail(CLIPK_EINVAL, "null pointer argument");
    if (p->ldx < p->d || p->ldy < p->d || (p->ldx * 2) % 16 != 0 || (p->ldy * 2) % 16 != 0 ||
        (reinterpret_cast<uintptr_t>(p->x) & 15) != 0 || (reinterpret_cast<uintptr_t>(p->y) & 15) != 0)
        return fail(CLIPK_EINVAL, "feature rows must be 16-byte aligned and at least d wide");
    if ((reinterpret_cast<uintptr_t>(p->workspace) & 255) != 0) return fail(CLIPK_EINVAL, "workspace must be 256-byte aligned");
    if (p->workspace_bytes < sig_carve(p->rows, p->cols, p->d).total) return fail(CLIPK_EWORKSPACE, "workspace too small");
    return CLIPK_OK;
}
}  // namespace

size_t clipk_siglip_workspace_bytes(const clipk_siglip* p) {
    if (!p || p->rows <= 0 || p->cols <= 0 || p->d <= 0) return 0;
    return sig_carve(p->rows, p->cols, p->d).total;
}

int clipk_siglip_forward(const clipk_siglip* p) {
    int rc;
    if ((rc = sig_check(p))) return rc;
    DevInfo di;
    if ((rc = device_info(&di))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(p->stream);
    const int rows = p->rows, cols = p->cols, d = p->d;
    const SigCarve cv = sig_carve(rows, cols, d);
    char* ws = static_cast<char*>(p->workspace);
    CUtensorMap ta, tb;
    if ((rc = tmap_kmajor(&ta, p->x, rows, d, p->ldx, BM))) return rc;
    if ((rc = tmap_kmajor(&tb, p->y, cols, d, p->ldy, BN / 2))) return rc;
    SweepGeom g{};
    g.num_kb = d / BK; g.n_tiles = cdiv(cols, BN); g.m_pairs = cdiv(rows, 2 * BM);
    const int nc = int(std::min<long long>(di.sms / 2, (long long)g.m_pairs * g.n_tiles));
    SigArgs a{};
    a.M = rows; a.N = cols; a.scale = p->logit_scale; a.bias = p->logit_bias; a.diag_offset = p->diag_offset;
    a.part_a = reinterpret_cast<float*>(ws + cv.part_a); a.part_b = reinterpret_cast<float*>(ws + cv.part_b);
    a.pos = reinterpret_cast<float*>(ws + cv.pos);
    rc = g.num_kb <= ARES_KB ? launch_sig_fwd<true>(ta, tb, a, g, nc, st) : launch_sig_fwd<false>(ta, tb, a, g, nc, st);
    if (rc) return rc;
    float* row_a = reinterpret_cast<float*>(ws + cv.row_a);
    float* row_b = reinterpret_cast<float*>(ws + cv.row_b);
    siglip_rows_kernel<<<cdiv(rows, 256), 256, 0, st>>>(a.part_a, a.part_b, rows, g, nc, 1, 0, row_a, row_b);
    count_launch("siglip_rows_kernel", st);
    siglip_reduce_kernel<<<1, 1024, 0, st>>>(row_a, row_b, a.pos, rows, p->state, nullptr, nullptr, nullptr);
    count_launch("siglip_reduce_kernel", st);
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}

int clipk_siglip_backward(const clipk_siglip* p) {
    int rc;
    if ((rc = sig_check(p))) return rc;
    if (!p->grad_out) return fail(CLIPK_EINVAL, "null grad_out");
    const bool want_feat = p->d_x || p->d_y;
    if (!want_feat && !p->d_scale && !p->d_bias) return CLIPK_OK;
    DevInfo di;
    if ((rc = device_info(&di))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(p->stream);
    const int rows = p->rows, cols = p->cols, d = p->d;
    const SigCarve cv = sig_carve(rows, cols, d);
    char* ws = static_cast<char*>(p->workspace);
    float* state = p->state;
    siglip_bwd_prep_kernel<<<1, 1, 0, st>>>(state, p->grad_out, p->logit_scale, rows);
    count_launch("siglip_bwd_prep_kernel", st);
    CK_CUDA(cudaGetLastError());
    // exact fp16 copies of both operands for the gradient GEMMs (fp16 x fp16: the G panel needs fp16's mantissa)
    __half* Xg = reinterpret_cast<__half*>(ws + cv.xg);
    __half* Yg = reinterpret_cast<__half*>(ws + cv.yg);
    float* scale_io = reinterpret_cast<float*>(ws + cv.scale_io);     // [0..1] of Xg, [2..3] of Yg; [1], [3] = inv_scale
    if (want_feat) {
        if ((rc = to_f16_impl(p->x, CLIPK_BF16, rows, d, p->ldx, Xg, 1, d, scale_io, nullptr, p->stream))) return rc;
        if ((rc = to_f16_impl(p->y, CLIPK_BF16, cols, d, p->ldy, Yg, 1, d, scale_io + 2, nullptr, p->stream))) return rc;
    }
    long long rp, cp;
    choose_panel(rows, cols, d, 1, di.sms, cv.g_bytes, &rp, &cp);
    if (round_up(rp, 2 * BM) * cp * 2 > cv.g_bytes) return fail(CLIPK_EWORKSPACE, "panel does not fit the workspace");
    __half* G = reinterpret_cast<__half*>(ws + cv.g);
    float* part_a = reinterpret_cast<float*>(ws + cv.part_a);
    float* part_b = reinterpret_cast<float*>(ws + cv.part_b);
    float* row_a = reinterpret_cast<float*>(ws + cv.row_a);
    float* row_b = reinterpret_cast<float*>(ws + cv.row_b);
    const char* Xb = static_cast<const char*>(p->x);
    const char* Yb = static_cast<const char*>(p->y);
    const int nt = cdiv(d, BN), num_kb = d / BK;
    PeerOut no_peers;
    memset(&no_peers, 0, sizeof(no_peers));
    for (long long r0 = 0; r0 < rows; r0 += rp) {
        const int nr = int(std::min<long long>(rows - r0, rp));
        for (long long c0 = 0; c0 < cols; c0 += cp) {
            const int nc = int(std::min<long long>(cols - c0, cp));
            // ---- recompute the panel: G = fp16(g * 2^e), row sums of g and g x.y
            CUtensorMap ta, tb, tc;
            if ((rc = tmap_kmajor(&ta, Xb + r0 * p->ldx * 2, nr, d, p->ldx, BM))) return rc;
            if ((rc = tmap_kmajor(&tb, Yb + c0 * p->ldy * 2, nc, d, p->ldy, BN / 2))) return rc;
            if ((rc = tmap_g_store_dense32(&tc, G, round_up(nr, 2 * BM), cp, cp))) return rc;
            SigArgs a{};
            a.M = nr; a.N = nc; a.scale = p->logit_scale; a.bias = p->logit_bias; a.diag_offset = p->diag_offset + r0 - c0;
            a.part_a = part_a; a.part_b = part_b; a.p2e = state + SIG_P2E;
            SweepGeom g{};
            g.num_kb = num_kb; g.n_tiles = cdiv(nc, BN); g.m_pairs = cdiv(nr, 2 * BM);
            const int ncl = int(std::min<long long>(di.sms / 2, (long long)g.m_pairs * g.n_tiles));
            rc = num_kb <= ARES_KB ? launch_sig_grad<true>(ta, tb, tc, a, g, ncl, st) : launch_sig_grad<false>(ta, tb, tc, a, g, ncl, st);
            if (rc) return rc;
            siglip_rows_kernel<<<cdiv(nr, 256), 256, 0, st>>>(part_a, part_b, nr, g, ncl, 0, c0 > 0 ? 1 : 0, row_a + r0, row_b + r0);
            count_launch("siglip_rows_kernel", st);
            CK_CUDA(cudaGetLastError());
            if (!want_feat) continue;
            // ---- job 0: d_x[r0:r0+nr] (+)= G Yg[c0:c0+nc];  job 1: d_y[c0:c0+nc] (+)= G^T Xg[r0:r0+nr];
            //      scaled by go * s / (b * 2^e) (state) and the fp16 copy's inverse scale
            CUtensorMap ta0, tb0, tc0, ta1, tb1, tc1;
            KArgs a0{}, a1{};
            int jobs0 = 0, jobs1 = 0;
            if (p->d_x) {
                if ((rc = tmap_kmajor(&ta0, G, nr, nc, cp, BM))) return rc;
                if ((rc = tmap_mnmajor(&tb0, Yg + c0 * d, d, nc, d))) return rc;
                if ((rc = tmap_out_f32(&tc0, p->d_x + r0 * d, nr, d, d))) return rc;
                a0.M = nr; a0.N = d; a0.n_tiles = nt; a0.tiles_per_unit = 1; a0.a_mn = 0; a0.b_mn = 1;
                set_segments(a0, 1, nc, cp, d);
                a0.out = p->d_x + r0 * d; a0.ldo = d; a0.accumulate = c0 > 0 ? 1 : 0;
                a0.oscale0 = state + SIG_OSCALE; a0.oscale1 = scale_io + 3; a0.oconst = 1.f;
                jobs0 = cdiv(nr, 2 * BM) * nt;
            }
            if (p->d_y) {
                if ((rc = tmap_mnmajor(&ta1, G, nc, nr, cp))) return rc;
                if ((rc = tmap_mnmajor(&tb1, Xg + r0 * d, d, nr, d))) return rc;
                if ((rc = tmap_out_f32(&tc1, p->d_y + c0 * d, nc, d, d))) return rc;
                a1.M = nc; a1.N = d; a1.n_tiles = nt; a1.tiles_per_unit = 1; a1.a_mn = 1; a1.b_mn = 1;
                set_segments(a1, 1, nr, cp, d);
                a1.out = p->d_y + c0 * d; a1.ldo = d; a1.accumulate = r0 > 0 ? 1 : 0;
                a1.oscale0 = state + SIG_OSCALE; a1.oscale1 = scale_io + 1; a1.oconst = 1.f;
                jobs1 = cdiv(nc, 2 * BM) * nt;
            }
            if (p->d_x && p->d_y) rc = launch_pair(ta0, tb0, tc0, a0, jobs0, ta1, tb1, tc1, a1, jobs1, no_peers, st);
            else if (p->d_x) rc = launch_gemm<MODE_OUT, 1>(ta0, tb0, tc0, a0, nt, cdiv(nr, 2 * BM), st);
            else rc = launch_gemm<MODE_OUT, 1>(ta1, tb1, tc1, a1, nt, cdiv(nc, 2 * BM), st);
            if (rc) return rc;
        }
    }
    if (p->d_scale || p->d_bias) {
        siglip_reduce_kernel<<<1, 1024, 0, st>>>(row_a, row_b, nullptr, rows, state, p->grad_out, p->d_scale, p->d_bias);
        count_launch("siglip_reduce_kernel", st);
        CK_CUDA(cudaGetLastError());
    }
    return CLIPK_OK;
}

int clipk_bwd_panel(int rows, int cols, int d, long long* panel_rows, long long* panel_cols) {
    if (rows <= 0 || cols <= 0 || d <= 0 || !panel_rows || !panel_cols) return fail(CLIPK_EINVAL, "bad argument");
    DevInfo di;
    int rc = device_info(&di);
    if (rc) return rc;
    choose_panel(rows, cols, d, 1, di.sms, panel_budget_for(rows, cols, 1), panel_rows, panel_cols);
    return CLIPK_OK;
}

int clipk_profile_begin(void* stream) {
    if (g_prof_on.load()) return fail(CLIPK_EINVAL, "profile already running");
    for (ProfEntry& e : g_prof) cudaEventDestroy(e.ev);
    g_prof.clear();
    cudaEvent_t ev;
    CK_CUDA(cudaEventCreate(&ev));
    CK_CUDA(cudaEventRecord(ev, static_cast<cudaStream_t>(stream)));
    g_prof.push_back(ProfEntry{"", ev});
    g_prof_on.store(1);
    return CLIPK_OK;
}

int clipk_profile_end(char* out, size_t out_bytes) {
    if (!g_prof_on.load()) return fail(CLIPK_EINVAL, "no profile running");
    g_prof_on.store(0);
    if (!out || out_bytes < 64) return fail(CLIPK_EINVAL, "output buffer too small");
    if (!g_prof.empty()) CK_CUDA(cudaEventSynchronize(g_prof.back().ev));
    struct Agg { const char* name; int n; double ms; };
    std::vector<Agg> agg;
    for (size_t i = 1; i < g_prof.size(); ++i) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, g_prof[i - 1].ev, g_prof[i].ev) != cudaSuccess) ms = 0.f;
        bool found = false;
        for (Agg& a : agg)
            if (strcmp(a.name, g_prof[i].name) == 0) { a.n += 1; a.ms += ms; found = true; break; }
        if (!found) agg.push_back(Agg{g_prof[i].name, 1, ms});
    }
    size_t off = 0;
    out[0] = 0;
    for (const Agg& a : agg) {
        const int w = snprintf(out + off, out_bytes - off, "%s:%d:%.6f;", a.name, a.n, a.ms);
        if (w < 0 || size_t(w) >= out_bytes - off) break;
        off += size_t(w);
    }
    for (ProfEntry& e : g_prof) cudaEventDestroy(e.ev);
    g_prof.clear();
    return CLIPK_OK;
}

int clipk_debug_tmem_layout(int* out, void* stream) {
    if (!out) return fail(CLIPK_EINVAL, "null pointer");
    DevInfo di;
    int rc = device_info(&di);
    if (rc) return rc;
    tmem_layout_kernel<<<1, 128, 0, static_cast<cudaStream_t>(stream)>>>(out);
    count_launch("tmem_layout_kernel", static_cast<cudaStream_t>(stream));
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}

int clipk_cast(const float* src, void* dst, long long n, int dtype, void* stream) {
    if (!src || !dst || n < 0) return fail(CLIPK_EINVAL, "bad argument");
    if (dtype != CLIPK_BF16 && dtype != CLIPK_F32) return fail(CLIPK_EUNSUPPORTED, "dtype %d", dtype);
    if (n == 0) return CLIPK_OK;
    cast_kernel<<<cdiv(cdiv(n, 4), 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(src, dst, n, dtype);
    count_launch("cast_kernel", static_cast<cudaStream_t>(stream));
    CK_CUDA(cudaGetLastError());
    return CLIPK_OK;
}

int clipk_gemm16(const void* A, const void* B, float* D, int M, int N, int K, long long lda, long long ldb,
                 long long ldd, int a_mn, int b_mn, int f16, int accumulate, void* stream) {
    if (!A || !B || !D || M <= 0 || N <= 0 || K <= 0) return fail(CLIPK_EINVAL, "bad argument");
    if (N % 4 != 0 || ldd % 4 != 0) return fail(CLIPK_EUNSUPPORTED, "N and ldd must be multiples of 4");
    DevInfo di;
    int rc = device_info(&di);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CUtensorMap ta, tb, tc;
    if (a_mn) rc = tmap_mnmajor(&ta, A, M, K, lda); else rc = tmap_kmajor(&ta, A, M, K, lda, BM);
    if (rc) return rc;
    if (b_mn) rc = tmap_mnmajor(&tb, B, N, K, ldb); else rc = tmap_kmajor(&tb, B, N, K, ldb, BN / 2);
    if (rc) return rc;
    if ((rc = tmap_out_f32(&tc, D, M, N, ldd))) return rc;
    KArgs a{};
    a.M = M; a.N = N; a.n_tiles = cdiv(N, BN); a.tiles_per_unit = 1; a.a_mn = a_mn ? 1 : 0; a.b_mn = b_mn ? 1 : 0;
    set_segments(a, 1, K, 0, 0);
    a.out = D; a.ldo = int(ldd); a.accumulate = accumulate; a.oconst = 1.f;
    if (f16) return launch_gemm<MODE_OUT, 1>(ta, tb, tc, a, a.n_tiles, cdiv(M, 2 * BM), st);
    return launch_gemm<MODE_OUT, 0>(ta, tb, tc, a, a.n_tiles, cdiv(M, 2 * BM), st);
}

}  // extern "C"
