// monoloco_b200 -- tensor-core feasibility probe (tools/probe_tc.py; NOT on the product path).
//
// Question it answers on a real B200 (DESIGN.md "What comes next"): does an error-compensated TF32 product on the 5th-gen
// tensor cores stay inside the 1e-5 parity rule, i.e. how does tcgen05.mma round its fp32 accumulator?
//
//   D[128, 128] = A[128, K] . W[128, K]^T,   a = a_hi + a_lo,  w = w_hi + w_lo  (cvt.rna.tf32.f32 twice)
//   mode 0: a_hi.w_hi only (plain TF32)
//   mode 1: a_lo.w_hi + a_hi.w_lo + a_hi.w_hi into ONE TMEM accumulator
//   mode 2: a_hi.w_hi into the main accumulator, the two cross terms into a second one (returned separately)
//
// One CTA, 128 threads.  Per K block of 32: the threads split their rows into hi / lo TF32 planes and store them in the
// canonical K-major no-swizzle UMMA layout (core matrix = 8 rows x 16 B; SBO = 128 B between 8-row groups, LBO = rows x 16 B
// between 16-byte K chunks), fence.proxy.async, one thread issues the kind::tf32 MMAs (M = 128, N = 128, K = 8 each) and
// tcgen05.commit signals an mbarrier; the accumulators come back with tcgen05.ld 32x32b.x8.
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"
#include "host_error.h"

namespace mlb {

constexpr int PM = 128, PN = 128, PKB = 32;     // tile rows, tile columns, K per staged block
constexpr uint32_t P_SBO = 128;                  // bytes between 8-row groups
constexpr uint32_t P_LBO = PM * 16;              // bytes between 16-byte K chunks (PM == PN)

__device__ __forceinline__ float to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start >> 4 [0,14), LBO >> 4 [16,30), SBO >> 4 [32,46),
// version = 1 [46,48), base offset 0, layout type SWIZZLE_NONE [61,64)
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}

// instruction descriptor (cute::UMMA::InstrDescriptor): D = F32 [4,6), A = B = TF32 [7,10) [10,13), both K-major, N >> 3 [17,23),
// M >> 4 [24,29), dense, no negate
constexpr uint32_t P_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(PN >> 3) << 17) | ((uint32_t)(PM >> 4) << 24);

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(P_IDESC), "r"(accumulate), "r"(0u)
        : "memory");
}

__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// split one row's 32 values of a K block into TF32 hi / lo planes in the canonical layout
__device__ __forceinline__ void stage_row(const float* __restrict__ src, float* hi, float* lo, int row) {
#pragma unroll
    for (int c = 0; c < PKB / 4; ++c) {
        const float4 v = *reinterpret_cast<const float4*>(src + c * 4);
        const float4 h = make_float4(to_tf32(v.x), to_tf32(v.y), to_tf32(v.z), to_tf32(v.w));
        const float4 l = make_float4(to_tf32(v.x - h.x), to_tf32(v.y - h.y), to_tf32(v.z - h.z), to_tf32(v.w - h.w));
        const size_t off = ((size_t)c * P_LBO + (size_t)(row >> 3) * P_SBO + (size_t)(row & 7) * 16) / sizeof(float);
        *reinterpret_cast<float4*>(hi + off) = h;
        *reinterpret_cast<float4*>(lo + off) = l;
    }
}

__global__ void __launch_bounds__(128, 1) tc_probe_kernel(const float* __restrict__ A, const float* __restrict__ W, int K, int mode,
                                                          float* __restrict__ out_main, float* __restrict__ out_cross, int* err_flag) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    float* a_hi = reinterpret_cast<float*>(smem_raw);
    float* a_lo = a_hi + PM * PKB;
    float* w_hi = a_lo + PM * PKB;
    float* w_lo = w_hi + PN * PKB;
    __shared__ __align__(8) uint64_t mma_bar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5;

    if (tid == 0) {
        mbar_init(&mma_bar, 1);
        mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(&tmem_slot, 256);  // columns [0,128): main accumulator, [128,256): cross terms
    tmem_fence_before();
    __syncthreads();
    tmem_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t a_hi_s = smem_u32(a_hi), a_lo_s = smem_u32(a_lo), w_hi_s = smem_u32(w_hi), w_lo_s = smem_u32(w_lo);

    uint32_t main_started = 0, cross_started = 0;
    const int n_blocks = K / PKB;
    for (int kb = 0; kb < n_blocks; ++kb) {
        stage_row(A + (size_t)tid * K + (size_t)kb * PKB, a_hi, a_lo, tid);
        stage_row(W + (size_t)tid * K + (size_t)kb * PKB, w_hi, w_lo, tid);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy stores -> tensor-core (async proxy) reads
        __syncthreads();
        if (tid == 0) {
            tmem_fence_after();
#pragma unroll
            for (int j = 0; j < PKB / 8; ++j) {  // one K = 8 MMA step = two 16-byte chunks
                const uint32_t ko = (uint32_t)(2 * j) * P_LBO;
                const uint64_t ah = umma_desc(a_hi_s + ko, P_LBO, P_SBO), al = umma_desc(a_lo_s + ko, P_LBO, P_SBO);
                const uint64_t wh = umma_desc(w_hi_s + ko, P_LBO, P_SBO), wl = umma_desc(w_lo_s + ko, P_LBO, P_SBO);
                if (mode == 1) {
                    umma_tf32(tmem, al, wh, main_started), main_started = 1;
                    umma_tf32(tmem, ah, wl, 1u);
                } else if (mode == 2) {
                    umma_tf32(tmem + PN, al, wh, cross_started), cross_started = 1;
                    umma_tf32(tmem + PN, ah, wl, 1u);
                }
                umma_tf32(tmem, ah, wh, main_started), main_started = 1;
            }
            umma_commit(&mma_bar);  // arrives when every MMA issued so far has finished reading shared memory / writing TMEM
        }
        mbar_wait(&mma_bar, (uint32_t)(kb & 1), err_flag);
        tmem_fence_after();
    }
    // ---- accumulators -> global: warp w owns TMEM lanes (= rows) [32w, 32w + 32)
    const int row = tid;
    const uint32_t lane_base = tmem + ((uint32_t)(warp * 32) << 16);
    for (int c0 = 0; c0 < PN; c0 += 8) {
        float v[8];
        tmem_ld8(lane_base + (uint32_t)c0, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) out_main[(size_t)row * PN + c0 + j] = v[j];
        if (mode == 2 && out_cross != nullptr) {
            tmem_ld8(lane_base + (uint32_t)(PN + c0), v);
#pragma unroll
            for (int j = 0; j < 8; ++j) out_cross[(size_t)row * PN + c0 + j] = v[j];
        }
    }
    tmem_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}


// ================================================================================================================
// One whole layer on the tensor cores (round-2 candidate, timing probe):  Y[B, 1024] = X[B, 1024] . W[1024, 1024]^T
// ================================================================================================================
// Operands live in global memory already split into TF32 hi / lo planes in the canonical UMMA layout, one contiguous
// block per (row tile, k block): a stage is two 1-D TMA bulk copies, no tensor maps.
//   X planes: [B/128 row tiles][K/16 k blocks][hi | lo][128 rows x 16 k]   (8 KB per plane)
//   W planes: [N/256 col tiles][K/16 k blocks][hi | lo][256 rows x 16 k]   (16 KB per plane)
// CTA (row tile, col tile): 4-stage ring of 48 KB stages; warp 1 lane 0 streams the stages, warp 0 lane 0 issues per stage
// 2 k-steps x 3 kind::tf32 MMAs (M = 128, N = 256) into two TMEM accumulators (main: hi.hi, cross: lo.hi + hi.lo) and
// releases the stage with tcgen05.commit; all 128 threads read the accumulators back and store Y = main + cross.
constexpr int LM = 128, LN = 256, LKB = 16, LNST = 4;
constexpr uint32_t L_A_PLANE = LM * LKB * 4, L_W_PLANE = LN * LKB * 4;     // bytes
constexpr uint32_t L_STAGE = 2 * L_A_PLANE + 2 * L_W_PLANE;                  // 48 KB
constexpr uint32_t L_LBO_A = LM * 16, L_LBO_W = LN * 16;
constexpr uint32_t L_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(LN >> 3) << 17) | ((uint32_t)(LM >> 4) << 24);

__device__ __forceinline__ void umma_tf32_desc(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u)
        : "memory");
}

// row-major fp32 [rows][K] -> TF32 hi / lo planes, tiles of `tile_rows` rows, k blocks of 16
__global__ void tc_pack_planes_kernel(const float* __restrict__ src, float* __restrict__ dst, int rows, int K, int tile_rows) {
    const int kq = K / 4;
    const size_t plane = (size_t)tile_rows * LKB;  // floats per plane
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)rows * kq; i += (size_t)gridDim.x * blockDim.x) {
        const int row = (int)(i / kq), q = (int)(i % kq);
        const int tile = row / tile_rows, r = row % tile_rows, kb = (q * 4) / LKB, chunk = q % (LKB / 4);
        const float4 v = *reinterpret_cast<const float4*>(src + (size_t)row * K + (size_t)q * 4);
        const float4 h = make_float4(to_tf32(v.x), to_tf32(v.y), to_tf32(v.z), to_tf32(v.w));
        const float4 l = make_float4(to_tf32(v.x - h.x), to_tf32(v.y - h.y), to_tf32(v.z - h.z), to_tf32(v.w - h.w));
        float* blk = dst + ((size_t)tile * (K / LKB) + kb) * 2 * plane;
        const size_t off = (size_t)chunk * tile_rows * 4 + (size_t)(r >> 3) * 32 + (size_t)(r & 7) * 4;
        *reinterpret_cast<float4*>(blk + off) = h;
        *reinterpret_cast<float4*>(blk + plane + off) = l;
    }
}

__global__ void __launch_bounds__(128, 1) tc_layer_kernel(const float* __restrict__ xp, const float* __restrict__ wp, float* __restrict__ Y,
                                                          int K, int N, int* err_flag) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t full[LNST], empty[LNST], done;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int rb = blockIdx.x, nt = blockIdx.y, n_kb = K / LKB;

    if (tid == 0) {
        for (int s = 0; s < LNST; ++s) mbar_init(&full[s], 1), mbar_init(&empty[s], 1);
        mbar_init(&done, 1);
        mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(&tmem_slot, 512);  // [0,256) main accumulator, [256,512) cross terms
    tmem_fence_before();
    __syncthreads();
    tmem_fence_after();
    const uint32_t tmem = tmem_slot;

    // one lane per role; its 31 siblings park at the __syncwarp below instead of spinning on `done` beside it
    if (warp == 1 && lane == 0) {
        // ---- producer: one contiguous X block (hi|lo, 16 KB) + one W block (hi|lo, 32 KB) per stage
        const unsigned char* xsrc = reinterpret_cast<const unsigned char*>(xp) + (size_t)rb * n_kb * 2 * L_A_PLANE;
        const unsigned char* wsrc = reinterpret_cast<const unsigned char*>(wp) + (size_t)nt * n_kb * 2 * L_W_PLANE;
        for (int kb = 0; kb < n_kb; ++kb) {
            const int s = kb % LNST;
            if (kb >= LNST) mbar_wait(&empty[s], (uint32_t)((kb / LNST - 1) & 1), err_flag);
            unsigned char* st = smem_raw + (size_t)s * L_STAGE;
            mbar_expect_tx(&full[s], L_STAGE);
            tma_bulk_g2s(st, xsrc + (size_t)kb * 2 * L_A_PLANE, 2 * L_A_PLANE, &full[s]);
            tma_bulk_g2s(st + 2 * L_A_PLANE, wsrc + (size_t)kb * 2 * L_W_PLANE, 2 * L_W_PLANE, &full[s]);
        }
    } else if (warp == 0 && lane == 0) {
        // ---- MMA issuer
        uint32_t main_acc = 0, cross_acc = 0;
        for (int kb = 0; kb < n_kb; ++kb) {
            const int s = kb % LNST;
            mbar_wait(&full[s], (uint32_t)((kb / LNST) & 1), err_flag);
            tmem_fence_after();
            const uint32_t a_hi = smem_u32(smem_raw + (size_t)s * L_STAGE), a_lo = a_hi + L_A_PLANE;
            const uint32_t w_hi = a_hi + 2 * L_A_PLANE, w_lo = w_hi + L_W_PLANE;
#pragma unroll
            for (int j = 0; j < LKB / 8; ++j) {
                const uint64_t ah = umma_desc(a_hi + 2 * j * L_LBO_A, L_LBO_A, P_SBO), al = umma_desc(a_lo + 2 * j * L_LBO_A, L_LBO_A, P_SBO);
                const uint64_t wh = umma_desc(w_hi + 2 * j * L_LBO_W, L_LBO_W, P_SBO), wl = umma_desc(w_lo + 2 * j * L_LBO_W, L_LBO_W, P_SBO);
                umma_tf32_desc(tmem + LN, al, wh, L_IDESC, cross_acc), cross_acc = 1;
                umma_tf32_desc(tmem + LN, ah, wl, L_IDESC, 1u);
                umma_tf32_desc(tmem, ah, wh, L_IDESC, main_acc), main_acc = 1;
            }
            umma_commit(&empty[s]);  // the stage is free once these MMAs have read it
        }
        umma_commit(&done);
    }
    __syncwarp();
    // ---- epilogue: thread = row of the tile; Y = main + cross
    mbar_wait_backoff(&done, 0, err_flag);
    tmem_fence_after();
    const uint32_t lane_base = tmem + ((uint32_t)(warp * 32) << 16);
    float* yrow = Y + ((size_t)rb * LM + tid) * N + (size_t)nt * LN;
    for (int c0 = 0; c0 < LN; c0 += 8) {
        float m[8], c[8];
        tmem_ld8(lane_base + (uint32_t)c0, m);
        tmem_ld8(lane_base + (uint32_t)(LN + c0), c);
        *reinterpret_cast<float4*>(yrow + c0) = make_float4(m[0] + c[0], m[1] + c[1], m[2] + c[2], m[3] + c[3]);
        *reinterpret_cast<float4*>(yrow + c0 + 4) = make_float4(m[4] + c[4], m[5] + c[5], m[6] + c[6], m[7] + c[7]);
    }
    tmem_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

}  // namespace mlb

extern "C" int mlb_probe_tf32x3(const float* A_dev, const float* W_dev, int K, int mode, float* out_main_dev, float* out_cross_dev,
                                void* stream) {
    using namespace mlb;
    if (!A_dev || !W_dev || !out_main_dev || K < PKB || (K % PKB) != 0 || mode < 0 || mode > 2)
        return mlb_fail("mlb_probe_tf32x3: A [128,K], W [128,K] (K a multiple of 32), out [128,128], mode 0..2");
    const size_t smem = (size_t)(2 * PM + 2 * PN) * PKB * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute(tc_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) {
        tc_probe_kernel<<<1, 128, smem, (cudaStream_t)stream>>>(A_dev, W_dev, K, mode, out_main_dev, out_cross_dev, nullptr);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return mlb_fail(std::string("mlb_probe_tf32x3: ") + cudaGetErrorString(e));
    mlb_count_launch();
    return 0;
}

// stages (bit mask): 1 = split X [B,K] into planes (x_planes, 2*B*K floats), 2 = split W [N,K] (w_planes, 2*N*K floats),
// 4 = the layer GEMM Y[B,N] from the planes.  B % 128 == 0, N % 256 == 0, K % 16 == 0.
extern "C" int mlb_probe_tc_layer(const float* X_dev, const float* W_dev, float* Y_dev, int B, int N, int K, float* x_planes_dev,
                                  float* w_planes_dev, int stages, void* stream) {
    using namespace mlb;
    if (!x_planes_dev || !w_planes_dev || B < LM || (B % LM) || N < LN || (N % LN) || K < LKB || (K % LKB))
        return mlb_fail("mlb_probe_tc_layer: B % 128 == 0, N % 256 == 0, K % 16 == 0 and both plane buffers are required");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaSuccess;
    if ((stages & 1) && X_dev) tc_pack_planes_kernel<<<296, 256, 0, st>>>(X_dev, x_planes_dev, B, K, LM), mlb_count_launch();
    if ((stages & 2) && W_dev) tc_pack_planes_kernel<<<296, 256, 0, st>>>(W_dev, w_planes_dev, N, K, LN), mlb_count_launch();
    if ((stages & 4) && Y_dev) {
        const size_t smem = (size_t)LNST * L_STAGE;
        e = cudaFuncSetAttribute(tc_layer_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) {
            tc_layer_kernel<<<dim3(B / LM, N / LN), 128, smem, st>>>(x_planes_dev, w_planes_dev, Y_dev, K, N, nullptr);
            mlb_count_launch();
        }
    }
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) return mlb_fail(std::string("mlb_probe_tc_layer: ") + cudaGetErrorString(e));
    return 0;
}
