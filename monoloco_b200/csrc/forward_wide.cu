// monoloco_b200 -- latency kernel for one image's worth of detections (<= 32 rows): the WHOLE grid works on one row tile.
//
// What the reference does per image (net.py:92-124): preprocess_monoloco -> model(inputs) -> extract_outputs on the 1-30
// people of one frame.  At that size the forward pass is a stream of 33.8 MB of weights against a [<=32 x 1024] activation
// tile; a single CTA (forward.cu) or an 8-CTA cluster (forward_small.cu) can only pull the weights through 1 / 8 SMs'
// worth of L2 bandwidth.  Here every layer is split by OUTPUT COLUMNS over L/8 CTAs (128 at L = 1024):
//
//   CTA c owns columns [8c, 8c+8) of every layer.  Its weights are one contiguous slab  Wt[k][8]  per layer (32 KB at
//   K = 1024, re-packed at mlb_create), streamed by TMA through a 2-stage ring that runs ahead of the layer loop.
//   Per layer:  256 threads = (k-subset, row pair) compute partial sums of the [R x 8] block  ->  shared-memory reduction ->
//   folded-BN / ReLU / dropout / residual epilogue (one output per thread, residual kept in that thread's register) ->
//   the block goes to a global k-major exchange buffer xg[parity][L][R] -> grid barrier -> every CTA pulls the complete
//   next-layer input tile (L x R floats, L2-resident) back into shared memory with one TMA bulk copy.
//   Narrow heads (the same slab code over zero-padded [K][8] head slabs), decode and the stores run on CTA 0; the
//   other CTAs exit after the last exchange.
//
// Cooperative launch (co-residency for the hand-rolled grid barrier); the barrier counter is monotonic across launches
// (the host passes the base value), so no memset precedes the kernel.
#include <cuda_runtime.h>
#include <stdint.h>

#include "fwd_family.cuh"

namespace mlb {

constexpr int WC = 8;        // output columns per CTA
constexpr int WNT = 256;     // threads per CTA
constexpr int WNST = 2;      // weight-slab ring stages
constexpr int WPART = 8 * 16 * 32;  // floats of the partial-sum buffer

struct WideExtra {
    const float* wslab;                // per GEMM op: [L/8 CTAs][Kpad][8]; per head op: [ceil(N/8)][K][8]
    long long wslab_off[MLB_MAX_OPS];  // float offset of each op's slab block
    float* xg;                         // [2][L][32] exchange buffer (k-major tiles, double-buffered by layer parity)
    unsigned* bar;                     // monotonic grid-barrier counter
    unsigned bar_base;                 // counter value when this launch starts
};

__device__ __forceinline__ unsigned wide_ld_acquire(const unsigned* ptr) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ptr) : "memory");
    return v;
}

// profiling aid (mlb_debug_fwd_marks): thread 0 of CTA 0 (and of CTA 64, at +128) stamps globaltimer along the layer loop
__device__ unsigned long long* g_wide_marks = nullptr;
__device__ __forceinline__ void wmark(unsigned long long* marks, int slot) {
    if (marks != nullptr) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        marks[slot] = t;
    }
}

template <int R>  // row slots of the tile: 16 or 32
__global__ void __launch_bounds__(WNT, 1) loco_forward_wide_kernel(const __grid_constant__ FwdParams p,
                                                                   const __grid_constant__ WideExtra ex) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int S = 2 * WNT / R;  // k-subsets: thread (s, row pair q) accumulates k = s, s + S, s + 2S, ... for rows 2q, 2q+1
    const int tid = threadIdx.x;
    const int cta = blockIdx.x, L = p.L;

    float* act = reinterpret_cast<float*>(smem_raw);   // [L][R]  k-major input tile of the current layer
    float* ring = act + (size_t)L * R;                  // [WNST][L][WC] weight slabs
    float* part = ring + (size_t)WNST * L * WC;         // [S][WC][R] partial sums
    float* outs = part + WPART;                         // [R][OUT_LD]
    float* cen = outs + R * OUT_LD;                     // [R][4]
    float* sstab = cen + R * 4;                         // [n_ops][32]: folded-BN scale[16] | shift-or-bias[16] of this CTA's columns
    uint64_t* wfull = reinterpret_cast<uint64_t*>(sstab + MLB_MAX_OPS * 32);  // [WNST]
    uint64_t* gfull = wfull + WNST;                     // exchange-tile arrival

    unsigned long long* marks = (tid == 0 && (cta == 0 || cta == 64) && g_wide_marks != nullptr) ? g_wide_marks + (cta ? 128 : 0) : nullptr;
    wmark(marks, 0);
    if (tid == 0) {
        for (int s = 0; s < WNST; ++s) mbar_init(&wfull[s], 1);
        mbar_init(gfull, 1);
        mbar_fence_init();
    }
    for (int i = tid; i < R * OUT_LD; i += WNT) outs[i] = 0.f;
    // every layer's epilogue constants for this CTA's columns, fetched once up front (an L2 round trip per layer otherwise)
    for (int i = tid; i < p.n_ops * 32; i += WNT) {
        const mlb_op& op = p.ops[i >> 5];
        const int j = i & 15, shift = (i >> 4) & 1;
        float v = 0.f;
        if (op.type == MLB_OP_GEMM) {
            if (j < WC) v = __ldg(p.blob + (shift ? op.shift_off : op.scale_off) + cta * WC + j);
        } else if (shift && j < op.N) {
            v = __ldg(p.blob + op.shift_off + j);
        }
        sstab[i] = v;
    }
    __syncthreads();

    // ---- weight stream.  Item = one [Kpad][8] slab: every GEMM op contributes the CTA's column slab; on CTA 0 (which
    // also runs the narrow heads) a head op contributes ceil(N / 8) zero-padded slabs.  Item i lives in ring stage
    // i % WNST and is issued by thread 0 two items ahead of its use.
    auto n_items_of = [&](const mlb_op& op) { return op.type == MLB_OP_GEMM ? 1 : (cta == 0 ? (op.N + WC - 1) / WC : 0); };
    int n_items = 0;
    for (int oi = 0; oi < p.n_ops; ++oi) n_items += n_items_of(p.ops[oi]);
    int issue_op = 0, issue_sub = 0, issued = 0;  // stream cursor (thread 0)
    auto issue_next = [&]() {
        while (issue_op < p.n_ops && issue_sub >= n_items_of(p.ops[issue_op])) issue_op++, issue_sub = 0;
        if (issue_op >= p.n_ops) return;
        const mlb_op& op = p.ops[issue_op];
        const bool gemm = op.type == MLB_OP_GEMM;
        const int kp = gemm ? op.Kpad : op.K;
        const uint32_t bytes = (uint32_t)(kp * WC * sizeof(float));
        const float* src = ex.wslab + ex.wslab_off[issue_op] + (size_t)(gemm ? cta : issue_sub) * kp * WC;
        const int st = issued % WNST;
        mbar_expect_tx(&wfull[st], bytes);
        tma_bulk_g2s(ring + (size_t)st * L * WC, src, bytes, &wfull[st]);
        issued++, issue_sub++;
    };
    if (tid == 0)
        for (int i = 0; i < WNST; ++i) issue_next();

    const int row0 = p.row_base;
    const int rows_here = min(R, p.n_rows - row0);  // a single tile
    stage_input_tile(p, row0, rows_here, R, R, act, cen, tid, WNT, [] { __syncthreads(); });
    __syncthreads();
    if (cta == 0 && p.out_x != nullptr && p.input_kind != MLB_IN_X) {
        for (int idx = tid; idx < rows_here * p.in_size; idx += WNT) {
            const int r = idx / p.in_size, k = idx % p.in_size;
            p.out_x[(size_t)(row0 + r) * p.in_size + k] = act[k * R + r];
        }
    }
    wmark(marks, 1);

    // GEMM mapping: k-subset gs, row pair gq (a warp covers 32 / (R/2) consecutive k: contiguous, conflict-free LDS.64)
    const int gs = tid / (R / 2), gq = tid % (R / 2);
    // reduce / epilogue mapping (threads < WC * R): column ec of the slab's 8, row er
    const int ec = tid / R, er = tid % R;
    const bool epi = tid < WC * R;
    const int gcol = cta * WC + ec;
    int item = 0;  // items consumed so far
    // partial sums of the [R x 8] block of the slab in ring stage item % WNST over K = kp, reduced into `v` of thread (ec, er)
    auto slab_block = [&](int kp) -> float {
        const int st = item % WNST;
        mbar_wait(&wfull[st], (item / WNST) & 1, p.err_flag);
        const float* w = ring + (size_t)st * L * WC;
        // two rows per thread: one LDS.64 of activations + two broadcast LDS.128 of weights feed 16 FMAs
        float acc0[WC] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, acc1[WC] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
        for (int k = gs; k < kp; k += S) {
            const float2 a = *reinterpret_cast<const float2*>(act + k * R + 2 * gq);
            const float4 w0 = *reinterpret_cast<const float4*>(w + k * WC);
            const float4 w1 = *reinterpret_cast<const float4*>(w + k * WC + 4);
            const float wv[WC] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
            for (int c = 0; c < WC; ++c) acc0[c] = fmaf(a.x, wv[c], acc0[c]), acc1[c] = fmaf(a.y, wv[c], acc1[c]);
        }
#pragma unroll
        for (int c = 0; c < WC; ++c) *reinterpret_cast<float2*>(part + (gs * WC + c) * R + 2 * gq) = make_float2(acc0[c], acc1[c]);
        __syncthreads();  // partials complete; nobody reads this ring stage any more
        item++;
        if (tid == 0) issue_next();
        float v = 0.f;
        if (epi) {
#pragma unroll
            for (int s = 0; s < S; ++s) v += part[(s * WC + ec) * R + er];
        }
        return v;
    };

    float res = 0.f;
    int site = 0, g = 0, par = 0;
    unsigned bar_target = ex.bar_base;
    int n_gemm = 0;
    for (int oi = 0; oi < p.n_ops; ++oi) n_gemm += p.ops[oi].type == MLB_OP_GEMM;

    for (int oi = 0; oi < p.n_ops; ++oi) {
        const mlb_op& op = p.ops[oi];
        if (op.type == MLB_OP_GEMM) {
            wmark(marks, 2 + 4 * g);
            float v = slab_block(op.Kpad);
            wmark(marks, 3 + 4 * g);
            const bool last_gemm = g + 1 == n_gemm;
            if (epi) {
                v = fmaf(v, sstab[oi * 32 + ec], sstab[oi * 32 + 16 + ec]);
                if (op.flags & MLB_F_RELU) v = fmaxf(v, 0.f);
                if ((op.flags & MLB_F_DROPOUT) && (p.flags & MLB_FWD_DROPOUT)) {
                    bool keep;
                    if (p.drop_mask != nullptr)
                        keep = er < rows_here ? p.drop_mask[((size_t)site * p.n_rows + row0 + er) * L + gcol] != 0 : true;
                    else
                        keep = keep_draw(p.drop_seed, site, row0 + er, gcol, p.p_drop);
                    v = keep ? v * (1.0f / (1.0f - p.p_drop)) : 0.f;
                }
                if (op.flags & MLB_F_ADD_RES) v += res;
                if (op.flags & MLB_F_SAVE_RES) res = v;
                ex.xg[((size_t)par * L + gcol) * R + er] = er < rows_here ? v : 0.f;
            }
            if (op.flags & MLB_F_DROPOUT) site++;
            // ---- grid barrier, then pull the complete tile back (TMA bulk copy, L2 -> shared)
            __syncthreads();
            bar_target += gridDim.x;
            if (tid == 0)  // release-add: orders the CTA's exchange stores (observed through the barrier above) before the arrival
                asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ex.bar) : "memory");
            if (last_gemm && cta != 0) return;  // heads / decode / stores run on CTA 0 only
            if (tid == 0) {
                unsigned spins = 0;
                while ((int)(wide_ld_acquire(ex.bar) - bar_target) < 0) {
                    if (++spins > (1u << 24)) {
                        if (p.err_flag != nullptr) *reinterpret_cast<volatile int*>(p.err_flag) = 3;
                        __threadfence_system();
                        __trap();
                    }
                }
                wmark(marks, 4 + 4 * g);
                asm volatile("fence.proxy.async;" ::: "memory");  // peers' generic-proxy stores -> this async-proxy read
                const uint32_t bytes = (uint32_t)((size_t)L * R * sizeof(float));
                mbar_expect_tx(gfull, bytes);
                for (uint32_t off = 0; off < bytes; off += 32768u)
                    tma_bulk_g2s(reinterpret_cast<unsigned char*>(act) + off,
                                 reinterpret_cast<const unsigned char*>(ex.xg + (size_t)par * L * R) + off,
                                 min(32768u, bytes - off), gfull);
            }
            mbar_wait(gfull, g & 1, p.err_flag);
            wmark(marks, 5 + 4 * g);
            par ^= 1;
            g++;
        } else if (cta == 0) {
            // ---- narrow head on CTA 0: the same slab code over ceil(N / 8) zero-padded [K][8] slabs
            for (int sub = 0; sub * WC < op.N; ++sub) {
                const float v = slab_block(op.K);
                const int o = sub * WC + ec;
                if (epi && o < op.N) outs[er * OUT_LD + op.out_col + o] = v + sstab[oi * 32 + 16 + o];
                __syncthreads();  // `part` is rewritten by the next slab
            }
            wmark(marks, 2 + 4 * g);
        }
    }
    // ---- decode + store (CTA 0, one thread per row)
    __syncthreads();
    wmark(marks, 2 + 4 * n_gemm);
    if (tid < rows_here) store_row(p, (size_t)row0 + tid, outs + tid * OUT_LD, cen + tid * 4);
    if (p.n_gather) {
        __syncthreads();
        if (tid == 0) gather_finish(p);  // CTA 0 is the only storing CTA of this kernel
    }
    wmark(marks, 3 + 4 * n_gemm);
}

// W^T [Kpad][L] -> per-CTA slabs [L/8][Kpad][8]
__global__ void wide_pack_kernel(const float* __restrict__ wt, float* __restrict__ slab, int kpad, int L) {
    const int n = kpad * L;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int k = i / L, col = i % L;
        slab[((size_t)(col / WC) * kpad + k) * WC + col % WC] = wt[i];
    }
}

template <int R>
static size_t wide_smem(int L) {
    return ((size_t)L * R + (size_t)WNST * L * WC + (size_t)WPART + (size_t)R * OUT_LD + (size_t)R * 4 + (size_t)MLB_MAX_OPS * 32) * sizeof(float) +
           (WNST + 1) * sizeof(uint64_t);
}

}  // namespace mlb

using namespace mlb;

cudaError_t WideFamily::set_marks(unsigned long long* ptr) { return cudaMemcpyToSymbol(mlb::g_wide_marks, &ptr, sizeof(ptr)); }

// head weights W[N][K] -> ceil(N/8) zero-padded k-major slabs [K][8]
__global__ void wide_pack_head_kernel(const float* __restrict__ w, float* __restrict__ slab, int N, int K) {
    const int nsub = (N + mlb::WC - 1) / mlb::WC;
    const int n = nsub * K * mlb::WC;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int sub = i / (K * mlb::WC), k = (i / mlb::WC) % K, c = i % mlb::WC;
        const int o = sub * mlb::WC + c;
        slab[i] = o < N ? w[(size_t)o * K + k] : 0.f;
    }
}

cudaError_t WideFamily::repack(const float* blob, const mlb_op* ops, int n_ops, int L, cudaStream_t st) const {
    if (!available) return cudaSuccess;
    for (int i = 0; i < n_ops; ++i) {
        if (ops[i].type == MLB_OP_GEMM)
            wide_pack_kernel<<<128, 256, 0, st>>>(blob + ops[i].w_off, slab + slab_off[i], ops[i].Kpad, L);
        else
            wide_pack_head_kernel<<<32, 256, 0, st>>>(blob + ops[i].w_off, slab + slab_off[i], ops[i].N, ops[i].K);
    }
    return cudaGetLastError();
}

// can the whole grid (L/8 CTAs) be co-resident?  (cooperative launch requirement)
static bool wide_supported(int L, int n_sms) {
    if (L % 128 != 0 || L / WC > n_sms) return false;
    int occ = 0;
    if (cudaFuncSetAttribute(loco_forward_wide_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wide_smem<32>(L)) != cudaSuccess)
        return false;
    if (cudaFuncSetAttribute(loco_forward_wide_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wide_smem<16>(L)) != cudaSuccess)
        return false;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, loco_forward_wide_kernel<32>, WNT, wide_smem<32>(L)) != cudaSuccess || occ < 1)
        return false;
    return true;
}

cudaError_t WideFamily::setup(const float* blob, const mlb_op* ops, int n_ops, int L, int n_sms) {
    if (L > 1024 || !wide_supported(L, n_sms)) return cudaSuccess;
    // slab copy: GEMM [L/8][Kpad][8]; head [ceil(N/8)][K][8]
    size_t off = 0;
    for (int i = 0; i < n_ops; ++i) {
        slab_off[i] = (long long)off;
        if (ops[i].type == MLB_OP_GEMM)
            off += (size_t)ops[i].Kpad * L;
        else
            off += (size_t)((ops[i].N + WC - 1) / WC) * ops[i].K * WC;
    }
    cudaError_t e;
    if ((e = cudaMalloc(&slab, off * sizeof(float))) != cudaSuccess) return e;
    available = true;
    if ((e = repack(blob, ops, n_ops, L, 0)) != cudaSuccess) return e;
    if ((e = mlb_zalloc(&xg, (size_t)2 * L * 32 * sizeof(float))) != cudaSuccess) return e;
    return mlb_zalloc(&bar, sizeof(unsigned));
}

void WideFamily::release() {
    cudaFree(slab), cudaFree(xg), cudaFree(bar);
    slab = nullptr, xg = nullptr, bar = nullptr;
    available = false;
}

template <int R>
static cudaError_t launch_wide(void** args, int L, cudaStream_t st) {
    // (the opt-in shared-memory size is a per-function, per-process attribute: set it for THIS model's width on every launch)
    const cudaError_t e = cudaFuncSetAttribute(loco_forward_wide_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wide_smem<R>(L));
    if (e != cudaSuccess) return e;
    return cudaLaunchCooperativeKernel((void*)loco_forward_wide_kernel<R>, dim3(L / WC), dim3(WNT), args, wide_smem<R>(L), st);
}

cudaError_t WideFamily::launch(FwdParams p, const FwdPlan& pl, cudaStream_t st, int* issued) {
    WideExtra ex;
    ex.wslab = slab;
    for (int i = 0; i < MLB_MAX_OPS; ++i) ex.wslab_off[i] = i < p.n_ops ? slab_off[i] : 0;
    ex.xg = xg, ex.bar = bar;
    int n_gemm = 0;  // one grid barrier per GEMM: the counter advances by n_gemm * grid per launch
    for (int i = 0; i < p.n_ops; ++i) n_gemm += p.ops[i].type == MLB_OP_GEMM;
    const unsigned epoch = p.gather_epoch;
    void* args[] = {(void*)&p, (void*)&ex};
    p.n_tiles = 1;
    for (int t = 0; t < pl.launches; ++t) {
        p.row_base = 32 * t;
        p.gather_epoch = t + 1 == pl.launches ? epoch : 0;  // the last launch completes the batch for the all-gather
        ex.bar_base = bar_count;
        const cudaError_t e = p.n_rows - p.row_base <= 16 ? launch_wide<16>(args, p.L, st) : launch_wide<32>(args, p.L, st);
        if (e != cudaSuccess) return e;  // nothing ran: the device counter did not move
        bar_count += (unsigned)n_gemm * (unsigned)(p.L / WC);
        ++*issued;
    }
    return cudaSuccess;
}
