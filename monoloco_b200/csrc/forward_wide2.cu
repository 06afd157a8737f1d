// monoloco_b200 -- latency kernel, second generation, for one image's worth of detections (<= 16 rows per launch).
//
// forward_wide.cu splits every layer by output columns over 128 CTAs: each CTA then needs the COMPLETE [1024 x R] activation
// tile of the next layer, so a layer costs a grid barrier (atomic counter, ~1.5 us) plus a 64 KB exchange copy per CTA
// (~0.9 us) on top of ~1.7 us of math: 4.1 us x 10 layers.  Here the layer is split in TWO dimensions:
//
//   32 thread-block clusters x 4 CTAs.  Cluster j owns output columns [32j, 32j+32); CTA i of a cluster owns the K slice
//   [256i, 256i+256).  Its weights are one contiguous [256][32] slab per layer (32 KB, re-packed at mlb_create), streamed by
//   TMA through a 5-deep ring that is filled at t = 0 (half the network's weights in flight before the first layer starts).
//   Per layer:
//     1. poll this CTA's K slice of the previous layer's outputs [256 k][R] from a global buffer of (value, epoch) pairs
//        -- data and flag travel in the same 8 bytes (the "LL" protocol of collective libraries): ONE L2 hop, no barrier,
//        no separate copy; 32 KB per CTA instead of 64 KB;
//     2. 256 threads = (k-subset, 8-column group, row pair): 16 accumulators each, 512 FMAs;
//     3. every partial goes straight into the shared memory of the cluster CTA that finalises that column
//        (st.shared::cluster), one barrier.cluster;
//     4. 128 threads of each CTA sum the 32 partials of one output in a fixed order, apply folded BN / ReLU / dropout /
//        residual (the residual never leaves the thread's register) and publish (value, epoch) for the next layer.
//   Heads: every thread keeps the partial dot products of ITS output column with the head rows; one more LL hop collects the
//   128 CTAs' partials on CTA 0, which decodes and stores (fwd_common.cuh::store_row, incl. the fused all-gather peers).
//
// Buffers rotate over three layers: a CTA can run at most two layers ahead of the slowest one (it needs outputs that need
// everyone's previous outputs), so the third-oldest buffer is free.  Epochs grow monotonically across launches (the host passes
// the base), nothing is ever cleared.  All 128 CTAs must be co-resident: cooperative launch.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "fwd_family.cuh"

namespace mlb {

constexpr int W2_CL = 4;          // CTAs per cluster (K slices)
constexpr int W2_NC = 32;         // output columns per cluster
constexpr int W2_FC = 8;          // columns finalised per CTA
constexpr int W2_NT = 256;        // threads per CTA
constexpr int W2_NST = 5;         // weight-slab ring stages
constexpr int W2_HQ = 16;         // head rows (output columns of the network), max
constexpr int W2_R = 16;          // row slots

struct Wide2Extra {
    const float* wslab;                // per GEMM op: [clusters][W2_CL][kslice][W2_NC]
    long long wslab_off[MLB_MAX_OPS];
    unsigned long long* xg;            // [3][L][W2_R] (value, epoch) pairs
    unsigned long long* hg;            // [n_clusters][W2_HQ][W2_R] head partial pairs
    unsigned epoch_base;               // epochs of this launch: epoch_base + 1 + layer
};

__device__ __forceinline__ void w2_cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void w2_cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t w2_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t w2_mapa(uint32_t smem_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void w2_st_pair(unsigned long long* ptr, float v, unsigned epoch) {
    asm volatile("st.volatile.global.v2.u32 [%0], {%1, %2};" ::"l"(ptr), "r"(__float_as_uint(v)), "r"(epoch) : "memory");
}
__device__ __forceinline__ uint4 w2_ld_pairs(const unsigned long long* ptr) {  // two (value, epoch) pairs
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(ptr) : "memory");
    return v;
}

__device__ unsigned long long* g_wide2_marks = nullptr;
__device__ __forceinline__ void w2mark(unsigned long long* marks, int slot) {
    if (marks != nullptr) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        marks[slot] = t;
    }
}

__global__ void __cluster_dims__(W2_CL, 1, 1) __launch_bounds__(W2_NT, 1)
    loco_forward_wide2_kernel(const __grid_constant__ FwdParams p, const __grid_constant__ Wide2Extra ex) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int R = W2_R;
    const int tid = threadIdx.x;
    const int ci = (int)w2_ctarank();            // K slice / which 8 of the cluster's 32 columns this CTA finalises
    const int cj = (int)blockIdx.x / W2_CL;      // cluster = column block
    const int L = p.L, KS = L / W2_CL;           // K slice depth (256 at L = 1024)
    const int n_cta = (int)gridDim.x;

    float* ring = reinterpret_cast<float*>(smem_raw);          // [W2_NST][KS][W2_NC]
    float* act = ring + (size_t)W2_NST * KS * W2_NC;            // [KS][R]   k-major slice of the layer input
    float* inbox = act + (size_t)KS * R;                        // [2][32 partials][W2_FC * R]
    float* outs = inbox + 2 * 32 * W2_FC * R;                   // [R][OUT_LD]  (CTA 0)
    float* cen = outs + R * OUT_LD;                             // [R][4]
    float* sstab = cen + R * 4 + W2_HQ;                         // (+ head biases) [n_ops][2][W2_FC] scale | shift of the finalised columns
    float* hsm = sstab + MLB_MAX_OPS * 2 * W2_FC;               // [W2_HQ][W2_FC][R] head products
    uint64_t* wfull = reinterpret_cast<uint64_t*>(hsm + W2_HQ * W2_FC * R);  // [W2_NST]

    unsigned long long* marks = (tid == 0 && blockIdx.x == 0) ? g_wide2_marks : nullptr;
    w2mark(marks, 0);
    if (tid == 0) {
        for (int s = 0; s < W2_NST; ++s) mbar_init(&wfull[s], 1);
        mbar_fence_init();
    }
    // the output this thread finalises (threads < W2_FC * R): column fc of the CTA's 8, row fr
    const int fc = tid / R, fr = tid % R;
    const bool fin = tid < W2_FC * R;
    const int gcol = cj * W2_NC + ci * W2_FC + fc;
    for (int i = tid; i < p.n_ops * 2 * W2_FC; i += W2_NT) {
        const mlb_op& op = p.ops[i / (2 * W2_FC)];
        const int shift = (i / W2_FC) & 1, c = i % W2_FC;
        sstab[i] = op.type == MLB_OP_GEMM ? __ldg(p.blob + (shift ? op.shift_off : op.scale_off) + cj * W2_NC + ci * W2_FC + c) : 0.f;
    }
    __syncthreads();
    w2_cluster_arrive();
    w2_cluster_wait();   // every CTA of the cluster has initialised its barriers before a peer can touch its shared memory

    // ---- weight stream: one [kp][32] slab per GEMM op (kp = this CTA's share of the op's K, 0 for a slice beyond Kpad)
    auto kslice_of = [&](const mlb_op& op) { return max(0, min(KS, op.Kpad - ci * KS)); };
    int issue_op = 0, issued = 0;
    auto issue_next = [&]() {
        while (issue_op < p.n_ops && (p.ops[issue_op].type != MLB_OP_GEMM || kslice_of(p.ops[issue_op]) == 0)) issue_op++;
        if (issue_op >= p.n_ops) return;
        const mlb_op& op = p.ops[issue_op];
        const int kp = kslice_of(op);
        const uint32_t bytes = (uint32_t)(kp * W2_NC * sizeof(float));
        const float* src = ex.wslab + ex.wslab_off[issue_op] + ((size_t)cj * W2_CL + ci) * (size_t)min(KS, op.Kpad) * W2_NC;
        const int st = issued % W2_NST;
        mbar_expect_tx(&wfull[st], bytes);
        tma_bulk_g2s(ring + (size_t)st * KS * W2_NC, src, bytes, &wfull[st]);
        issued++, issue_op++;
    };
    if (tid == 0)
        for (int i = 0; i < W2_NST; ++i) issue_next();

    const int row0 = p.row_base;
    const int rows_here = min(R, p.n_rows - row0);
    // network input: every CTA evaluates the tile's pre-process; the first layer's K (<= 72) lies in slice 0
    stage_input_tile(p, row0, rows_here, R, R, act, cen, tid, W2_NT, [] { __syncthreads(); });
    __syncthreads();
    if (blockIdx.x == 0 && p.out_x != nullptr && p.input_kind != MLB_IN_X) {
        for (int idx = tid; idx < rows_here * p.in_size; idx += W2_NT) {
            const int r = idx / p.in_size, k = idx % p.in_size;
            p.out_x[(size_t)(row0 + r) * p.in_size + k] = act[k * R + r];
        }
    }
    w2mark(marks, 1);

    // GEMM mapping: k-subset gs (8), column group gc (4 x 8 columns = the 8 columns CTA gc of the cluster finalises), row pair gq (8)
    const int gq = tid & 7, gc = (tid >> 3) & 3, gs = tid >> 5;
    const uint32_t inbox_s = smem_u32(inbox);
    const uint32_t inbox_remote = w2_mapa(inbox_s, (uint32_t)gc);   // my partials of column group gc go to cluster CTA gc

    // head rows: my column's weight of every head row, fetched now (a cold L2 costs a DRAM round trip per head layer otherwise)
    float hacc[W2_HQ], hwt[W2_HQ];
#pragma unroll
    for (int q = 0; q < W2_HQ; ++q) hacc[q] = 0.f, hwt[q] = 0.f;
    if (fin) {
        for (int oj = 0; oj < p.n_ops; ++oj) {
            const mlb_op& hop = p.ops[oj];
            if (hop.type != MLB_OP_HEAD) continue;
#pragma unroll
            for (int q = 0; q < W2_HQ; ++q)
                if (q >= hop.out_col && q < hop.out_col + hop.N) hwt[q] = __ldg(p.blob + hop.w_off + (size_t)(q - hop.out_col) * hop.K + gcol);
        }
    }
    if (blockIdx.x == 0) {   // biases of the head rows (CTA 0 finishes the outputs); hsm is free until the end
        for (int t = tid; t < W2_HQ; t += W2_NT) {
            float bias = 0.f;
            for (int oj = 0; oj < p.n_ops; ++oj)
                if (p.ops[oj].type == MLB_OP_HEAD && t >= p.ops[oj].out_col && t < p.ops[oj].out_col + p.ops[oj].N)
                    bias = __ldg(p.blob + p.ops[oj].shift_off + (t - p.ops[oj].out_col));
            cen[R * 4 + t] = bias;
        }
    }
    int n_gemm = 0;
    for (int oi = 0; oi < p.n_ops; ++oi) n_gemm += p.ops[oi].type == MLB_OP_GEMM;

    float res = 0.f;
    int site = 0, g = 0, item = 0;
    for (int oi = 0; oi < p.n_ops; ++oi) {
        const mlb_op& op = p.ops[oi];
        if (op.type != MLB_OP_GEMM) continue;
        const unsigned epoch = ex.epoch_base + 1u + (unsigned)g;   // epoch of THIS layer's outputs
        const int kp = kslice_of(op);
        const int par = g & 1;
        w2mark(marks, 2 + 4 * g);
        // ---- 1. input slice: (value, epoch) pairs of the previous layer, one L2 hop (layer 0: the staged network input)
        if (g > 0) {
            const unsigned ep = epoch - 1u;
            const unsigned long long* src = ex.xg + ((size_t)(ep % 3u) * L + (size_t)ci * KS) * R;
            const int n_units = KS * R / 2;   // 16-byte units of two pairs: n_units / 256 per thread, all polled concurrently
            constexpr int UPT = 8;            // units per thread per pass (KS * R / 2 / 256 = 8 at L = 1024)
            for (int u0 = tid; u0 < n_units; u0 += W2_NT * UPT) {
                uint4 v[UPT];
                unsigned pending = 0, spins = 0;
#pragma unroll
                for (int m = 0; m < UPT; ++m)
                    if (u0 + m * W2_NT < n_units) pending |= 1u << m;
                while (pending) {
#pragma unroll
                    for (int m = 0; m < UPT; ++m)
                        if (pending & (1u << m)) v[m] = w2_ld_pairs(src + 2 * (u0 + m * W2_NT));
#pragma unroll
                    for (int m = 0; m < UPT; ++m)
                        if ((pending & (1u << m)) && v[m].y == ep && v[m].w == ep) {
                            *reinterpret_cast<float2*>(act + 2 * (u0 + m * W2_NT)) = make_float2(__uint_as_float(v[m].x), __uint_as_float(v[m].z));
                            pending &= ~(1u << m);
                        }
                    if (++spins > (1u << 22)) {
                        if (p.err_flag != nullptr) *reinterpret_cast<volatile int*>(p.err_flag) = 3;
                        __threadfence_system();
                        __trap();
                    }
                }
            }
            __syncthreads();
        }
        w2mark(marks, 3 + 4 * g);
        // ---- 2. partial sums over my k-subset of this CTA's K slice: 8 columns x 2 rows
        float acc0[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, acc1[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (kp > 0) {
            const int st = item % W2_NST;
            mbar_wait(&wfull[st], (item / W2_NST) & 1, p.err_flag);
            const float* w = ring + (size_t)st * KS * W2_NC + gc * 8;
            // 8 k per trip, all 24 shared-memory loads of the trip issued before its 128 FMAs (the loop was latency-bound:
            // 1.4 us for 512 FMAs per thread with two warps per scheduler)
            int k = gs;
            for (; k + 56 < kp; k += 64) {
                float2 a[8];
                float4 w0[8], w1[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    a[u] = *reinterpret_cast<const float2*>(act + (k + 8 * u) * R + 2 * gq);
                    w0[u] = *reinterpret_cast<const float4*>(w + (k + 8 * u) * W2_NC);
                    w1[u] = *reinterpret_cast<const float4*>(w + (k + 8 * u) * W2_NC + 4);
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const float wv[8] = {w0[u].x, w0[u].y, w0[u].z, w0[u].w, w1[u].x, w1[u].y, w1[u].z, w1[u].w};
#pragma unroll
                    for (int c = 0; c < 8; ++c) acc0[c] = fmaf(a[u].x, wv[c], acc0[c]), acc1[c] = fmaf(a[u].y, wv[c], acc1[c]);
                }
            }
            for (; k < kp; k += 8) {
                const float2 a = *reinterpret_cast<const float2*>(act + k * R + 2 * gq);
                const float4 w0 = *reinterpret_cast<const float4*>(w + k * W2_NC);
                const float4 w1 = *reinterpret_cast<const float4*>(w + k * W2_NC + 4);
                const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
                for (int c = 0; c < 8; ++c) acc0[c] = fmaf(a.x, wv[c], acc0[c]), acc1[c] = fmaf(a.y, wv[c], acc1[c]);
            }
            item++;
        }
        w2mark(marks, 64 + 2 * g);
        // ---- 3. every partial straight into the inbox of the cluster CTA that finalises the column
        {
            const uint32_t dst = inbox_remote + (uint32_t)((((size_t)par * 32 + (size_t)ci * 8 + gs) * (W2_FC * R) + 2 * gq) * sizeof(float));
#pragma unroll
            for (int c = 0; c < 8; ++c)
                asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(dst + (uint32_t)(c * R * sizeof(float))), "f"(acc0[c]), "f"(acc1[c])
                             : "memory");
        }
        w2mark(marks, 65 + 2 * g);
        w2_cluster_arrive();
        w2_cluster_wait();
        if (tid == 0 && kp > 0) issue_next();   // every thread of this CTA is past its reads of the ring stage
        w2mark(marks, 4 + 4 * g);
        // ---- 4. finalise my output: 32 partials in a fixed order, folded BN / ReLU / dropout / residual, publish
        if (fin) {
            const float* ib = inbox + (size_t)par * 32 * (W2_FC * R) + fc * R + fr;
            float v = 0.f;
#pragma unroll 8
            for (int s2 = 0; s2 < 32; ++s2) v += ib[(size_t)s2 * (W2_FC * R)];
            v = fmaf(v, sstab[(oi * 2 + 0) * W2_FC + fc], sstab[(oi * 2 + 1) * W2_FC + fc]);
            if (op.flags & MLB_F_RELU) v = fmaxf(v, 0.f);
            if ((op.flags & MLB_F_DROPOUT) && (p.flags & MLB_FWD_DROPOUT)) {
                bool keep;
                if (p.drop_mask != nullptr)
                    keep = fr < rows_here ? p.drop_mask[((size_t)site * p.n_rows + row0 + fr) * L + gcol] != 0 : true;
                else
                    keep = keep_draw(p.drop_seed, site, row0 + fr, gcol, p.p_drop);
                v = keep ? v * (1.0f / (1.0f - p.p_drop)) : 0.f;
            }
            if (op.flags & MLB_F_ADD_RES) v += res;
            if (op.flags & MLB_F_SAVE_RES) res = v;
            if (fr >= rows_here) v = 0.f;
            // narrow heads that read this layer's output: my column's share of every head row
            for (int oj = oi + 1; oj < p.n_ops && p.ops[oj].type == MLB_OP_HEAD; ++oj) {
                const mlb_op& hop = p.ops[oj];
#pragma unroll
                for (int q = 0; q < W2_HQ; ++q)
                    if (q >= hop.out_col && q < hop.out_col + hop.N) hacc[q] = fmaf(v, hwt[q], hacc[q]);
            }
            if (g + 1 < n_gemm) w2_st_pair(ex.xg + ((size_t)(epoch % 3u) * L + gcol) * R + fr, v, epoch);
        }
        if (op.flags & MLB_F_DROPOUT) site++;
        w2mark(marks, 5 + 4 * g);
        g++;
    }

    // ---- heads: sum my 8 columns' shares in shared memory, publish per (head row, detection); CTA 0 collects all CTAs
    const unsigned ep_h = ex.epoch_base + 1u + (unsigned)n_gemm;
    const int nq = p.out_size;
    if (fin) {
#pragma unroll
        for (int q = 0; q < W2_HQ; ++q)
            if (q < nq) hsm[((size_t)q * W2_FC + fc) * R + fr] = hacc[q];
    }
    __syncthreads();
    // my 8 columns' shares summed -> the cluster's rank-0 CTA (distributed shared memory; the inbox is idle now) -> one
    // (value, epoch) publication per cluster: CTA 0 then collects 32 publishers instead of 128
    {
        // [W2_CL][W2_HQ * R] on rank 0, in the inbox half the LAST layer did not use (rank 0 may still be summing the other)
        const uint32_t hin_off = (uint32_t)((((n_gemm - 1) & 1) ^ 1) * 32 * W2_FC * R * sizeof(float));
        const uint32_t hin_remote = w2_mapa(inbox_s, 0u) + hin_off;
        for (int t = tid; t < nq * R; t += W2_NT) {
            const int q = t / R, r = t % R;
            float s2 = 0.f;
#pragma unroll
            for (int c = 0; c < W2_FC; ++c) s2 += hsm[((size_t)q * W2_FC + c) * R + r];
            asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(hin_remote + (uint32_t)((ci * (W2_HQ * R) + t) * sizeof(float))), "f"(s2) : "memory");
        }
    }
    w2_cluster_arrive();
    w2_cluster_wait();
    if (ci != 0) return;   // no peer addresses this CTA's shared memory after the barrier
    for (int t = tid; t < nq * R; t += W2_NT) {
        float s2 = 0.f;
#pragma unroll
        for (int c = 0; c < W2_CL; ++c) s2 += inbox[(((n_gemm - 1) & 1) ^ 1) * 32 * W2_FC * R + c * (W2_HQ * R) + t];
        w2_st_pair(ex.hg + ((size_t)cj * W2_HQ + t / R) * R + t % R, s2, ep_h);
    }
    if (blockIdx.x != 0) return;
    w2mark(marks, 2 + 4 * n_gemm);
    // all clusters' head partials: every thread polls its share of the n_clusters x nq x R pairs concurrently into shared
    // memory (the weight ring is idle now), then nq x R threads add the partials of one output in a fixed order
    {
        float* hcol = ring;   // [n_clusters][nq * R]
        const int n_pub = n_cta / W2_CL, per_cta = nq * R, total = n_pub * per_cta;
        constexpr int PPT = 18;
        for (int i0 = tid; i0 < total; i0 += W2_NT * PPT) {
            unsigned lo[PPT], hi[PPT], pending = 0, spins = 0;
#pragma unroll
            for (int m = 0; m < PPT; ++m)
                if (i0 + m * W2_NT < total) pending |= 1u << m;
            while (pending) {
#pragma unroll
                for (int m = 0; m < PPT; ++m)
                    if (pending & (1u << m)) {
                        const int i = i0 + m * W2_NT, c = i / per_cta, qr = i % per_cta;
                        const unsigned long long* src = ex.hg + ((size_t)c * W2_HQ + qr / R) * R + qr % R;
                        asm volatile("ld.volatile.global.v2.u32 {%0, %1}, [%2];" : "=r"(lo[m]), "=r"(hi[m]) : "l"(src) : "memory");
                    }
#pragma unroll
                for (int m = 0; m < PPT; ++m)
                    if ((pending & (1u << m)) && hi[m] == ep_h) {
                        hcol[i0 + m * W2_NT] = __uint_as_float(lo[m]);
                        pending &= ~(1u << m);
                    }
                if (++spins > (1u << 22)) {
                    if (p.err_flag != nullptr) *reinterpret_cast<volatile int*>(p.err_flag) = 3;
                    __threadfence_system();
                    __trap();
                }
            }
        }
        __syncthreads();
        for (int t = tid; t < per_cta; t += W2_NT) {
            const int q = t / R, r = t % R;
            float s2 = 0.f;
            for (int c = 0; c < n_pub; ++c) s2 += hcol[c * per_cta + t];   // fixed order: deterministic
            outs[r * OUT_LD + q] = s2 + cen[R * 4 + q];
        }
    }
    __syncthreads();
    w2mark(marks, 3 + 4 * n_gemm);
    if (tid < rows_here) store_row(p, (size_t)row0 + tid, outs + tid * OUT_LD, cen + tid * 4);
    if (p.n_gather) {
        __syncthreads();
        if (tid == 0) gather_finish(p);   // CTA 0 is the only storing CTA of this kernel
    }
    w2mark(marks, 4 + 4 * n_gemm);
}

// W^T [Kpad][L] -> per (cluster j, K slice i) slabs [L/32][4][kb][32], kb = min(L/4, Kpad) (rows beyond Kpad zero)
__global__ void wide2_pack_kernel(const float* __restrict__ wt, float* __restrict__ slab, int kpad, int L) {
    const int KS = L / W2_CL, kb = kpad < KS ? kpad : KS;
    const size_t n = (size_t)(L / W2_NC) * W2_CL * kb * W2_NC;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % W2_NC), k = (int)((i / W2_NC) % kb), ci = (int)((i / ((size_t)W2_NC * kb)) % W2_CL),
                  cj = (int)(i / ((size_t)W2_NC * kb * W2_CL));
        const int kg = ci * KS + k;
        slab[i] = kg < kpad ? wt[(size_t)kg * L + cj * W2_NC + c] : 0.f;
    }
}

static size_t wide2_smem(int L) {
    const int KS = L / W2_CL;
    return ((size_t)W2_NST * KS * W2_NC + (size_t)KS * W2_R + 2 * 32 * W2_FC * W2_R + (size_t)W2_R * OUT_LD + W2_R * 4 + W2_HQ +
            (size_t)MLB_MAX_OPS * 2 * W2_FC + (size_t)W2_HQ * W2_FC * W2_R) * sizeof(float) + W2_NST * sizeof(uint64_t) + 16;
}

}  // namespace mlb

using namespace mlb;

cudaError_t Wide2Family::set_marks(unsigned long long* ptr) { return cudaMemcpyToSymbol(mlb::g_wide2_marks, &ptr, sizeof(ptr)); }

cudaError_t Wide2Family::repack(const float* blob, const mlb_op* ops, int n_ops, int L, cudaStream_t st) const {
    if (!available) return cudaSuccess;
    for (int i = 0; i < n_ops; ++i)
        if (ops[i].type == MLB_OP_GEMM) wide2_pack_kernel<<<128, 256, 0, st>>>(blob + ops[i].w_off, slab + slab_off[i], ops[i].Kpad, L);
    return cudaGetLastError();
}

// all L/8 CTAs (L/32 clusters of 4) must be co-resident; heads and layer widths the kernel is written for
static bool wide2_supported(const mlb_op* ops, int n_ops, int L, int out_size, int n_sms) {
    if (L % 128 != 0 || L / W2_FC > n_sms || out_size > W2_HQ) return false;
    for (int i = 0; i < n_ops; ++i)
        if (ops[i].type == MLB_OP_GEMM && (ops[i].flags & MLB_F_IN_XIN) && ops[i].Kpad > L / W2_CL) return false;
    if (cudaFuncSetAttribute(loco_forward_wide2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wide2_smem(L)) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(L / W2_FC), cfg.blockDim = dim3(W2_NT), cfg.dynamicSmemBytes = wide2_smem(L);
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, loco_forward_wide2_kernel, &cfg) != cudaSuccess || n < L / W2_NC) {
        cudaGetLastError();
        return false;
    }
    return true;
}

cudaError_t Wide2Family::setup(const float* blob, const mlb_op* ops, int n_ops, int L, int out_size, int n_sms) {
    if (L > 1024 || !wide2_supported(ops, n_ops, L, out_size, n_sms)) return cudaSuccess;
    size_t off = 0;
    const int KS = L / W2_CL;
    for (int i = 0; i < n_ops; ++i) {
        slab_off[i] = (long long)off;
        if (ops[i].type == MLB_OP_GEMM) off += (size_t)(L / W2_NC) * W2_CL * (ops[i].Kpad < KS ? ops[i].Kpad : KS) * W2_NC;
    }
    cudaError_t e;
    if ((e = cudaMalloc(&slab, off * sizeof(float))) != cudaSuccess) return e;
    available = true;
    if ((e = repack(blob, ops, n_ops, L, 0)) != cudaSuccess) return e;
    if ((e = mlb_zalloc(&xg, (size_t)3 * L * W2_R * sizeof(unsigned long long))) != cudaSuccess) return e;
    return mlb_zalloc(&hg, (size_t)(L / W2_NC) * W2_HQ * W2_R * sizeof(unsigned long long));
}

void Wide2Family::release() {
    cudaFree(slab), cudaFree(xg), cudaFree(hg);
    slab = nullptr, xg = nullptr, hg = nullptr;
    available = false;
}

cudaError_t Wide2Family::launch(FwdParams p, const FwdPlan&, cudaStream_t st, int* issued) {
    Wide2Extra ex;
    ex.wslab = slab;
    for (int i = 0; i < MLB_MAX_OPS; ++i) ex.wslab_off[i] = i < p.n_ops ? slab_off[i] : 0;
    ex.xg = xg, ex.hg = hg, ex.epoch_base = epoch;
    p.n_tiles = 1, p.row_base = 0;
    // the opt-in shared-memory size is a per-function attribute of the PROCESS: another handle with a narrower model may have
    // lowered it since this one was created
    cudaError_t e = cudaFuncSetAttribute(loco_forward_wide2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wide2_smem(p.L));
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(p.L / W2_FC), cfg.blockDim = dim3(W2_NT), cfg.dynamicSmemBytes = wide2_smem(p.L), cfg.stream = st;
    cudaLaunchAttribute at;
    at.id = cudaLaunchAttributeCooperative;   // co-residency of all clusters: they spin on each other's outputs
    at.val.cooperative = 1;
    cfg.attrs = &at, cfg.numAttrs = 1;
    if ((e = cudaLaunchKernelEx(&cfg, loco_forward_wide2_kernel, p, ex)) != cudaSuccess) return e;
    unsigned n_epochs = 2;  // epochs one launch consumes
    for (int i = 0; i < p.n_ops; ++i) n_epochs += p.ops[i].type == MLB_OP_GEMM;
    epoch += n_epochs;
    ++*issued;
    return cudaSuccess;
}
