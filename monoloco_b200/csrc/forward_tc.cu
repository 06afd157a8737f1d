// monoloco_b200 -- throughput kernel on the 5th-gen tensor cores: the fp32 network as error-compensated TF32 products.
//
// The 1e-5 parity rule excludes plain TF32 / BF16 (SURVEY.md §0.4).  Here every fp32 operand is split into two TF32 terms,
// a = a_hi + a_lo (cvt.rna twice), and each layer product runs as THREE tcgen05.mma kind::tf32: a_hi.w_hi into a main TMEM
// accumulator, a_lo.w_hi + a_hi.w_lo into a second one (the dropped a_lo.w_lo term is 2^-22 relative).  Measured on the
// hardware (tools/probe_tc.py, tests/test_probe_tc_gpu.py): 2.6e-6 of max|ref| per 1024-deep layer against 6.8e-7 for an
// fp32 SGEMM -- the whole network stays at ~0.5 of the parity tolerance (tests force this kernel on every fixture).
//
// Replaces, like forward.cu, in ONE launch per detection batch (reference file:line):
//   monoloco/network/process.py:25-67 (pre-process), architectures.py:48-71 / 88-102 / 135-145 (network),
//   process.py:231-278, 330-360 + utils/camera.py:161-177, 202-237 (decode, xyz_from_distance).
//
//   weights      re-packed once per model: per GEMM op  [L/256 column tiles][K/16 k blocks][hi | lo][256 x 16]  (canonical
//                K-major no-swizzle UMMA layout: core matrix 8 rows x 16 B, SBO 128 B, LBO rows x 16 B) -> a pipeline stage
//                is two 1-D TMA bulk copies (16 KB of X planes + 32 KB of W planes), no tensor maps
//   kernel       persistent thread-block clusters, L/256 CTAs each (4 at L = 1024).  A cluster owns a private workspace slot
//                (input planes, two ping-pong activation plane sets, the fp32 residual: 2.6 MB, L2-resident for every
//                cluster at once) and walks 128-row tiles.  CTA n owns output columns [256n, 256n + 256) of every layer.
//   per tile     prologue: thread = row: pre-process the raw keypoints (process.py:47-67 / 25-44) straight into hi / lo planes
//                per layer: warp 1 lane 0 streams the stages through a 4-slot ring, warp 0 lane 0 issues 2 k-steps x 3 MMAs
//                (M 128, N 256, K 8) per stage and releases the stage with tcgen05.commit; all 128 threads (thread = row) read
//                main + cross back (tcgen05.ld), apply folded BN / ReLU / dropout / residual and write the result straight
//                into the next layer's hi / lo planes; narrow heads (w_aux, w_fin, MonolocoModel.w2) are accumulated on the
//                CUDA cores from the same registers; barrier.cluster separates the layers
//   tail         head partial sums -> CTA 0 through distributed shared memory -> decode_row -> stores (raw, decoded, xyz of
//                the bbox-centre ray, fused all-gather peers), exactly the epilogue of the FFMA kernels (fwd_common.cuh).
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "fwd_family.cuh"

namespace mlb {

constexpr int TCM = 128, TCN = 256, TCH = 128, TCKB = 16, TCNST = 4;   // row tile, columns per CTA, columns per epilogue half, k block, ring
constexpr uint32_t TC_A_PLANE = TCM * TCKB * 4;   // bytes of one X plane block (128 rows x 16 k)
constexpr uint32_t TC_W_PLANE = TCN * TCKB * 4;   // bytes of one W plane block (256 output columns x 16 k)
constexpr uint32_t TC_STAGE = 2 * TC_A_PLANE + 2 * TC_W_PLANE;   // 48 KB: X hi|lo + W hi|lo
constexpr uint32_t TC_LBO_A = TCM * 16, TC_LBO_W = TCN * 16, TC_SBO = 128;
constexpr uint32_t TC_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TCN >> 3) << 17) | ((uint32_t)(TCM >> 4) << 24);
constexpr int TC_MAX_CT = 8;       // column tiles = CTAs per cluster (L <= 2048)
constexpr int TC_HW = 16;          // head output columns in total (output_size <= 16)
constexpr int TC_EPI = 256;        // epilogue threads: (row, column half) -- warps w and w + 4 share a TMEM lane quarter
constexpr int TC_THREADS = 256;    // 8 warps: all epilogue; thread 0 also issues the MMAs, thread 128 also drives the TMA ring
constexpr size_t TC_RING_BYTES = (size_t)TCNST * TC_STAGE;                      // 192 KB
constexpr size_t TC_SST_BYTES = 2 * TCN * sizeof(float);                        // folded-BN scale | shift of the layer
constexpr size_t TC_HW_BYTES = (size_t)TC_HW * TCN * sizeof(float);             // head weights of the layer
constexpr size_t TC_SMEM_BYTES = TC_RING_BYTES + TC_SST_BYTES + TC_HW_BYTES;    // 210 KB

struct TcExtra {
    const float* wplanes[MLB_MAX_OPS];  // per GEMM op: [L/256 column tiles][n_kb][hi|lo][256 x 16]
    int n_kb[MLB_MAX_OPS];              // K blocks of 16 (K zero-padded)
    float* ws;                          // workspace, one slot per cluster
    unsigned long long slot_floats;
    int n_tiles;                        // 128-row tiles of this launch
    // narrow heads: rows of all head ops concatenated (q = 0 .. n_head_rows-1)
    int n_head_rows;
    int head_src[TC_HW];                // op index of the GEMM whose output head row q reads
    int head_col[TC_HW];                // raw output column of head row q
    long long head_w[TC_HW];            // float offset of head row q's K weights in the blob
    long long head_b[TC_HW];            // float offset of its bias
};

__device__ __forceinline__ float tc_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start >> 4 [0,14), LBO >> 4 [16,30), SBO >> 4 [32,46),
// version = 1 [46,48), layout type SWIZZLE_NONE [61,64)
__device__ __forceinline__ uint64_t tc_desc(uint32_t smem_addr, uint32_t lbo_bytes) {
    uint64_t d = (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((TC_SBO >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(TC_IDESC), "r"(accumulate), "r"(0u)
        : "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_epi_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }  // the 8 epilogue warps
__device__ __forceinline__ uint32_t tc_cluster_id() {  // clusters are laid out along x: one cluster per blockIdx.x
    return blockIdx.x;
}
// 16 consecutive TMEM columns of this thread's lane, asynchronous: complete after tc_ld_wait()
__device__ __forceinline__ void tc_ld16_async(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// float offset of element (row r, k) inside one [tile_rows x 16] plane
__device__ __forceinline__ size_t tc_plane_off(int r, int k_in_block, int tile_rows = TCM) {
    return (size_t)(k_in_block >> 2) * tile_rows * 4 + (size_t)(r >> 3) * 32 + (size_t)(r & 7) * 4 + (k_in_block & 3);
}

// W^T [Kpad][L] (the packed blob's layout) -> W planes [L/256][n_kb][hi|lo][256 x 16] with K padded to n_kb * 16
__global__ void tc_pack_weights_kernel(const float* __restrict__ wt, float* __restrict__ planes, int Kpad, int L, int n_kb) {
    const int K = n_kb * TCKB;
    const size_t plane = (size_t)TCN * TCKB;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)L * K; i += (size_t)gridDim.x * blockDim.x) {
        const int k = (int)(i / L), n = (int)(i % L);  // consecutive threads -> consecutive n: coalesced reads of W^T
        const float v = k < Kpad ? wt[(size_t)k * L + n] : 0.f;
        const float h = tc_tf32(v), l = tc_tf32(v - h);
        float* blk = planes + ((size_t)(n / TCN) * n_kb + k / TCKB) * 2 * plane;
        const size_t off = tc_plane_off(n % TCN, k % TCKB, TCN);
        blk[off] = h;
        blk[plane + off] = l;
    }
}

// profiling aid (mlb_debug_fwd_marks): CTA (0,0) stamps %globaltimer per layer of its first tile: thread 0 at [8g+0] layer start,
// [8g+3] accumulators complete, [8g+4] epilogue done, [8g+5] cluster barrier passed; MMA lane at [8g+1] first stage landed,
// [8g+2] all MMAs issued; producer lane at [8g+6] all stages issued
__device__ unsigned long long* g_tc_marks = nullptr;
__device__ __forceinline__ void tmark(unsigned long long* marks, int slot) {
    if (marks != nullptr) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        marks[slot] = t;
    }
}

struct TcEpi {            // what one epilogue pass over a 128-column half needs
    uint32_t tmem_main;   // TMEM address of this thread's lane, main accumulator of the half (cross terms at + 256)
    const float* sst;     // shared: scale[256] | shift[256] of the CTA's columns
    const float* hw;      // shared: [NQ][256] weights of the head rows this layer feeds (zero rows beyond the real ones)
    float* nxt;           // next layer's X planes (cluster slot)
    float* res;           // fp32 residual [L/4][128][4] (cluster slot)
    int col0;             // first global column of the half
    int ccol0;            // first CTA-local column of the half (0 or 128)
    int tid, grow, site;
    bool live, relu, add_res, save_res, drop, write_planes;
    const uint8_t* drop_mask;
    int n_rows, L;
    uint32_t rm, thr;
    float inv_keep;
    uint64_t keep;        // L2 evict_last policy for the residual
};

// The fp32 residual of a stage is written two layers before it is read: ~110 MB of other L2 traffic pass in between and
// plain LRU had evicted it to HBM by then (100 MB of DRAM round trips per batch of 4096).  L2::evict_last keeps it resident.
__device__ __forceinline__ uint64_t tc_policy_evict_last() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void tc_st_keep(float* ptr, float4 v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(ptr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol)
                 : "memory");
}
__device__ __forceinline__ float4 tc_ld_keep(const float* ptr, uint64_t pol) {
    float4 v;
    asm volatile("ld.global.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(ptr), "l"(pol));
    return v;
}

// MC-dropout of four consecutive columns (rare path, kept out of line: the epilogue loops must stay small enough for the
// instruction cache -- fully unrolled they were 140 KB per instantiation and every first use cost ~15 us of code fetch)
__device__ __noinline__ float4 tc_dropout4(float4 v, const uint8_t* mask_row, uint32_t rm, uint32_t thr, float inv_keep, int gc, int site,
                                           int live) {
    float o[4] = {v.x, v.y, v.z, v.w};
    if (mask_row != nullptr) {
        if (live) {
            const uint32_t mk = *reinterpret_cast<const uint32_t*>(mask_row + gc);
#pragma unroll
            for (int t = 0; t < 4; ++t) o[t] = ((mk >> (8 * t)) & 0xFFu) ? o[t] * inv_keep : 0.f;
        }
    } else {
#pragma unroll
        for (int t = 0; t < 4; ++t) o[t] = drop_keep(rm, drop_col_hash((uint32_t)(gc + t), (uint32_t)site), thr) ? o[t] * inv_keep : 0.f;
    }
    return make_float4(o[0], o[1], o[2], o[3]);
}

constexpr int TC_CW = 16;   // accumulator columns per epilogue chunk (one tcgen05.ld x16 per accumulator)

// One 16-column chunk of this thread's row: BN affine / ReLU / dropout / residual, head partial sums, hi / lo planes out.
template <int NQ, int OFF, bool ADD>
__device__ __forceinline__ void tc_epilogue_chunk(const TcEpi& e, int ch, const uint32_t* mb, const uint32_t* cb, const float4* rr,
                                                  float* hacc) {
    constexpr size_t plane = (size_t)TCM * TCKB;
#pragma unroll
    for (int j4 = 0; j4 < TC_CW / 4; ++j4) {
        const int lc = e.ccol0 + TC_CW * ch + 4 * j4;   // CTA-local column
        const int gc = e.col0 + TC_CW * ch + 4 * j4;    // global column = k index of the next layer
        const float4 sc = *reinterpret_cast<const float4*>(e.sst + lc);
        const float4 sh = *reinterpret_cast<const float4*>(e.sst + TCN + lc);
        float v[4];
        v[0] = fmaf(__uint_as_float(mb[4 * j4 + 0]) + __uint_as_float(cb[4 * j4 + 0]), sc.x, sh.x);
        v[1] = fmaf(__uint_as_float(mb[4 * j4 + 1]) + __uint_as_float(cb[4 * j4 + 1]), sc.y, sh.y);
        v[2] = fmaf(__uint_as_float(mb[4 * j4 + 2]) + __uint_as_float(cb[4 * j4 + 2]), sc.z, sh.z);
        v[3] = fmaf(__uint_as_float(mb[4 * j4 + 3]) + __uint_as_float(cb[4 * j4 + 3]), sc.w, sh.w);
        if (e.relu) {
#pragma unroll
            for (int t = 0; t < 4; ++t) v[t] = fmaxf(v[t], 0.f);
        }
        if (e.drop) {
            const uint8_t* mrow = e.drop_mask ? e.drop_mask + ((size_t)e.site * e.n_rows + e.grow) * e.L : nullptr;
            const float4 d = tc_dropout4(make_float4(v[0], v[1], v[2], v[3]), mrow, e.rm, e.thr, e.inv_keep, gc, e.site, (int)e.live);
            v[0] = d.x, v[1] = d.y, v[2] = d.z, v[3] = d.w;
        }
        float* rq = e.res + ((size_t)(gc >> 2) * TCM + e.tid) * 4;   // a warp touches 512 contiguous bytes
        if (ADD) {
            const float4 r = rr[j4];
            v[0] += r.x, v[1] += r.y, v[2] += r.z, v[3] += r.w;
        }
        if (e.save_res) tc_st_keep(rq, make_float4(v[0], v[1], v[2], v[3]), e.keep);
#pragma unroll
        for (int q = 0; q < NQ; ++q) {   // narrow heads on this layer's output: partial dot products over my columns
            const float4 w = *reinterpret_cast<const float4*>(e.hw + q * TCN + lc);
            hacc[OFF + q] = fmaf(v[3], w.w, fmaf(v[2], w.z, fmaf(v[1], w.y, fmaf(v[0], w.x, hacc[OFF + q]))));
        }
        if (e.write_planes) {   // the last layer's output only feeds the heads
            float* blk = e.nxt + (size_t)(gc / TCKB) * 2 * plane;
            const float4 h = make_float4(tc_tf32(v[0]), tc_tf32(v[1]), tc_tf32(v[2]), tc_tf32(v[3]));
            const float4 l = make_float4(tc_tf32(v[0] - h.x), tc_tf32(v[1] - h.y), tc_tf32(v[2] - h.z), tc_tf32(v[3] - h.w));
            const size_t off = tc_plane_off(e.tid, gc % TCKB);
            *reinterpret_cast<float4*>(blk + off) = h;
            *reinterpret_cast<float4*>(blk + plane + off) = l;
        }
    }
}

// The 128 accumulator columns of this thread's row, two chunks per (rolled) loop trip; TMEM loads and residual loads are
// double-buffered: the next chunk is in flight while the current one is processed.
template <int NQ, int OFF, bool ADD>
__device__ __forceinline__ void tc_epilogue_half(const TcEpi& e, float* hacc) {
    constexpr int NCH = TCH / TC_CW, RW = ADD ? TC_CW / 4 : 1;
    uint32_t mb0[TC_CW], cb0[TC_CW], mb1[TC_CW], cb1[TC_CW];
    float4 rr0[RW], rr1[RW];
    const float* res_row = e.res + ((size_t)(e.col0 >> 2) * TCM + e.tid) * 4;   // + 512 floats per 4 columns
    auto fetch = [&](int ch, uint32_t* mb, uint32_t* cb, float4* rr) {
        tc_ld16_async(e.tmem_main + (uint32_t)(TC_CW * ch), mb);
        tc_ld16_async(e.tmem_main + 256u + (uint32_t)(TC_CW * ch), cb);
        if (ADD) {
#pragma unroll
            for (int j4 = 0; j4 < TC_CW / 4; ++j4)
                rr[j4] = tc_ld_keep(res_row + (size_t)(ch * (TC_CW / 4) + j4) * TCM * 4, e.keep);
        }
    };
    fetch(0, mb0, cb0, rr0);
    tc_ld_wait();
#pragma unroll 1
    for (int ch = 0; ch < NCH; ch += 2) {
        fetch(ch + 1, mb1, cb1, rr1);
        tc_epilogue_chunk<NQ, OFF, ADD>(e, ch, mb0, cb0, rr0, hacc);
        tc_ld_wait();
        if (ch + 2 < NCH) fetch(ch + 2, mb0, cb0, rr0);
        tc_epilogue_chunk<NQ, OFF, ADD>(e, ch + 1, mb1, cb1, rr1, hacc);
        tc_ld_wait();
    }
}

__global__ void __launch_bounds__(TC_THREADS, 1) loco_forward_tc_kernel(const __grid_constant__ FwdParams p,
                                                                        const __grid_constant__ TcExtra ex) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t full[TCNST], empty[TCNST], done;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nt = blockIdx.y, nct = gridDim.y, L = p.L;
    const bool epi_thread = true, prod_lane = tid == 128, mma_lane = tid == 0;
    const int half = (tid >> 7) & 1;   // epilogue threads: which 128 columns of the CTA's 256
    float* sst = reinterpret_cast<float*>(smem_raw + TC_RING_BYTES);                 // [2][256]
    float* hw = reinterpret_cast<float*>(smem_raw + TC_RING_BYTES + TC_SST_BYTES);   // [TC_HW][256]
    float* hpart = reinterpret_cast<float*>(smem_raw);                               // [2 nct][128][TC_HW] on CTA 0; aliases the idle ring

    if (tid == 0) {
        for (int s = 0; s < TCNST; ++s) mbar_init(&full[s], 1), mbar_init(&empty[s], 1);
        mbar_init(&done, 1);
        mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(&tmem_slot, 512);  // main accumulator [0,256), cross terms [256,512)
    tmem_fence_before();
    __syncthreads();
    tmem_fence_after();
    tc_cluster_sync();  // every CTA of the cluster is resident before any remote shared-memory store can be issued
    const uint32_t tmem = tmem_slot;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);

    // this cluster's workspace slot
    int first_gemm = 0;
    while (p.ops[first_gemm].type != MLB_OP_GEMM) ++first_gemm;
    const int n_kb0 = ex.n_kb[first_gemm];
    const size_t plane = (size_t)TCM * TCKB;
    float* slot = ex.ws + (size_t)tc_cluster_id() * ex.slot_floats;
    float* xin = slot;                                   // [n_kb0][hi|lo][128 x 16]
    float* xpl[2] = {xin + (size_t)n_kb0 * 2 * plane, xin + (size_t)n_kb0 * 2 * plane + (size_t)(L / TCKB) * 2 * plane};
    float* res = xpl[1] + (size_t)(L / TCKB) * 2 * plane;  // [L/4][128][4] fp32

    const float zm = p.z_met;
    const float k0 = p.kinv[0], k1 = p.kinv[1], k2 = p.kinv[2], k3 = p.kinv[3], k4 = p.kinv[4], k5 = p.kinv[5];
    const bool mc_drop = (p.flags & MLB_FWD_DROPOUT) != 0;
    // head rows are grouped by the layer that feeds them (at most two groups: w_aux | w_fin, or MonolocoModel.w2); group g
    // accumulates into hacc[off_g .. off_g + nq_g), nq_g = its row count rounded up to 4 (zero weights beyond the real rows)
    int grp_src[2] = {-1, -1}, grp_q0[2] = {0, 0}, grp_n[2] = {0, 0};
    for (int q = 0; q < ex.n_head_rows; ++q) {
        const int g = (grp_src[0] < 0 || grp_src[0] == ex.head_src[q]) ? 0 : 1;
        if (grp_n[g] == 0) grp_src[g] = ex.head_src[q], grp_q0[g] = q;
        grp_n[g]++;
    }
    int n_gemm = 0;
    for (int oi = 0; oi < p.n_ops; ++oi) n_gemm += p.ops[oi].type == MLB_OP_GEMM;
    const int grp_nq[2] = {(grp_n[0] + 3) & ~3, (grp_n[1] + 3) & ~3};
    const int grp_off[2] = {0, grp_nq[0]};

    unsigned long long* marks = (blockIdx.x == 0 && blockIdx.y == 0 && (tid == 0 || tid == 128)) ? g_tc_marks : nullptr;
    unsigned it_p = 0, it_m = 0;  // stages issued / consumed so far (producer lane, MMA lane)
    unsigned n_done = 0;          // layers finished by this CTA (parity of `done`)
    for (int rb = (int)tc_cluster_id(); rb < ex.n_tiles; rb += (int)gridDim.x) {
        const int row = tid & 127;            // epilogue threads: my row of the tile
        const int grow = rb * TCM + row;      // my detection
        const bool live = epi_thread && grow < p.n_rows;
        const bool row_owner = epi_thread && half == 0;   // one thread per row does the prologue / the final store
        float cenrow[4] = {0.f, 0.f, 0.f, 0.f};

        // ------------------------------------------------------------ prologue: network input of my row -> hi / lo planes
        // every CTA of the cluster evaluates its row (cheap); CTA nt writes k blocks nt, nt + nct, ...
        if (row_owner) {
            float xr[KIN_MAX + 8];
#pragma unroll
            for (int k = 0; k < KIN_MAX + 8; ++k) xr[k] = 0.f;
            if (live) {
                if (p.input_kind == MLB_IN_X) {
#pragma unroll
                    for (int k = 0; k < KIN_MAX; ++k)
                        if (k < p.in_size) xr[k] = __ldg(p.x + (size_t)grow * p.in_size + k);
                } else {
                    const bool stereo = p.input_kind == MLB_IN_KPS_STEREO;
                    const float* kp = p.x + (size_t)(stereo ? grow / p.n_right : grow) * 51;
                    const float* kr = stereo ? p.xr + (size_t)(grow % p.n_right) * 51 : nullptr;
                    float umin = __ldg(kp), umax = umin, vmin = __ldg(kp + 17), vmax = vmin;
                    for (int j = 1; j < 17; ++j) {
                        const float u = __ldg(kp + j), v = __ldg(kp + 17 + j);
                        umin = fminf(umin, u), umax = fmaxf(umax, u);
                        vmin = fminf(vmin, v), vmax = fmaxf(vmax, v);
                    }
                    const float uc = __fadd_rn(__fdiv_rn(__fsub_rn(umax, umin), 2.f), umin);  // camera.py:82-86
                    const float vc = __fadd_rn(__fdiv_rn(__fsub_rn(vmax, vmin), 2.f), vmin);
                    cenrow[0] = uc, cenrow[1] = vc;
                    cenrow[2] = (uc * k0 + vc * k1 + k2) * zm;
                    cenrow[3] = (uc * k3 + vc * k4 + k5) * zm;
                    const bool zc = (p.flags & MLB_FWD_ZERO_CENTER) != 0;
#pragma unroll
                    for (int j = 0; j < 17; ++j) {
                        const float u = __ldg(kp + j), v = __ldg(kp + 17 + j);
                        float xl = (u * k0 + v * k1 + k2) * zm;  // camera.py:26-27, rows 0/1 of [u v 1] K^-T
                        float yl = (u * k3 + v * k4 + k5) * zm;
                        if (stereo) {
                            const float ur = __ldg(kr + j), vr = __ldg(kr + 17 + j);
                            xr[34 + 2 * j] = xl - (ur * k0 + vr * k1 + k2) * zm;  // process.py:41 cat(l, l - r)
                            xr[35 + 2 * j] = yl - (ur * k3 + vr * k4 + k5) * zm;
                        } else if (zc) {
                            xl -= cenrow[2];  // process.py:61-62
                            yl -= cenrow[3];
                        }
                        xr[2 * j] = xl, xr[2 * j + 1] = yl;
                    }
                }
                if (nt == 0 && p.out_x != nullptr && p.input_kind != MLB_IN_X) {
#pragma unroll
                    for (int k = 0; k < KIN_MAX; ++k)
                        if (k < p.in_size) p.out_x[(size_t)grow * p.in_size + k] = xr[k];
                }
            }
#pragma unroll
            for (int kb = 0; kb < (KIN_MAX + 8) / TCKB; ++kb) {
                if (kb < n_kb0 && (kb % nct) == nt) {
                    float* blk = xin + (size_t)kb * 2 * plane;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float4 v = make_float4(xr[kb * 16 + 4 * q], xr[kb * 16 + 4 * q + 1], xr[kb * 16 + 4 * q + 2], xr[kb * 16 + 4 * q + 3]);
                        const float4 h = make_float4(tc_tf32(v.x), tc_tf32(v.y), tc_tf32(v.z), tc_tf32(v.w));
                        const float4 l = make_float4(tc_tf32(v.x - h.x), tc_tf32(v.y - h.y), tc_tf32(v.z - h.z), tc_tf32(v.w - h.w));
                        const size_t off = tc_plane_off(row, 4 * q);
                        *reinterpret_cast<float4*>(blk + off) = h;
                        *reinterpret_cast<float4*>(blk + plane + off) = l;
                    }
                }
            }
        }
        tc_cluster_sync();  // the input planes of this tile are complete (and the previous tile's tail is over everywhere)

        float hacc[TC_HW];
#pragma unroll
        for (int q = 0; q < TC_HW; ++q) hacc[q] = 0.f;

        int par = 0, site = 0, gi = 0;  // gi: GEMM ops done in this tile
        for (int oi = 0; oi < p.n_ops; ++oi) {
            const mlb_op& op = p.ops[oi];
            if (op.type != MLB_OP_GEMM) continue;
            const int n_kb = ex.n_kb[oi];
            const float* xsrc_f = gi == 0 ? xin : xpl[par];
            unsigned long long* mk = (rb == 0 && gi < 15) ? marks : nullptr;
            if (tid == 0) tmark(mk, 8 * gi + 0);
            const int hg = grp_src[0] == oi ? 0 : (grp_src[1] == oi ? 1 : -1);   // head group fed by this layer
            const bool head_layer = hg >= 0;

            if (prod_lane) {
                // ---- producer: this row tile's X planes and this column tile's W planes, 48 KB per stage
                asm volatile("fence.proxy.async;" ::: "memory");  // peers' generic-proxy stores (planes, hpart) -> async-proxy TMA
                const unsigned char* xsrc = reinterpret_cast<const unsigned char*>(xsrc_f);
                const unsigned char* wsrc = reinterpret_cast<const unsigned char*>(ex.wplanes[oi]) + (size_t)nt * n_kb * 2 * TC_W_PLANE;
                for (int kb = 0; kb < n_kb; ++kb, ++it_p) {
                    const unsigned s = it_p % TCNST;
                    if (it_p >= TCNST) mbar_wait(&empty[s], ((it_p / TCNST) - 1) & 1, p.err_flag);
                    unsigned char* st = smem_raw + (size_t)s * TC_STAGE;
                    mbar_expect_tx(&full[s], TC_STAGE);
                    tma_bulk_g2s(st, xsrc + (size_t)kb * 2 * TC_A_PLANE, 2 * TC_A_PLANE, &full[s]);
                    tma_bulk_g2s(st + 2 * TC_A_PLANE, wsrc + (size_t)kb * 2 * TC_W_PLANE, 2 * TC_W_PLANE, &full[s]);
                }
                tmark(mk, 8 * gi + 6);
            } else if (mma_lane) {
                // ---- MMA issuer: 2 k-steps x 3 MMAs (M 128, N 256, K 8) per stage
                tmem_fence_after();
                uint32_t main_acc = 0, cross_acc = 0;
                for (int kb = 0; kb < n_kb; ++kb, ++it_m) {
                    const unsigned s = it_m % TCNST;
                    mbar_wait(&full[s], (it_m / TCNST) & 1, p.err_flag);
                    if (kb == 0) tmark(mk, 8 * gi + 1);
                    tmem_fence_after();
                    const uint32_t a_hi = smem_u32(smem_raw + (size_t)s * TC_STAGE), a_lo = a_hi + TC_A_PLANE;
                    const uint32_t w_hi = a_hi + 2 * TC_A_PLANE, w_lo = w_hi + TC_W_PLANE;
#pragma unroll
                    for (int j = 0; j < TCKB / 8; ++j) {
                        const uint64_t ah = tc_desc(a_hi + 2 * j * TC_LBO_A, TC_LBO_A), al = tc_desc(a_lo + 2 * j * TC_LBO_A, TC_LBO_A);
                        const uint64_t wh = tc_desc(w_hi + 2 * j * TC_LBO_W, TC_LBO_W), wl = tc_desc(w_lo + 2 * j * TC_LBO_W, TC_LBO_W);
                        tc_mma(tmem + 256u, al, wh, cross_acc), cross_acc = 1;
                        tc_mma(tmem + 256u, ah, wl, 1u);
                        tc_mma(tmem, ah, wh, main_acc), main_acc = 1;
                    }
                    tc_commit(&empty[s]);
                }
                tc_commit(&done);
                tmark(mk, 8 * gi + 2);
            } else if (warp != 0 && warp != 4) {
                // ---- the other six warps, while the MMAs run: this layer's epilogue constants -> shared memory
                const int st = tid < 128 ? tid - 32 : tid - 64;   // 0 .. 191
                for (int i = st; i < 2 * TCN; i += 192)
                    sst[i] = __ldg(p.blob + (i < TCN ? op.scale_off : op.shift_off) + nt * TCN + (i & (TCN - 1)));
                if (head_layer) {
                    for (int i = st; i < grp_nq[hg] * TCN; i += 192) {
                        const int r = i / TCN, c = i % TCN;
                        hw[i] = r < grp_n[hg] ? __ldg(p.blob + ex.head_w[grp_q0[hg] + r] + nt * TCN + c) : 0.f;
                    }
                }
            }
            __syncwarp();
            {
                tc_epi_sync();
                TcEpi e;
                e.sst = sst, e.hw = hw, e.nxt = xpl[gi == 0 ? 0 : (par ^ 1)], e.res = res;
                e.tid = row, e.grow = grow, e.site = site, e.live = live;
                e.relu = (op.flags & MLB_F_RELU) != 0, e.add_res = (op.flags & MLB_F_ADD_RES) != 0;
                e.save_res = (op.flags & MLB_F_SAVE_RES) != 0, e.drop = mc_drop && (op.flags & MLB_F_DROPOUT) != 0;
                e.write_planes = gi + 1 < n_gemm;
                e.drop_mask = p.drop_mask, e.n_rows = p.n_rows, e.L = L;
                e.rm = drop_row_mix(drop_seed_mix(p.drop_seed), (uint32_t)grow), e.thr = drop_threshold(p.p_drop);
                e.inv_keep = 1.0f / (1.0f - p.p_drop);
                e.keep = tc_policy_evict_last();
                mbar_wait_backoff(&done, (uint32_t)(n_done & 1), p.err_flag);
                tmem_fence_after();
                if (tid == 0) tmark(mk, 8 * gi + 3);
                e.tmem_main = lane_base + (uint32_t)(TCH * half);
                e.ccol0 = TCH * half, e.col0 = nt * TCN + TCH * half;
                if (!head_layer) {
                    if (e.add_res) tc_epilogue_half<0, 0, true>(e, hacc);
                    else tc_epilogue_half<0, 0, false>(e, hacc);
                } else if (e.add_res) {   // MonolocoModel: the last stage's output (x + y) feeds the only head
                    const int nqg = grp_nq[hg];
                    if (nqg <= 4) tc_epilogue_half<4, 0, true>(e, hacc);
                    else if (nqg <= 8) tc_epilogue_half<8, 0, true>(e, hacc);
                    else if (nqg <= 12) tc_epilogue_half<12, 0, true>(e, hacc);
                    else tc_epilogue_half<16, 0, true>(e, hacc);
                } else {   // (rows of this group rounded to 4, offset of the group)
                    const int nqg = grp_nq[hg], off = grp_off[hg];
                    if (off == 0) {
                        if (nqg <= 4) tc_epilogue_half<4, 0, false>(e, hacc);
                        else if (nqg <= 8) tc_epilogue_half<8, 0, false>(e, hacc);
                        else if (nqg <= 12) tc_epilogue_half<12, 0, false>(e, hacc);
                        else tc_epilogue_half<16, 0, false>(e, hacc);
                    } else if (off == 4) {
                        if (nqg <= 4) tc_epilogue_half<4, 4, false>(e, hacc);
                        else if (nqg <= 8) tc_epilogue_half<8, 4, false>(e, hacc);
                        else tc_epilogue_half<12, 4, false>(e, hacc);
                    } else if (off == 8) {
                        if (nqg <= 4) tc_epilogue_half<4, 8, false>(e, hacc);
                        else tc_epilogue_half<8, 8, false>(e, hacc);
                    } else {
                        tc_epilogue_half<4, 12, false>(e, hacc);
                    }
                }
                if (tid == 0) tmark(mk, 8 * gi + 4);
            }
            ++n_done;
            if (op.flags & MLB_F_DROPOUT) site++;
            __syncwarp();
            tmem_fence_before();
            tc_cluster_sync();  // all column tiles of this row tile are written; TMEM reads are complete
            tmem_fence_after();
            if (tid == 0) tmark(mk, 8 * gi + 5);
            // The planes this layer read are dead now (every CTA of the cluster is past its MMAs) and will be fully
            // rewritten before their next use: drop the dirty lines from L2 instead of letting them be written back to
            // HBM (discard.global.L2; without it the workspace churn was 255 MB of DRAM writes per batch of 4096).
            {
                const size_t lines = (size_t)n_kb * 2 * TC_A_PLANE / 128;   // 128-byte lines; CTA nt takes lines nt, nt + nct, ...
                const unsigned char* base = reinterpret_cast<const unsigned char*>(xsrc_f);
                for (size_t ln = (size_t)nt + (size_t)nct * tid; ln < lines; ln += (size_t)nct * TC_THREADS)
                    asm volatile("discard.global.L2 [%0], 128;" ::"l"(base + ln * 128) : "memory");
                if ((op.flags & MLB_F_ADD_RES) && !(op.flags & MLB_F_SAVE_RES)) {   // last use of the stage residual
                    const unsigned char* rb = reinterpret_cast<const unsigned char*>(res + (size_t)(nt * TCN / 4) * TCM * 4);
                    for (size_t o = (size_t)tid * 128; o < (size_t)TCN * TCM * 4; o += (size_t)TC_THREADS * 128)
                        asm volatile("discard.global.L2 [%0], 128;" ::"l"(rb + o) : "memory");
                }
            }
            if (gi > 0) par ^= 1;
            ++gi;
        }

        // ------------------------------------------------------------ tail: head partials -> CTA 0 -> decode + stores
        if (epi_thread) {
            const uint32_t local = smem_u32(hpart + ((size_t)(2 * nt + half) * TCM + row) * TC_HW);
            uint32_t remote;
            asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local), "r"(0u));
#pragma unroll
            for (int q4 = 0; q4 < TC_HW / 4; ++q4)
                asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(remote + 16u * q4), "f"(hacc[4 * q4]),
                             "f"(hacc[4 * q4 + 1]), "f"(hacc[4 * q4 + 2]), "f"(hacc[4 * q4 + 3])
                             : "memory");
        }
        tc_cluster_sync();
        if (nt == 0 && live && row_owner) {
            float o[OUT_LD];
#pragma unroll
            for (int k = 0; k < OUT_LD; ++k) o[k] = 0.f;
            for (int q = 0; q < ex.n_head_rows; ++q) {
                const int g = (q >= grp_q0[1] && grp_n[1] > 0) ? 1 : 0;
                const int slot = grp_off[g] + (q - grp_q0[g]);
                float s = 0.f;
                for (int t = 0; t < 2 * nct; ++t) s += hpart[((size_t)t * TCM + row) * TC_HW + slot];  // fixed order: deterministic
                o[ex.head_col[q]] = s + __ldg(p.blob + ex.head_b[q]);
            }
            store_row(p, (size_t)grow, o, cenrow, p.n_gather ? hw + (size_t)row * MLB_GATHER_LD : nullptr);
        }
        if (nt == 0 && p.n_gather) {
            // fused all-gather: the tile's rows ([<=128][20] floats, contiguous in every gather buffer) leave as coalesced
            // 16-byte stores -- 128-byte NVLink packets instead of 11 scattered 4..16-byte stores per row and peer
            // (`hw` is free here: the head layers are done; it is re-staged in the next tile's first head layer)
            __syncthreads();
            const int rows_live = min(TCM, p.n_rows - rb * TCM);
            const int n4 = rows_live * (MLB_GATHER_LD / 4);
            const float4* src = reinterpret_cast<const float4*>(hw);
            for (int pg = 0; pg < p.n_gather; ++pg) {
                float4* dst = reinterpret_cast<float4*>(p.gather[pg] + (size_t)(p.gather_row0 + (long long)rb * TCM) * MLB_GATHER_LD);
                for (int i = tid; i < n4; i += TC_THREADS) dst[i] = src[i];
            }
            __syncthreads();   // peer stores ordered before this CTA's arrival in gather_finish() (barrier + its fence)
        }
        // the next tile's prologue ends with a cluster barrier: CTA 0 has finished reading hpart before any peer writes it
        // again, and before its own producer refills the ring that hpart aliases (program order + fence.proxy.async)
    }
    if (nt == 0) {
        __syncthreads();  // every storing thread has fenced its peer stores (store_row)
        if (tid == 0) gather_finish(p);  // fused all-gather: one arrival per cluster leader
    }
    tc_cluster_sync();  // no CTA exits while a peer may still address its shared memory
    tmem_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

}  // namespace mlb

// ================================================================================================ host side
using namespace mlb;

cudaError_t TcFamily::set_marks(unsigned long long* ptr) { return cudaMemcpyToSymbol(mlb::g_tc_marks, &ptr, sizeof(ptr)); }

static void tc_config(cudaLaunchConfig_t* cfg, cudaLaunchAttribute* at, int clusters, int nct, cudaStream_t st) {
    memset(cfg, 0, sizeof(*cfg));
    cfg->gridDim = dim3(clusters, nct);
    cfg->blockDim = dim3(TC_THREADS);
    cfg->dynamicSmemBytes = TC_SMEM_BYTES;
    cfg->stream = st;
    at->id = cudaLaunchAttributeClusterDimension;
    at->val.clusterDim.x = 1, at->val.clusterDim.y = nct, at->val.clusterDim.z = 1;
    cfg->attrs = at;
    cfg->numAttrs = 1;
}

cudaError_t TcFamily::repack(const float* blob, const mlb_op* ops, int n_ops, int L, cudaStream_t st) const {
    if (!available) return cudaSuccess;
    for (int i = 0; i < n_ops; ++i)
        if (ops[i].type == MLB_OP_GEMM)
            tc_pack_weights_kernel<<<296, 256, 0, st>>>(blob + ops[i].w_off, wplanes[i], ops[i].Kpad, L, n_kb[i]);
    return cudaGetLastError();
}

// widths the tensor-core kernel covers: 256 output columns per CTA, clusters of up to 8 CTAs
bool TcFamily::covers(int L) { return L >= TCN && L % TCN == 0 && L / TCN <= TC_MAX_CT; }

// pack the weight planes, size the workspace (one slot per co-resident cluster)
cudaError_t TcFamily::setup(const float* blob, const mlb_op* ops, int n_ops, int L) {
    if (!covers(L)) return cudaSuccess;
    nct = L / TCN;
    cudaError_t e = cudaFuncSetAttribute(loco_forward_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM_BYTES);
    int first = -1;
    for (int i = 0; i < n_ops && e == cudaSuccess; ++i) {
        if (ops[i].type != MLB_OP_GEMM) continue;
        if (first < 0) first = i;
        n_kb[i] = (ops[i].Kpad + TCKB - 1) / TCKB;
        e = cudaMalloc(&wplanes[i], (size_t)2 * n_kb[i] * TCKB * L * sizeof(float));
    }
    available = e == cudaSuccess;
    if (e == cudaSuccess) e = repack(blob, ops, n_ops, L, 0);
    if (e == cudaSuccess) {
        cudaLaunchConfig_t cfg;
        cudaLaunchAttribute at;
        tc_config(&cfg, &at, 64, nct, 0);
        if (cudaOccupancyMaxActiveClusters(&max_clusters, loco_forward_tc_kernel, &cfg) != cudaSuccess || max_clusters < 1) {
            cudaGetLastError();
            max_clusters = 148 / nct / 2;
        }
        const size_t plane = (size_t)TCM * TCKB;
        slot_floats = (size_t)n_kb[first] * 2 * plane + 2 * (size_t)(L / TCKB) * 2 * plane + (size_t)TCM * L;
        e = cudaMalloc(&ws, (size_t)max_clusters * slot_floats * sizeof(float));
    }
    if (e == cudaSuccess) e = cudaMemsetAsync(ws, 0, (size_t)max_clusters * slot_floats * sizeof(float), 0);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) release();
    return e;
}

void TcFamily::release() {
    for (int i = 0; i < MLB_MAX_OPS; ++i) cudaFree(wplanes[i]), wplanes[i] = nullptr;
    cudaFree(ws);
    ws = nullptr;
    available = false;
}

cudaError_t TcFamily::launch(FwdParams p, const FwdPlan& pl, cudaStream_t st, int* issued) const {
    TcExtra ex;
    memset(&ex, 0, sizeof(ex));
    for (int i = 0; i < MLB_MAX_OPS; ++i) ex.wplanes[i] = wplanes[i], ex.n_kb[i] = n_kb[i];
    ex.ws = ws, ex.slot_floats = slot_floats;
    ex.n_tiles = (p.n_rows + TCM - 1) / TCM;
    int last_gemm = -1;
    for (int i = 0; i < p.n_ops; ++i) {
        const mlb_op& op = p.ops[i];
        if (op.type == MLB_OP_GEMM) {
            last_gemm = i;
        } else {
            if (last_gemm < 0) return cudaErrorInvalidValue;
            for (int o = 0; o < op.N; ++o) {
                if (ex.n_head_rows >= TC_HW) return cudaErrorInvalidValue;
                const int q = ex.n_head_rows++;
                ex.head_src[q] = last_gemm, ex.head_col[q] = op.out_col + o;
                ex.head_w[q] = op.w_off + (long long)o * op.K, ex.head_b[q] = op.shift_off + o;
            }
        }
    }
    p.flags &= ~MLB_FWD_RES_TMEM;  // the residual always goes through the scratch here
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute at;
    tc_config(&cfg, &at, pl.clusters, nct, st);
    cudaError_t e = cudaLaunchKernelEx(&cfg, loco_forward_tc_kernel, p, ex);
    if (e == cudaSuccess) ++*issued;
    return e;
}
