// Latency-oriented inference kernel for SMALL detection batches (the reference's real per-image regime: m = 1..30
// detections per call, predict.py:231; BASELINE configs[0]/[1] batch 1 / 256).
//
// The throughput kernel (forward.cu) gives one CTA a whole row tile, so a batch of <= 32 detections runs on ONE SM and
// is bound by that SM's L2->SMEM weight stream (34 MB at ~40 B/clk = 1 ms).  Here a thread-block CLUSTER of 8 CTAs
// shares a tile of 16 detections and splits every 1024-wide layer by output columns: CTA r owns columns
// [128 r, 128 r + 128) and streams only its 4 KB-per-chunk weight slab (TMA, slab-major copy of W^T), its 8 warps split
// the K range (chunk c -> warp c % 8, private 3-stage ring per warp, each warp refills its own ring), partial sums are
// reduced through shared memory, and the finished 16 x 128 output block is written into the activation tile of ALL 8
// CTAs through distributed shared memory (st.shared::cluster) between two cluster barriers.  Same layer program, same
// folded-BN epilogue, same dropout masks, same decode as forward.cu.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "fwd_family.cuh"

namespace mlb {

constexpr int CL = 8;        // CTAs per cluster
constexpr int SR = 16;       // detections per cluster tile (act row stride)
constexpr int SC = 128;      // output columns per CTA
constexpr int SNST = 3;      // per-warp ring depth
constexpr int SCHUNK = KC * SC;  // floats per chunk (4 KB)

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_id_x() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t n_clusters_x() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t map_to_cta(uint32_t smem_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_cluster_v4(uint32_t addr, float4 v) {
    asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// per-warp weight stream: chunk c of a GEMM op belongs to warp c % 8; the sequence repeats for every tile of the cluster
struct WStream {
    int tile, op, c;
};
__device__ __forceinline__ bool wstream_next(const FwdParams& p, WStream& ws, int warp, int tile_stride, int rank,
                                             const float* slab, const long long* slab_off, const float*& src) {
    while (ws.tile < p.n_tiles) {
        const mlb_op& op = p.ops[ws.op];
        if (op.type == MLB_OP_GEMM && ws.c < op.Kpad / KC) {
            src = slab + slab_off[ws.op] + ((size_t)rank * op.Kpad + (size_t)ws.c * KC) * SC;
            ws.c += 8;
            return true;
        }
        ws.op++;
        ws.c = warp;
        if (ws.op == p.n_ops) ws.op = 0, ws.tile += tile_stride;
    }
    return false;
}

struct SmallExtra {
    const float* slab;                 // slab-major W^T copies: per GEMM op [8][Kpad][128]
    long long slab_off[MLB_MAX_OPS];   // float offset of each op's slab block
};

__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(256, 1)
    loco_forward_cluster_kernel(const __grid_constant__ FwdParams p, const __grid_constant__ SmallExtra ex) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int rank = (int)cluster_ctarank();
    const int g = lane >> 4, c16 = lane & 15;
    const int L = p.L;  // 1024

    float* act = reinterpret_cast<float*>(smem_raw);      // [L][SR]   k-major activation tile (every CTA holds all of it)
    float* red = act + (size_t)L * SR;                     // [8][SR][SC] per-warp partial sums
    float* rings = red + 8 * SR * SC;                      // [8][SNST][KC][SC]
    float* outs = rings + 8 * SNST * SCHUNK;               // [SR][OUT_LD]
    float* cen = outs + SR * OUT_LD;                       // [SR][4]
    uint64_t* full = reinterpret_cast<uint64_t*>(cen + SR * 4);  // [8][SNST]

    for (int i = tid; i < L * SR; i += 256) act[i] = 0.f;
    if (tid == 0) {
        for (int s = 0; s < 8 * SNST; ++s) mbar_init(&full[s], 1);
        mbar_fence_init();
    }
    __syncthreads();
    cluster_arrive();
    cluster_wait();  // every CTA's barriers / act are initialised before any remote store can land

    const int n_clusters = (int)n_clusters_x();
    float* my_ring = rings + (size_t)warp * SNST * SCHUNK;
    uint64_t* my_full = full + warp * SNST;
    WStream ws = {(int)cluster_id_x(), 0, warp};
    unsigned cons = 0;  // chunks consumed by this warp
    // prologue: fill the ring
    if (lane == 0) {
        for (int s = 0; s < SNST; ++s) {
            const float* src;
            if (!wstream_next(p, ws, warp, n_clusters, rank, ex.slab, ex.slab_off, src)) break;
            mbar_expect_tx(&my_full[s], SCHUNK * sizeof(float));
            tma_bulk_g2s(my_ring + (size_t)s * SCHUNK, src, SCHUNK * sizeof(float), &my_full[s]);
        }
    }

    const float zm = p.z_met;
    const float k0 = p.kinv[0], k1 = p.kinv[1], k2 = p.kinv[2], k3 = p.kinv[3], k4 = p.kinv[4], k5 = p.kinv[5];
    const uint32_t act_s = smem_u32(act);
    // reduce/epilogue mapping: this thread owns column `ecol` of the slab and 8 rows
    const int ecol = tid & 127, ehalf = tid >> 7;
    const int gcol = rank * SC + ecol;

    for (int tile = (int)cluster_id_x(); tile < p.n_tiles; tile += n_clusters) {
        const int row0 = tile * SR;
        const int rows_here = min(SR, p.n_rows - row0);

        // ------------------------------------------------------------ pre-process -> act[k][row] (every CTA, redundantly)
        if (p.input_kind == MLB_IN_X) {
            for (int idx = tid; idx < SR * p.kpad0; idx += 256) {
                const int r = idx / p.kpad0, k = idx % p.kpad0;
                float v = 0.f;
                if (r < rows_here && k < p.in_size) v = __ldg(p.x + (size_t)(row0 + r) * p.in_size + k);
                act[k * SR + r] = v;
            }
        } else {
            const bool stereo = p.input_kind == MLB_IN_KPS_STEREO;
            if (tid < SR) {
                const int r = tid;
                float uc = 0.f, vc = 0.f;
                if (r < rows_here) {
                    const float* kp = p.x + (size_t)(stereo ? (row0 + r) / p.n_right : (row0 + r)) * 51;
                    float umin = __ldg(kp), umax = umin, vmin = __ldg(kp + 17), vmax = vmin;
                    for (int j = 1; j < 17; ++j) {
                        const float u = __ldg(kp + j), v = __ldg(kp + 17 + j);
                        umin = fminf(umin, u), umax = fmaxf(umax, u);
                        vmin = fminf(vmin, v), vmax = fmaxf(vmax, v);
                    }
                    uc = __fadd_rn(__fdiv_rn(__fsub_rn(umax, umin), 2.f), umin);
                    vc = __fadd_rn(__fdiv_rn(__fsub_rn(vmax, vmin), 2.f), vmin);
                }
                cen[r * 4 + 0] = uc;
                cen[r * 4 + 1] = vc;
                cen[r * 4 + 2] = (uc * k0 + vc * k1 + k2) * zm;
                cen[r * 4 + 3] = (uc * k3 + vc * k4 + k5) * zm;
            }
            if (p.flags & MLB_FWD_ZERO_CENTER) __syncthreads();
            for (int idx = tid; idx < SR * 17; idx += 256) {
                const int r = idx / 17, j = idx % 17;
                float xl = 0.f, yl = 0.f, xd = 0.f, yd = 0.f;
                if (r < rows_here) {
                    const int grow = row0 + r;
                    const float* kp = p.x + (size_t)(stereo ? grow / p.n_right : grow) * 51;
                    const float u = __ldg(kp + j), v = __ldg(kp + 17 + j);
                    xl = (u * k0 + v * k1 + k2) * zm;
                    yl = (u * k3 + v * k4 + k5) * zm;
                    if (stereo) {
                        const float* kr = p.xr + (size_t)(grow % p.n_right) * 51;
                        const float ur = __ldg(kr + j), vr = __ldg(kr + 17 + j);
                        xd = xl - (ur * k0 + vr * k1 + k2) * zm;
                        yd = yl - (ur * k3 + vr * k4 + k5) * zm;
                    } else if (p.flags & MLB_FWD_ZERO_CENTER) {
                        xl -= cen[r * 4 + 2];
                        yl -= cen[r * 4 + 3];
                    }
                }
                act[(2 * j) * SR + r] = xl;
                act[(2 * j + 1) * SR + r] = yl;
                if (stereo) {
                    act[(34 + 2 * j) * SR + r] = xd;
                    act[(35 + 2 * j) * SR + r] = yd;
                }
            }
            for (int idx = tid; idx < SR * (p.kpad0 - p.in_size); idx += 256)  // zero the K padding rows
                act[(p.in_size + idx / SR) * SR + idx % SR] = 0.f;
        }
        __syncthreads();
        if (rank == 0 && p.out_x != nullptr && p.input_kind != MLB_IN_X) {
            for (int idx = tid; idx < rows_here * p.in_size; idx += 256) {
                const int r = idx / p.in_size, k = idx % p.in_size;
                p.out_x[(size_t)(row0 + r) * p.in_size + k] = act[k * SR + r];
            }
        }

        // ------------------------------------------------------------ layer program
        float res[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        int site = 0;
        for (int oi = 0; oi < p.n_ops; ++oi) {
            const mlb_op& op = p.ops[oi];
            if (op.type == MLB_OP_GEMM) {
                const int nchunks = op.Kpad / KC;
                unsigned long long acc2[4][8];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc2[i][j] = 0ull;
                for (int ch = warp; ch < nchunks; ch += 8, ++cons) {
                    const unsigned stage = cons % SNST;
                    mbar_wait(&my_full[stage], (cons / SNST) & 1, p.err_flag);
                    const float* b_ptr = my_ring + (size_t)stage * SCHUNK + c16 * 4;
                    const float* a_ptr = act + (size_t)ch * KC * SR + g * 8;
#pragma unroll
                    for (int kk = 0; kk < KC; ++kk) {
                        const ulonglong2 t0 = *reinterpret_cast<const ulonglong2*>(a_ptr + kk * SR);
                        const ulonglong2 t1 = *reinterpret_cast<const ulonglong2*>(a_ptr + kk * SR + 4);
                        const unsigned long long a2[4] = {t0.x, t0.y, t1.x, t1.y};
                        const float4 b0 = *reinterpret_cast<const float4*>(b_ptr + kk * SC);
                        const float4 b1 = *reinterpret_cast<const float4*>(b_ptr + kk * SC + 64);
                        const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const unsigned long long bd = pack2(b[j], b[j]);
#pragma unroll
                            for (int i = 0; i < 4; ++i) acc2[i][j] = ffma2(a2[i], bd, acc2[i][j]);
                        }
                    }
                    __syncwarp();
                    if (lane == 0) {  // refill this stage with the warp's chunk SNST ahead (may belong to a later op / tile)
                        const float* src;
                        if (wstream_next(p, ws, warp, n_clusters, rank, ex.slab, ex.slab_off, src)) {
                            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                            mbar_expect_tx(&my_full[stage], SCHUNK * sizeof(float));
                            tma_bulk_g2s(my_ring + (size_t)stage * SCHUNK, src, SCHUNK * sizeof(float), &my_full[stage]);
                        }
                    }
                }
                // ---- partial sums -> red[warp][row][col]
                {
                    float* rw = red + (size_t)warp * SR * SC + c16 * 4;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        float lo[8], hi[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) unpack2(acc2[i][j], lo[j], hi[j]);
                        float* r0 = rw + (size_t)(g * 8 + 2 * i) * SC;
                        *reinterpret_cast<float4*>(r0) = make_float4(lo[0], lo[1], lo[2], lo[3]);
                        *reinterpret_cast<float4*>(r0 + 64) = make_float4(lo[4], lo[5], lo[6], lo[7]);
                        *reinterpret_cast<float4*>(r0 + SC) = make_float4(hi[0], hi[1], hi[2], hi[3]);
                        *reinterpret_cast<float4*>(r0 + SC + 64) = make_float4(hi[4], hi[5], hi[6], hi[7]);
                    }
                }
                __syncthreads();
                cluster_arrive();  // this CTA no longer reads `act` as the layer input
                // ---- reduce the 8 partials, folded-BN epilogue for (8 rows, column gcol)
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    float s = 0.f;
#pragma unroll
                    for (int w = 0; w < 8; ++w) s += red[(size_t)w * SR * SC + (size_t)(ehalf * 8 + i) * SC + ecol];
                    v[i] = s;
                }
                {
                    const float sc = __ldg(p.blob + op.scale_off + gcol), sh = __ldg(p.blob + op.shift_off + gcol);
                    const bool relu = (op.flags & MLB_F_RELU) != 0;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float y = fmaf(v[i], sc, sh);
                        v[i] = relu ? fmaxf(y, 0.f) : y;
                    }
                }
                if (op.flags & MLB_F_DROPOUT) {
                    if (p.flags & MLB_FWD_DROPOUT) {
                        const float inv_keep = 1.0f / (1.0f - p.p_drop);
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const int grow = row0 + ehalf * 8 + i;
                            bool keep;
                            if (p.drop_mask != nullptr)
                                keep = grow < p.n_rows ? p.drop_mask[((size_t)site * p.n_rows + grow) * L + gcol] != 0 : true;
                            else
                                keep = keep_draw(p.drop_seed, site, grow, gcol, p.p_drop);
                            v[i] = keep ? v[i] * inv_keep : 0.f;
                        }
                    }
                    site++;
                }
                if (op.flags & MLB_F_ADD_RES) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] += res[i];
                }
                if (op.flags & MLB_F_SAVE_RES) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) res[i] = v[i];
                }
                cluster_wait();  // every CTA of the cluster has finished reading its `act`
                // ---- all-gather through distributed shared memory: my 16 x 128 block into every CTA's tile
                {
                    const uint32_t local = act_s + (uint32_t)(((size_t)gcol * SR + ehalf * 8) * sizeof(float));
                    const float4 lo = make_float4(v[0], v[1], v[2], v[3]), hi = make_float4(v[4], v[5], v[6], v[7]);
#pragma unroll
                    for (int r = 0; r < CL; ++r) {
                        const uint32_t ra = map_to_cta(local, (uint32_t)((rank + r) & (CL - 1)));
                        st_cluster_v4(ra, lo);
                        st_cluster_v4(ra + 16, hi);
                    }
                }
                cluster_arrive();
                cluster_wait();  // all 8 blocks have landed everywhere
            } else if (rank == 0) {
                // ---- narrow head on the leader CTA: one warp per output column, lanes = 16 rows x 2 K-halves
                for (int o = 7 - warp; o < op.N; o += 8) {
                    const float* w = p.blob + op.w_off + (size_t)o * op.K;
                    const int row = lane & 15, kh = lane >> 4, kbeg = kh * (op.K / 2);
                    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 8
                    for (int k = kbeg; k < kbeg + op.K / 2; k += 4) {
                        const float4 wv = __ldg(reinterpret_cast<const float4*>(w + k));
                        a0 = fmaf(act[(k + 0) * SR + row], wv.x, a0);
                        a1 = fmaf(act[(k + 1) * SR + row], wv.y, a1);
                        a2 = fmaf(act[(k + 2) * SR + row], wv.z, a2);
                        a3 = fmaf(act[(k + 3) * SR + row], wv.w, a3);
                    }
                    float s = (a0 + a1) + (a2 + a3);
                    s += __shfl_xor_sync(0xffffffffu, s, 16);
                    if (kh == 0) outs[row * OUT_LD + op.out_col + o] = s + __ldg(p.blob + op.shift_off + o);
                }
            }
        }

        // ------------------------------------------------------------ decode + store (leader CTA, one thread per row)
        if (rank == 0) {
            __syncthreads();
            if (tid < rows_here) {
                store_row(p, (size_t)row0 + tid, outs + tid * OUT_LD, cen + tid * 4);
            }
            __syncthreads();
        }
    }
    if (rank == 0 && tid == 0) gather_finish(p);  // fused all-gather: one arrival per cluster leader
    cluster_arrive();
    cluster_wait();  // no CTA exits while a peer may still address its shared memory
}

// W^T [Kpad][L] -> slab-major [8][Kpad][128] (one contiguous 4 KB TMA chunk per (slab, 8 k-rows))
__global__ void slab_pack_kernel(const float* __restrict__ wt, float* __restrict__ slab, int kpad, int L) {
    const size_t n = (size_t)kpad * L;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int k = (int)(i / L), col = (int)(i % L);
        slab[((size_t)(col / SC) * kpad + k) * SC + col % SC] = wt[i];
    }
}

}  // namespace mlb

using namespace mlb;

static size_t small_smem_bytes(int L) {
    const size_t fl = (size_t)L * SR + 8 * SR * SC + 8 * SNST * SCHUNK + SR * OUT_LD + SR * 4;
    return fl * sizeof(float) + 8 * SNST * sizeof(uint64_t) + 16;
}

cudaError_t ClusterFamily::repack(const float* blob, const mlb_op* ops, int n_ops, int L, cudaStream_t st) const {
    if (!available) return cudaSuccess;
    for (int i = 0; i < n_ops; ++i)
        if (ops[i].type == MLB_OP_GEMM) slab_pack_kernel<<<256, 256, 0, st>>>(blob + ops[i].w_off, slab + slab_off[i], ops[i].Kpad, L);
    return cudaGetLastError();
}

// how many 8-CTA clusters of this kernel can be resident at once (GPC packing decides: measured 11-16 on a B200)
static int small_max_clusters(int L) {
    const size_t smem = small_smem_bytes(L);
    if (cudaFuncSetAttribute(loco_forward_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return 0;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(CL * 64);
    cfg.blockDim = dim3(256);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at;
    at.id = cudaLaunchAttributeClusterDimension;
    at.val.clusterDim.x = CL, at.val.clusterDim.y = 1, at.val.clusterDim.z = 1;
    cfg.attrs = &at;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, loco_forward_cluster_kernel, &cfg) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

cudaError_t ClusterFamily::setup(const float* blob, const mlb_op* ops, int n_ops, int L) {
    if (L != 1024) return cudaSuccess;
    long long off = 0;
    for (int i = 0; i < n_ops; ++i) {
        slab_off[i] = off;
        if (ops[i].type == MLB_OP_GEMM) off += (long long)ops[i].Kpad * L;
    }
    cudaError_t e = cudaMalloc(&slab, (size_t)off * sizeof(float));
    if (e != cudaSuccess) return e;
    available = true;
    if ((e = repack(blob, ops, n_ops, L, 0)) != cudaSuccess) return e;
    conc = small_max_clusters(L);
    if (conc < 1) conc = 8;
    return cudaSuccess;
}

void ClusterFamily::release() {
    cudaFree(slab);
    slab = nullptr;
    available = false;
}

cudaError_t ClusterFamily::launch(FwdParams p, const FwdPlan& pl, cudaStream_t st, int* issued) const {
    SmallExtra ex;
    ex.slab = slab;
    memcpy(ex.slab_off, slab_off, sizeof(ex.slab_off));
    p.n_tiles = (p.n_rows + 15) / 16;
    const size_t smem = small_smem_bytes(p.L);
    cudaError_t e = cudaFuncSetAttribute(loco_forward_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    loco_forward_cluster_kernel<<<pl.clusters * CL, 256, smem, st>>>(p, ex);
    if ((e = cudaGetLastError()) == cudaSuccess) ++*issued;
    return e;
}
