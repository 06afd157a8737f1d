// Fused monoloco inference forward for B200 (sm_100a):  pre-process -> stacked Linear+BN+ReLU(+Dropout)
// residual stages -> heads -> Laplace / spherical / orientation decode, one persistent CTA per SM.
//
// Replaces, in one launch per detection batch (reference file:line):
//   monoloco/network/process.py:47-67   preprocess_monoloco   (+ utils/camera.py:10-29, 82-86)
//   monoloco/network/process.py:25-44   preprocess_monstereo  (all-vs-all rows built on the fly)
//   monoloco/network/architectures.py:48-71 / 88-102 / 135-145 / 162-176   LocoModel / MonolocoModel forward
//   monoloco/network/process.py:231-278, 330-360, 125-133   extract_outputs(_mono), unnormalize_bi
//   monoloco/utils/camera.py:161-177, 202-208, 226-237      xyz_from_distance, back_correct_angles, to_cartesian
//
// Data layout (see DESIGN.md §3):
//   * a CTA owns a tile of 4*TM detections for the whole network; the [L, 32] activation tile lives in shared
//     memory k-major (act[k*32 + row]) so a warp's A fragment is a broadcast LDS.128 and the next layer's K
//     index is this layer's N index;
//   * weights are pre-packed per layer as chunks [KC][L] of W^T; one elected thread streams them L2 -> smem
//     with 1-D TMA bulk copies (cp.async.bulk ... mbarrier::complete_tx) through a NSTAGE ring guarded by
//     full/empty mbarriers; the stream runs ahead across layer and tile boundaries;
//   * 8 consumer warps (+1 producer warp) register-tile the [2*TM, L] x [L, L] product: a warp owns 128 output
//     columns, lanes = 2 row groups x 16 column groups, each thread holds TM x 8 fp32 accumulators (TM <= 16);
//     per k-step TM/4 broadcast LDS.128 (A) + 2 conflict-free LDS.128 (B) feed 8*TM FFMA -- the tall thread tile
//     keeps the shared-memory pipe (128 B/clk/SM, the binding limit of an 8x8 tile) at ~55 % of the FFMA time;
//   * the residual `x` of MyLinearSimple is stashed per thread in an L2-resident scratch (or Tensor Memory).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "fwd_family.cuh"

namespace mlb {

// stand-alone decode of a raw [B, out] tensor (extract_outputs on outputs that did not come from the fused kernel)
__global__ void decode_kernel(const float* __restrict__ raw, int n_rows, int out_size, int kind, float* __restrict__ dec) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    float o[OUT_LD];
    for (int k = 0; k < out_size; ++k) o[k] = raw[(size_t)row * out_size + k];
    float x, y, z, d, bi, yaw_p, yaw_o, aux;
    decode_row(kind, out_size, o, x, y, z, d, bi, yaw_p, yaw_o, aux);
    float4* dst = reinterpret_cast<float4*>(dec + (size_t)row * 8);
    dst[0] = make_float4(x, y, z, d);
    dst[1] = make_float4(bi, yaw_p, yaw_o, aux);
}

// local row r of a tile -> shared-memory row (2 groups of 16 slots, TM used per group)
__device__ __forceinline__ int smem_row(int r, int tm) { return (r / tm) * 16 + (r % tm); }

__device__ __forceinline__ void consumer_sync(int n_consumer_threads) {
    asm volatile("bar.sync 1, %0;" ::"r"(n_consumer_threads) : "memory");
}

// The weight stream: every GEMM chunk of every tile this CTA owns, in consumption order.
__device__ __forceinline__ void producer_loop(const FwdParams& p, float* ring, uint64_t* full, uint64_t* empty, int L) {
    unsigned q = 0, stage = 0, parity = 0;  // parity of the fill this iteration performs on `stage`
    const uint32_t bytes = (uint32_t)(KC * L * sizeof(float));
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        for (int oi = 0; oi < p.n_ops; ++oi) {
            const mlb_op& op = p.ops[oi];
            if (op.type != MLB_OP_GEMM) continue;
            const float* src = p.blob + op.w_off;
            const int nchunks = op.Kpad / KC;
            for (int ch = 0; ch < nchunks; ++ch, ++q) {
                if (q >= NSTAGE) mbar_wait_backoff(&empty[stage], parity ^ 1, p.err_flag);  // consumers released fill #(q/NSTAGE - 1)
                mbar_expect_tx(&full[stage], bytes);
                tma_bulk_g2s(ring + (size_t)stage * KC * L, src + (size_t)ch * KC * L, bytes, &full[stage]);
                if (++stage == NSTAGE) stage = 0, parity ^= 1;
            }
        }
    }
}

// profiling aid (mlb_debug_fwd_marks): when set, thread 0 of CTA 0 stamps globaltimer at points of the layer program
__device__ unsigned long long* g_fwd_marks = nullptr;
__device__ __forceinline__ void fmark(unsigned long long* marks, int slot) {
    if (marks != nullptr) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        marks[slot] = t;
    }
}

template <int TM>
__global__ void __launch_bounds__(MAX_THREADS, 1) loco_forward_kernel(const __grid_constant__ FwdParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int L = p.L;
    const int nwarps = L >> 7;          // active consumer warps: one per 128 hidden columns
    const int nthreads = nwarps << 5;   // active consumer threads
    const int prod_warp = (int)(blockDim.x >> 5) - 4;  // first warp of the producer warpgroup
    const int g = lane >> 4, c = lane & 15;
    constexpr int ROWS = 2 * TM;
    constexpr int A4 = (TM + 3) / 4;  // LDS.128 per k-step for the A fragment
    constexpr int RES_STRIDE = 256;   // residual scratch: [cta][TM*8][256 consumer threads], thread-private

    float* act = reinterpret_cast<float*>(smem_raw);  // [L][MP]
    float* xin = act;                                  // network input tile [kpad0][MP]: dead once w1's epilogue writes act
    float* outs = act + (size_t)L * MP;                // [MP][OUT_LD]
    float* cen = outs + MP * OUT_LD;                   // [MP][4]  (u_c, v_c, cx*z_met, cy*z_met)
    float* ring = cen + MP * 4;                        // [NSTAGE][KC][L]
    uint64_t* full = reinterpret_cast<uint64_t*>(ring + (size_t)NSTAGE * KC * L);
    uint64_t* empty = full + NSTAGE;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(empty + NSTAGE);

    const bool res_tmem = (p.flags & MLB_FWD_RES_TMEM) != 0;
    const uint32_t tmem_cols = nwarps <= 1 ? 128u : (nwarps <= 4 ? 128u : 256u);

    for (int i = tid; i < L * MP + MP * OUT_LD + MP * 4; i += blockDim.x) act[i] = 0.f;
    if (tid == 0) {
        for (int s = 0; s < NSTAGE; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], nwarps);
        }
        mbar_fence_init();
    }
    if (res_tmem) {
        if (warp == 0) tmem_alloc(tmem_slot, tmem_cols);
        tmem_fence_before();
    }
    __syncthreads();
    if (res_tmem) tmem_fence_after();

    if (warp >= prod_warp) {
        // ================================================================ producer warpgroup (1 elected thread works)
        asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");
        if (warp == prod_warp && lane == 0) producer_loop(p, ring, full, empty, L);
    } else {
        // ================================================================ consumer warpgroups
        asm volatile("setmaxnreg.inc.sync.aligned.u32 240;");
        if (warp < nwarps) {
        uint32_t tmem_base = 0;
        if (res_tmem) tmem_base = *tmem_slot + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)((warp >> 2) * 128);
        unsigned q = 0;  // chunks consumed so far (identical in every consumer warp)
        unsigned stage = 0, parity = 0;
        unsigned total_chunks = 0;
        for (int oi = 0; oi < p.n_ops; ++oi)
            if (p.ops[oi].type == MLB_OP_GEMM) total_chunks += p.ops[oi].Kpad / KC;
        total_chunks *= (unsigned)((p.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x);
        mbar_wait(&full[0], 0, p.err_flag);  // chunk 0
        const float zm = p.z_met;
        const float k0 = p.kinv[0], k1 = p.kinv[1], k2 = p.kinv[2], k3 = p.kinv[3], k4 = p.kinv[4], k5 = p.kinv[5];
        // this thread's 8 output columns: n0 + {0..3} and n0 + 64 + {0..3}
        const int n0 = warp * 128 + c * 4;
        unsigned long long* marks = (tid == 0 && blockIdx.x == 0) ? g_fwd_marks : nullptr;
        fmark(marks, 0);

        for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
            const int row0 = tile * ROWS;
            const int rows_here = min(ROWS, p.n_rows - row0);

            // ---------------------------------------------------------------- pre-process -> xin[k][row]
            if (p.input_kind == MLB_IN_X) {
                // nn.Module.forward input [B, in]; transpose into the k-major tile, zero-fill padding
                for (int idx = tid; idx < ROWS * p.kpad0; idx += nthreads) {
                    const int r = idx / p.kpad0, k = idx % p.kpad0;
                    float v = 0.f;
                    if (r < rows_here && k < p.in_size) v = __ldg(p.x + (size_t)(row0 + r) * p.in_size + k);
                    xin[k * MP + smem_row(r, TM)] = v;
                }
            } else {
                const bool stereo = p.input_kind == MLB_IN_KPS_STEREO;
                // bbox centre of the (left) pose's 17 keypoints (camera.py:82-86): zero-centering + xyz_from_distance ray
                if (tid < ROWS) {
                    const int r = tid, sr = smem_row(r, TM);
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
                    cen[sr * 4 + 0] = uc;
                    cen[sr * 4 + 1] = vc;
                    cen[sr * 4 + 2] = (uc * k0 + vc * k1 + k2) * zm;
                    cen[sr * 4 + 3] = (uc * k3 + vc * k4 + k5) * zm;
                }
                if (p.flags & MLB_FWD_ZERO_CENTER) consumer_sync(nthreads);
                for (int idx = tid; idx < ROWS * 17; idx += nthreads) {
                    const int r = idx / 17, j = idx % 17, sr = smem_row(r, TM);
                    float xl = 0.f, yl = 0.f, xd = 0.f, yd = 0.f;
                    if (r < rows_here) {
                        const int grow = row0 + r;
                        const int li = stereo ? grow / p.n_right : grow;
                        const float* kp = p.x + (size_t)li * 51;
                        const float u = __ldg(kp + j), v = __ldg(kp + 17 + j);
                        xl = (u * k0 + v * k1 + k2) * zm;  // camera.py:26-27, rows 0/1 of [u v 1] K^-T
                        yl = (u * k3 + v * k4 + k5) * zm;
                        if (stereo) {
                            const float* kr = p.xr + (size_t)(grow % p.n_right) * 51;
                            const float ur = __ldg(kr + j), vr = __ldg(kr + 17 + j);
                            xd = xl - (ur * k0 + vr * k1 + k2) * zm;  // process.py:41 cat(l, l - r)
                            yd = yl - (ur * k3 + vr * k4 + k5) * zm;
                        } else if (p.flags & MLB_FWD_ZERO_CENTER) {
                            xl -= cen[sr * 4 + 2];  // process.py:61-62
                            yl -= cen[sr * 4 + 3];
                        }
                    }
                    xin[(2 * j) * MP + sr] = xl;
                    xin[(2 * j + 1) * MP + sr] = yl;
                    if (stereo) {
                        xin[(34 + 2 * j) * MP + sr] = xd;
                        xin[(35 + 2 * j) * MP + sr] = yd;
                    }
                }
            }
            consumer_sync(nthreads);
            if (p.out_x != nullptr && p.input_kind != MLB_IN_X) {
                for (int idx = tid; idx < rows_here * p.in_size; idx += nthreads) {
                    const int r = idx / p.in_size, k = idx % p.in_size;
                    p.out_x[(size_t)(row0 + r) * p.in_size + k] = xin[k * MP + smem_row(r, TM)];
                }
            }

            fmark(marks, 1);
            // ---------------------------------------------------------------- layer program
            int site = 0;
            for (int oi = 0; oi < p.n_ops; ++oi) {
                const mlb_op& op = p.ops[oi];
                if (op.type == MLB_OP_GEMM) {
                    const float* in = (op.flags & MLB_F_IN_XIN) ? xin : act;
                    const int nchunks = op.Kpad / KC;
                    // accumulators as packed f32x2 pairs over two consecutive rows (lo = row 2*ip, hi = row 2*ip + 1):
                    // fma.rn.f32x2 (SASS FFMA2) does both rows in one issue slot, so 2 warps/SMSP keep the FMA pipe fed
                    unsigned long long acc2[TM / 2][8];
#pragma unroll
                    for (int i = 0; i < TM / 2; ++i)
#pragma unroll
                        for (int j = 0; j < 8; ++j) acc2[i][j] = 0ull;

                    const float* a_ptr = in + g * 16;
                    // two / four 8-k-step chunks per loop trip: halves the loop-carried register shuffling (measured:
                    // 1.357 -> 1.264 -> 1.245 ms at B=4096; the 128-accumulator TM=16 tile spills beyond 2)
#pragma unroll(TM <= 14 ? 4 : 2)
                    for (int ch = 0; ch < nchunks; ++ch, ++q) {
                        // invariant: chunk q has landed (waited for at the end of the previous iteration).
                        // Probe the NEXT stage now, non-blocking, so the mbarrier round trip hides under this chunk's FFMAs.
                        unsigned nstage = stage + 1, nparity = parity;
                        if (nstage == NSTAGE) nstage = 0, nparity ^= 1;
                        const bool has_next = q + 1 < total_chunks;
                        const bool next_ready = has_next ? mbar_test_wait(&full[nstage], nparity) : true;
                        const float* b_ptr = ring + (size_t)stage * KC * L + n0;
#pragma unroll
                        for (int kk = 0; kk < KC; ++kk) {
                            unsigned long long a2[(TM + 1) / 2];
                            const float* ap = a_ptr + (ch * KC + kk) * MP;
#pragma unroll
                            for (int v = 0; v < TM / 4; ++v) {
                                const ulonglong2 t = *reinterpret_cast<const ulonglong2*>(ap + v * 4);
                                a2[v * 2 + 0] = t.x, a2[v * 2 + 1] = t.y;
                            }
                            if (TM % 4) a2[(TM / 4) * 2] = *reinterpret_cast<const unsigned long long*>(ap + (TM / 4) * 4);
                            const float4 b0 = *reinterpret_cast<const float4*>(b_ptr + kk * L);
                            const float4 b1 = *reinterpret_cast<const float4*>(b_ptr + kk * L + 64);
                            const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const unsigned long long bd = pack2(b[j], b[j]);
#pragma unroll
                                for (int i = 0; i < TM / 2; ++i) acc2[i][j] = ffma2(a2[i], bd, acc2[i][j]);
                            }
                        }
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&empty[stage]);
                        if (!next_ready) mbar_wait(&full[nstage], nparity, p.err_flag);
                        stage = nstage, parity = nparity;
                    }
                    fmark(marks, 2 + 4 * oi);
                    float acc[TM][8];
#pragma unroll
                    for (int i = 0; i < TM / 2; ++i)
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            unpack2(acc2[i][j], acc[2 * i][j], acc[2 * i + 1][j]);
                        }

                    // ---- epilogue: folded BatchNorm affine, ReLU, dropout, residual
                    {
                        const float4 s0 = __ldg(reinterpret_cast<const float4*>(p.blob + op.scale_off + n0));
                        const float4 s1 = __ldg(reinterpret_cast<const float4*>(p.blob + op.scale_off + n0 + 64));
                        const float4 t0 = __ldg(reinterpret_cast<const float4*>(p.blob + op.shift_off + n0));
                        const float4 t1 = __ldg(reinterpret_cast<const float4*>(p.blob + op.shift_off + n0 + 64));
                        const float sc[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
                        const float sh[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
                        const bool relu = (op.flags & MLB_F_RELU) != 0;
#pragma unroll
                        for (int i = 0; i < TM; ++i)
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                float v = fmaf(acc[i][j], sc[j], sh[j]);
                                acc[i][j] = relu ? fmaxf(v, 0.f) : v;
                            }
                    }
                    if (op.flags & MLB_F_DROPOUT) {
                        if (p.flags & MLB_FWD_DROPOUT) {
                            // one mask-vs-hash branch per row; per-launch / per-column parts of the hash hoisted (common.cuh)
                            const float inv_keep = 1.0f / (1.0f - p.p_drop);
                            const uint32_t seed_mix = drop_seed_mix(p.drop_seed), thr = drop_threshold(p.p_drop);
                            uint32_t ch[8];
#pragma unroll
                            for (int j = 0; j < 8; ++j) ch[j] = drop_col_hash((uint32_t)(n0 + (j & 3) + (j >> 2) * 64), (uint32_t)site);
#pragma unroll
                            for (int i = 0; i < TM; ++i) {
                                const int grow = row0 + g * TM + i;
                                uint32_t kb = 0xFFu;
                                if (p.drop_mask != nullptr) {
                                    if (grow < p.n_rows) {
                                        const uint8_t* m = p.drop_mask + ((size_t)site * p.n_rows + grow) * L + n0;
                                        kb = bytes_to_bits(*reinterpret_cast<const uint32_t*>(m)) |
                                             (bytes_to_bits(*reinterpret_cast<const uint32_t*>(m + 64)) << 4);
                                    }
                                } else {
                                    const uint32_t rm = drop_row_mix(seed_mix, (uint32_t)grow);
                                    kb = 0;
#pragma unroll
                                    for (int j = 0; j < 8; ++j) kb |= (drop_keep(rm, ch[j], thr) ? 1u : 0u) << j;
                                }
#pragma unroll
                                for (int j = 0; j < 8; ++j) acc[i][j] = (kb >> j) & 1u ? acc[i][j] * inv_keep : 0.f;
                            }
                        }
                        site++;
                    }
                    if (op.flags & MLB_F_ADD_RES) {
                        if (res_tmem) {
#pragma unroll
                            for (int i = 0; i < TM; ++i) {
                                float r[8];
                                tmem_ld8(tmem_base + i * 8, r);
#pragma unroll
                                for (int j = 0; j < 8; ++j) acc[i][j] += r[j];
                            }
                        } else {
                            const float* rs = p.res_scratch + (size_t)blockIdx.x * (128 * RES_STRIDE) + tid;
#pragma unroll
                            for (int i = 0; i < TM; ++i)
#pragma unroll
                                for (int j = 0; j < 8; ++j) acc[i][j] += rs[(i * 8 + j) * RES_STRIDE];
                        }
                    }
                    if (op.flags & MLB_F_SAVE_RES) {
                        if (res_tmem) {
#pragma unroll
                            for (int i = 0; i < TM; ++i) tmem_st8(tmem_base + i * 8, acc[i]);
                            tmem_st_wait();
                        } else {
                            float* rs = p.res_scratch + (size_t)blockIdx.x * (128 * RES_STRIDE) + tid;
#pragma unroll
                            for (int i = 0; i < TM; ++i)
#pragma unroll
                                for (int j = 0; j < 8; ++j) rs[(i * 8 + j) * RES_STRIDE] = acc[i][j];
                        }
                    }
                    fmark(marks, 3 + 4 * oi);
                    consumer_sync(nthreads);  // every warp has finished reading `act` as this layer's input
                    fmark(marks, 4 + 4 * oi);
                    // k-major write of the new activation tile.  Lane c of a row group owns rows k = n0 + j (stride 512 B
                    // between neighbouring lanes -> the same banks), so the 16-byte row quads are written in a per-lane
                    // rotated order, quad (t + c) & 3 at step t: the 8 lanes of a quarter-warp then cover all 4 quads of
                    // their 64-byte half-row (2-way instead of 8-way bank conflicts; 4.1 -> ~1 us per layer at L = 1024).
                    // The rotation is a 2-level select network over the statically indexed accumulators.
                    {
                        const bool r1 = (c & 1) != 0, r2 = (c & 2) != 0;
                        auto quad = [&](int v, int j, int e) -> float {  // element e of row quad v (rows 4v..4v+3) of column j
                            return (v * 4 + e < TM) ? acc[(v * 4 + e < TM) ? v * 4 + e : 0][j] : 0.f;
                        };
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            float* dst = act + (size_t)(n0 + (j & 3) + (j >> 2) * 64) * MP + g * 16;
                            float lv1[4][4];  // [t][e] = r1 ? quad(t + 1) : quad(t)
#pragma unroll
                            for (int t = 0; t < 4; ++t)
#pragma unroll
                                for (int e = 0; e < 4; ++e) lv1[t][e] = r1 ? quad((t + 1) & 3, j, e) : quad(t, j, e);
#pragma unroll
                            for (int t = 0; t < 4; ++t) {
                                float4 o;
                                o.x = r2 ? lv1[(t + 2) & 3][0] : lv1[t][0];
                                o.y = r2 ? lv1[(t + 2) & 3][1] : lv1[t][1];
                                o.z = r2 ? lv1[(t + 2) & 3][2] : lv1[t][2];
                                o.w = r2 ? lv1[(t + 2) & 3][3] : lv1[t][3];
                                *reinterpret_cast<float4*>(dst + ((t + c) & 3) * 4) = o;
                            }
                        }
                    }
                    fmark(marks, 5 + 4 * oi);
                    consumer_sync(nthreads);
                } else {
                    // ---- narrow head: one warp per output column, lane = tile row slot
                    for (int o = nwarps - 1 - warp; o < op.N; o += nwarps)
                        outs[lane * OUT_LD + op.out_col + o] = head_column(p.blob + op.w_off + (size_t)o * op.K,
                                                                           __ldg(p.blob + op.shift_off + o), op.K, act, lane, lane, MP);
                    fmark(marks, 5 + 4 * oi);
                }
            }
            consumer_sync(nthreads);
            fmark(marks, 2 + 4 * p.n_ops);

            // ---------------------------------------------------------------- decode + store (one thread per row)
            if (tid < MP) {
                const int sr = tid, grp = sr >> 4, i = sr & 15;
                const int r = grp * TM + i;
                if (i < TM && r < rows_here) {
                    store_row(p, (size_t)row0 + r, outs + sr * OUT_LD, cen + sr * 4);
                }
            }
            consumer_sync(nthreads);
            fmark(marks, 3 + 4 * p.n_ops);
        }
        if (tid == 0) gather_finish(p);  // fused all-gather: last CTA publishes this rank's epoch and waits for the peers'
        }  // active consumer warp
    }

    if (res_tmem) tmem_fence_before();
    __syncthreads();
    if (res_tmem && warp == 0) tmem_dealloc(*tmem_slot, tmem_cols);
}

// ------------------------------------------------------------------------------------------------
// stand-alone pre-process (process.py:47-67) for callers that never run the network
// ------------------------------------------------------------------------------------------------
__global__ void preprocess_kernel(const float* __restrict__ kps, int n_rows, float k0, float k1, float k2, float k3,
                                  float k4, float k5, float zm, int zero_center, float* __restrict__ out_x) {
    const int row = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= n_rows) return;
    const float* kp = kps + (size_t)row * 51;
    float u = 0.f, v = 0.f;
    if (lane < 17) u = __ldg(kp + lane), v = __ldg(kp + 17 + lane);
    float cx = 0.f, cy = 0.f;
    if (zero_center) {
        float umin = lane < 17 ? u : INFINITY, umax = lane < 17 ? u : -INFINITY;
        float vmin = lane < 17 ? v : INFINITY, vmax = lane < 17 ? v : -INFINITY;
        for (int s = 16; s > 0; s >>= 1) {
            umin = fminf(umin, __shfl_xor_sync(0xffffffffu, umin, s));
            umax = fmaxf(umax, __shfl_xor_sync(0xffffffffu, umax, s));
            vmin = fminf(vmin, __shfl_xor_sync(0xffffffffu, vmin, s));
            vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, s));
        }
        const float uc = __fadd_rn(__fdiv_rn(__fsub_rn(umax, umin), 2.f), umin);
        const float vc = __fadd_rn(__fdiv_rn(__fsub_rn(vmax, vmin), 2.f), vmin);
        cx = (uc * k0 + vc * k1 + k2) * zm;
        cy = (uc * k3 + vc * k4 + k5) * zm;
    }
    if (lane < 17) {
        out_x[(size_t)row * 34 + 2 * lane] = (u * k0 + v * k1 + k2) * zm - cx;
        out_x[(size_t)row * 34 + 2 * lane + 1] = (u * k3 + v * k4 + k5) * zm - cy;
    }
}

// ------------------------------------------------------------------------------------------------
// MC-dropout epistemic spread (net.py:135-161 + process.py:101-122): for every detection, draw n_samples
// Laplace(mu_n, |b_n|) samples for each of the n_pass stochastic forwards and return the unbiased std over all
// n_pass * n_samples draws (torch: cat over passes -> .std(0)).  Inverse-CDF sampling with a counter RNG
// (the reference reseeds torch's generator per pass: not reproducible here, equal in distribution).
// ------------------------------------------------------------------------------------------------
__global__ void laplace_std_kernel(const float* __restrict__ d_bi, int n_pass, int n_rows, int n_samples,
                                   unsigned long long seed, float* __restrict__ out_std) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    double mean = 0.0, m2 = 0.0;
    long cnt = 0;
    for (int n = 0; n < n_pass; ++n) {
        const float mu = d_bi[((size_t)n * n_rows + row) * 2 + 0];
        const float b = fabsf(d_bi[((size_t)n * n_rows + row) * 2 + 1]);  // process.py:105
        for (int s = 0; s < n_samples; ++s) {
            const uint32_t r = mix32((((uint64_t)row << 32) | ((uint64_t)n << 16) | (uint64_t)s) ^ (seed * 0x9E3779B97F4A7C15ULL));
            // 23 random bits: (r >> 9) + 0.5 is exact in fp32, so u stays strictly inside (-0.5, 0.5); with 24 bits the top
            // value rounded up to u = 0.5 -> log1p(-1) = -inf -> NaN std once per 2^24 draws (found by the 200k-draw test)
            const float u = ((float)(r >> 9) + 0.5f) * (1.0f / 8388608.0f) - 0.5f;
            const float x = mu - b * copysignf(1.f, u) * log1pf(-2.f * fabsf(u));
            ++cnt;
            const double dlt = (double)x - mean;
            mean += dlt / (double)cnt;
            m2 += dlt * ((double)x - mean);
        }
    }
    out_std[row] = cnt > 1 ? (float)sqrt(m2 / (double)(cnt - 1)) : 0.f;
}

// ------------------------------------------------------------------------------------------------
// FP32 FFMA throughput probe: 16 independent chains per thread
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512) ffma_probe_kernel(int iters, float* sink) {
    float a[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = (float)(threadIdx.x + i) * 1e-3f;
    const float b = 1.0000001f, cc = 1e-7f * (float)blockIdx.x;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
#pragma unroll
            for (int i = 0; i < 16; ++i) a[i] = fmaf(a[i], b, cc);
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += a[i];
    if (s == 123.456f) sink[0] = s;
}

// packed variant: fma.rn.f32x2 (SASS FFMA2), 2 FMAs per lane per instruction
__global__ void __launch_bounds__(512) ffma2_probe_kernel(int iters, float* sink) {
    unsigned long long a[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float lo = (float)(threadIdx.x + i) * 1e-3f, hi = lo + 0.5f;
        a[i] = ((unsigned long long)__float_as_uint(hi) << 32) | __float_as_uint(lo);
    }
    const float bf = 1.0000001f, cf = 1e-7f * (float)blockIdx.x;
    const unsigned long long b = ((unsigned long long)__float_as_uint(bf) << 32) | __float_as_uint(bf);
    const unsigned long long cc = ((unsigned long long)__float_as_uint(cf) << 32) | __float_as_uint(cf);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
#pragma unroll
            for (int i = 0; i < 8; ++i) asm volatile("fma.rn.f32x2 %0, %0, %1, %2;" : "+l"(a[i]) : "l"(b), "l"(cc));
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += __uint_as_float((unsigned)a[i]) + __uint_as_float((unsigned)(a[i] >> 32));
    if (s == 123.456f) sink[0] = s;
}

}  // namespace mlb

// ================================================================================================
// host side: the row-tile family and the stand-alone entry points
// ================================================================================================
using namespace mlb;

cudaError_t TileFamily::set_marks(unsigned long long* ptr) { return cudaMemcpyToSymbol(mlb::g_fwd_marks, &ptr, sizeof(ptr)); }

bool TileFamily::covers(int L) { return L >= 128 && L <= 1024 && (L % 128) == 0; }

void TileFamily::setup(int L, int n_sms) {
    available = covers(L);
    // consumer warpgroups (one active warp per 128 hidden columns) + one producer warpgroup (setmaxnreg split)
    threads = ((L / 128 + 3) / 4) * 128 + 128;
    smem = ((size_t)L * MP + MP * OUT_LD + MP * 4 + (size_t)NSTAGE * KC * L) * sizeof(float) + 2 * NSTAGE * sizeof(uint64_t) + 16;
    int ctas_per_sm = (int)((227 * 1024) / (smem + 1024));
    if (ctas_per_sm < 1) ctas_per_sm = 1;
    if (ctas_per_sm > 4) ctas_per_sm = 4;
    if (ctas_per_sm > 65536 / (threads * 168)) ctas_per_sm = 65536 / (threads * 168) > 0 ? 65536 / (threads * 168) : 1;
    max_ctas[0] = n_sms * (ctas_per_sm > 2 ? 2 : ctas_per_sm);  // a residual in Tensor Memory allows 2 CTAs per SM
    max_ctas[1] = n_sms * ctas_per_sm;
}

template <int TM>
static cudaError_t launch_fwd(const FwdParams& p, int grid, int threads, size_t smem, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(loco_forward_kernel<TM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    loco_forward_kernel<TM><<<grid, threads, smem, st>>>(p);
    return cudaGetLastError();
}

cudaError_t TileFamily::launch(FwdParams p, const FwdPlan& pl, cudaStream_t st, int* issued) const {
    p.n_tiles = (p.n_rows + 2 * pl.tm - 1) / (2 * pl.tm);
    cudaError_t e;
    switch (pl.tm) {
        case 8: e = launch_fwd<8>(p, pl.grid, threads, smem, st); break;
        case 10: e = launch_fwd<10>(p, pl.grid, threads, smem, st); break;
        case 12: e = launch_fwd<12>(p, pl.grid, threads, smem, st); break;
        case 14: e = launch_fwd<14>(p, pl.grid, threads, smem, st); break;
        default: e = launch_fwd<16>(p, pl.grid, threads, smem, st); break;
    }
    if (e == cudaSuccess) ++*issued;
    return e;
}

extern "C" int mlb_preprocess(const float* kps, int n_rows, const float kinv[9], float z_met, int zero_center, float* out_x,
                              void* stream) {
    if (n_rows == 0) return 0;
    if (!kps || !kinv || !out_x || n_rows < 0) return mlb_fail("mlb_preprocess: bad argument");
    const int wpb = 8;
    preprocess_kernel<<<(n_rows + wpb - 1) / wpb, wpb * 32, 0, (cudaStream_t)stream>>>(
        kps, n_rows, kinv[0], kinv[1], kinv[2], kinv[3], kinv[4], kinv[5], z_met != 0.f ? z_met : 10.f, zero_center, out_x);
    MLB_CU(cudaGetLastError());
    mlb_count_launch();
    return 0;
}

extern "C" int mlb_decode(const float* raw, int n_rows, int out_size, int decode_kind, float* dec, void* stream) {
    if (n_rows == 0) return 0;
    if (!raw || !dec || n_rows < 0 || out_size < 1 || out_size > OUT_LD) return mlb_fail("mlb_decode: bad argument");
    if (decode_kind == MLB_DECODE_LOCO && out_size < 9) return mlb_fail("mlb_decode: extract_outputs needs >= 9 columns");
    if (decode_kind == MLB_DECODE_MONO && out_size < 9) return mlb_fail("mlb_decode: extract_outputs_mono needs 9 columns");
    if (decode_kind == MLB_DECODE_DB && out_size < 2) return mlb_fail("mlb_decode: needs 2 columns");
    decode_kernel<<<(n_rows + 127) / 128, 128, 0, (cudaStream_t)stream>>>(raw, n_rows, out_size, decode_kind, dec);
    MLB_CU(cudaGetLastError());
    mlb_count_launch();
    return 0;
}

extern "C" int mlb_laplace_std(const float* d_bi, int n_pass, int n_rows, int n_samples, uint64_t seed, float* out_std,
                               void* stream) {
    if (n_rows == 0) return 0;
    if (!d_bi || !out_std || n_pass < 1 || n_rows < 0 || n_samples < 1) return mlb_fail("mlb_laplace_std: bad argument");
    laplace_std_kernel<<<(n_rows + 127) / 128, 128, 0, (cudaStream_t)stream>>>(d_bi, n_pass, n_rows, n_samples, seed, out_std);
    MLB_CU(cudaGetLastError());
    mlb_count_launch();
    return 0;
}

extern "C" int mlb_ipc_alloc(int device, size_t bytes, void** dev_ptr, unsigned char handle[MLB_IPC_HANDLE_BYTES]) {
    if (!dev_ptr || !handle || bytes == 0) return mlb_fail("mlb_ipc_alloc: bad argument");
    static_assert(sizeof(cudaIpcMemHandle_t) <= MLB_IPC_HANDLE_BYTES, "handle size");
    MLB_CU(cudaSetDevice(device));
    void* ptr = nullptr;
    MLB_CU(cudaMalloc(&ptr, bytes));
    MLB_CU(cudaMemset(ptr, 0, bytes));
    cudaIpcMemHandle_t hd;
    MLB_CU(cudaIpcGetMemHandle(&hd, ptr));
    memset(handle, 0, MLB_IPC_HANDLE_BYTES);
    memcpy(handle, &hd, sizeof(hd));
    *dev_ptr = ptr;
    return 0;
}

extern "C" int mlb_ipc_open(int device, const unsigned char handle[MLB_IPC_HANDLE_BYTES], void** dev_ptr) {
    if (!dev_ptr || !handle) return mlb_fail("mlb_ipc_open: bad argument");
    MLB_CU(cudaSetDevice(device));
    cudaIpcMemHandle_t hd;
    memcpy(&hd, handle, sizeof(hd));
    void* ptr = nullptr;
    MLB_CU(cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess));
    *dev_ptr = ptr;
    return 0;
}

extern "C" int mlb_ipc_close(void* dev_ptr) {
    if (dev_ptr) MLB_CU(cudaIpcCloseMemHandle(dev_ptr));
    return 0;
}

extern "C" int mlb_ipc_free(void* dev_ptr) {
    if (dev_ptr) MLB_CU(cudaFree(dev_ptr));
    return 0;
}

extern "C" int mlb_probe_ffma(int device, int blocks, int iters, double* flops, void* stream) {
    MLB_CU(cudaSetDevice(device));
    static float* sink = nullptr;
    if (!sink) MLB_CU(cudaMalloc(&sink, 16));
    if (iters < 0)
        ffma2_probe_kernel<<<blocks, 512, 0, (cudaStream_t)stream>>>(-iters, sink);  // packed fma.rn.f32x2 variant
    else
        ffma_probe_kernel<<<blocks, 512, 0, (cudaStream_t)stream>>>(iters, sink);
    MLB_CU(cudaGetLastError());
    if (iters < 0) iters = -iters;
    mlb_count_launch();
    if (flops) *flops = (double)blocks * 512.0 * (double)iters * 8.0 * 16.0 * 2.0;
    return 0;
}
