// Fused monoloco training step for B200 (sm_100a): train-mode forward, multi-task Laplace loss and the full
// backward pass as ONE persistent cooperative kernel (or forward / backward halves for the autograd drop-in).
//
// Replaces (reference file:line):
//   monoloco/train/trainer.py:153-161      outputs = model(inputs); loss, _ = mt_loss(outputs, labels); loss.backward()
//   monoloco/network/architectures.py:48-71, 88-102   LocoModel / MyLinearSimple forward in train mode
//                                          (nn.BatchNorm1d batch statistics + running-stat update, nn.Dropout)
//   monoloco/train/losses.py:46-73, 28-43  MultiTaskLoss / AutoTuneMultiTaskLoss.forward
//   monoloco/train/losses.py:104-142       LaplacianLoss;  nn.L1Loss, nn.BCEWithLogitsLoss (losses.py:81-83)
//   torch autograd backward of all of the above
//
// Structure: the grid is persistent (one CTA per SM, cooperative launch) and walks a PHASE list separated by
// grid-wide barriers; the activations of a layer live in L2/HBM between phases, every GEMM-shaped phase reuses the
// inference kernel's machinery (warp-specialised TMA weight stream + register-tiled FFMA2 consumers):
//   PACK                 W -> W^T chunks for the forward stream, zero the accumulators
//   FWD(i)               [normalise block i-1 with its batch statistics -> ReLU -> Dropout -> (+x)] -> Linear i,
//                        per-feature sum / sum-of-squares (fp64 atomics) for block i's BatchNorm
//   FWD_FINAL            last normalise, w_fin head, outputs, (fused) loss + dL/dout
//   BWD_HEAD             head gradients, dL/d(last activation), BN-backward sums of the last block
//   BWD(i)               BN backward of block i (needs the grid-wide sums) -> dX GEMM with the native W ->
//                        dL/d(previous activation) (+ residual / aux-head terms) -> sums for the previous BN
//   DW                   dW_i = Gz_i^T A_i as 32-row x 1024-col tiles streamed over the batch dimension
#include <cuda_runtime.h>
#include <cooperative_groups.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "gemm_tile.cuh"
#include "host_error.h"

namespace mlb {

constexpr int NT = 256;  // consumer threads (8 warps); +128 producer-warpgroup threads
constexpr int MAX_PHASES = 48;
enum { PH_PACK = 0, PH_FWD = 1, PH_FWD_FINAL = 2, PH_BWD_INIT = 3, PH_BWD_HEAD = 4, PH_BWD = 5, PH_DW = 6 };

struct TBlk {
    int K, Kpad, has_bn, res_src, skip_to, bn_index;
    const float *W, *b, *gamma, *beta;
    float *rmean, *rvar, *dW, *db, *dgamma, *dbeta;
    float* Wt;     // [Kpad][L] transposed weights (forward stream)
    float* Z;      // [Bpad][L] Linear output (pre-BN)
    float* Aout;   // [Bpad][L] block output (input of the next block)
    float* G;      // [Bpad][L] dL/dAout
    float* Gz;     // [Bpad][L] dL/dZ
    double* stat;  // [4][L]: sum z, sum z^2, sum gy, sum gy*zhat
};

struct TrainParams {
    TBlk blk[MLB_MAX_BLOCKS];
    int n_blocks, aux_block, L, in_size, out_size, n_rows, n_rows_pad, n_tiles;
    int phase_type[MAX_PHASES], phase_blk[MAX_PHASES], n_phases;
    float p_drop, eps, momentum;
    int update_running;
    unsigned long long seed;
    const uint8_t* drop_mask;
    const float* x;
    float* out;
    const float* g_out_in;
    float* g_out;  // [Bpad][16]
    const float *W_aux, *b_aux, *W_fin, *b_fin;
    float *dW_aux, *db_aux, *dW_fin, *db_fin;
    const float* labels;
    int label_ld, n_tasks;
    int tasks[8];
    float task_scale[8];
    const float* task_scale_dev;  // optional device copy (overrides task_scale)
    float* loss_vals;
    double* loss_acc;  // [8]
    float4* ptab;      // [grid][L][2]
    unsigned* bar_counter;
    int* err_flag;
    unsigned long long* phase_ns;  // [MAX_PHASES + 1] globaltimer at kernel start and after every phase barrier (CTA 0)
};

__device__ __forceinline__ bool keep_elem(const TrainParams& p, int site, int grow, int col) {
    if (p.p_drop <= 0.f) return true;
    if (p.drop_mask != nullptr) return p.drop_mask[((size_t)site * p.n_rows + grow) * p.L + col] != 0;
    return keep_draw(p.seed, (uint32_t)site, (uint32_t)grow, (uint32_t)col, p.p_drop);
}
// Keep decisions of 8 elements of one row as a bit field (bit j <-> element j); ONE mask-vs-hash branch per row, the
// per-launch (seed_mix, thr) and per-column (ch) parts of the hash hoisted by the caller.
//   accumulator layout: columns n0..n0+3 and n0+64..n0+67
__device__ __forceinline__ uint32_t keep_bits_acc(const TrainParams& p, int site, uint32_t seed_mix, uint32_t thr,
                                                  const uint32_t (&ch)[8], size_t grow, int n0) {
    if (p.p_drop <= 0.f) return 0xFFu;
    if (p.drop_mask != nullptr) {
        const uint8_t* m = p.drop_mask + ((size_t)site * p.n_rows + grow) * p.L + n0;
        return bytes_to_bits(*reinterpret_cast<const uint32_t*>(m)) | (bytes_to_bits(*reinterpret_cast<const uint32_t*>(m + 64)) << 4);
    }
    const uint32_t rm = drop_row_mix(seed_mix, (uint32_t)grow);
    uint32_t bits = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) bits |= (drop_keep(rm, ch[j], thr) ? 1u : 0u) << j;
    return bits;
}
//   8 consecutive columns col0..col0+7 (col0 % 8 == 0)
__device__ __forceinline__ uint32_t keep_bits_run(const TrainParams& p, int site, uint32_t seed_mix, uint32_t thr, size_t grow,
                                                  int col0) {
    if (p.p_drop <= 0.f) return 0xFFu;
    if (p.drop_mask != nullptr) {
        const uint8_t* m = p.drop_mask + ((size_t)site * p.n_rows + grow) * p.L + col0;
        return bytes_to_bits(*reinterpret_cast<const uint32_t*>(m)) | (bytes_to_bits(*reinterpret_cast<const uint32_t*>(m + 4)) << 4);
    }
    const uint32_t rm = drop_row_mix(seed_mix, (uint32_t)grow);
    uint32_t bits = 0;
#pragma unroll
    for (int e = 0; e < 8; ++e) bits |= (drop_keep(rm, drop_col_hash((uint32_t)(col0 + e), (uint32_t)site), thr) ? 1u : 0u) << e;
    return bits;
}

// profiling aid: CTAs 0, grid/2 and n_tiles-1 stamp globaltimer at up to 4 points inside every phase
__device__ __forceinline__ void mark(const TrainParams& p, int ph, int slot, int tid) {
    if (tid != 0) return;
    const int b = blockIdx.x;
    const int sel = b == 0 ? 0 : (b == (int)gridDim.x / 2 ? 1 : (b == p.n_tiles - 1 ? 2 : -1));
    if (sel < 0) return;
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.phase_ns[MAX_PHASES + 1 + (ph * 3 + sel) * 8 + slot] = t;
}

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* ptr) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ptr) : "memory");
    return v;
}

// number of weight-stream chunks of a phase for ONE tile / item (producer and consumer walk the same sequence)
__device__ __forceinline__ int chain_end(const TrainParams& p, int i) {
    // BWD(i): dX GEMMs for cur = i, i-1, ... while the block below has no BatchNorm; returns the last `cur`
    int cur = i;
    while (cur >= 1 && !p.blk[cur - 1].has_bn && cur - 1 >= 1) cur--;
    return cur;
}

// ------------------------------------------------------------------------------------------------ producer
__device__ __forceinline__ void wait_released(volatile int* released, int need) {
    while (*released < need) __nanosleep(64);
}

template <int TM>
__device__ void train_producer(const TrainParams& p, float* ring, float* astage, uint64_t* full, uint64_t* empty,
                               volatile int* released) {
    RingState rs = {0u, 0u, 0u};
    const int L = p.L;
    bool waited_pack = false;
    auto acquire_slot = [&]() {
        if (rs.q >= NSTAGE) mbar_wait_backoff(&empty[rs.stage], rs.parity ^ 1, p.err_flag);
    };
    for (int ph = 0; ph < p.n_phases; ++ph) {
        const int type = p.phase_type[ph], bi = p.phase_blk[ph];
        if (type != PH_FWD && type != PH_BWD && type != PH_DW) continue;
        // Wt is written by the PACK phase and the DW operands by the backward phases: wait for that phase's barrier.
        // Native W (backward) and, after the first FWD phase, Wt are static -> the stream prefetches across barriers.
        const bool depends = type == PH_DW || (type == PH_FWD && !waited_pack);
        if (depends) {
            wait_released(released, ph);
            __threadfence();
            if (type == PH_FWD) waited_pack = true;
        }
        if (type == PH_FWD) {
            const TBlk& b = p.blk[bi];
            const uint32_t bytes = (uint32_t)(KC * L * sizeof(float));
            for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x)
                for (int ch = 0; ch < b.Kpad / KC; ++ch) {
                    acquire_slot();
                    mbar_expect_tx(&full[rs.stage], bytes);
                    tma_bulk_g2s(ring + (size_t)rs.stage * KC * L, b.Wt + (size_t)ch * KC * L, bytes, &full[rs.stage]);
                    ring_advance(rs);
                }
        } else if (type == PH_BWD) {
            if (bi == 0) continue;
            const int last = chain_end(p, bi);
            const uint32_t bytes = (uint32_t)(KC * L * sizeof(float));
            for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x)
                for (int cur = bi; cur >= last; --cur)
                    for (int ch = 0; ch < L / KC; ++ch) {  // native W [n][k]: KC rows of n, K == L columns
                        acquire_slot();
                        mbar_expect_tx(&full[rs.stage], bytes);
                        tma_bulk_g2s(ring + (size_t)rs.stage * KC * L, p.blk[cur].W + (size_t)ch * KC * L, bytes,
                                     &full[rs.stage]);
                        ring_advance(rs);
                    }
        } else {  // PH_DW: stream-K split of the linearised (item, b-chunk) space -> every CTA gets the same number of chunks
            const int n_items = (p.n_blocks - 1) * (L / 32);
            const int nchunks = p.n_rows_pad / KC;
            const long long total = (long long)n_items * nchunks;
            const long long u0 = total * blockIdx.x / gridDim.x, u1 = total * (blockIdx.x + 1) / gridDim.x;
            const uint32_t bytes = (uint32_t)(KC * L * sizeof(float) + KC * 32 * sizeof(float));
            for (long long u = u0; u < u1;) {
                const int item = (int)(u / nchunks), c0 = (int)(u % nchunks);
                const int c1 = (int)min((long long)nchunks, c0 + (u1 - u));
                const int b_i = 1 + item / (L / 32), n0 = (item % (L / 32)) * 32;
                const TBlk& b = p.blk[b_i];
                const float* ain = p.blk[b_i - 1].Aout;
                for (int ch = c0; ch < c1; ++ch) {
                    acquire_slot();
                    mbar_expect_tx(&full[rs.stage], bytes);
                    tma_bulk_g2s(ring + (size_t)rs.stage * KC * L, ain + (size_t)ch * KC * L, KC * L * sizeof(float),
                                 &full[rs.stage]);
#pragma unroll
                    for (int j = 0; j < KC; ++j)
                        tma_bulk_g2s(astage + ((size_t)rs.stage * KC + j) * 32, b.Gz + ((size_t)ch * KC + j) * L + n0,
                                     32 * sizeof(float), &full[rs.stage]);
                    ring_advance(rs);
                }
                u += c1 - c0;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------ consumer helpers
__device__ __forceinline__ void csync() { named_sync(1, NT); }

__device__ void grid_barrier(const TrainParams& p, unsigned& target, volatile int* released, int tid) {
    csync();
    if (tid == 0) {
        __threadfence();
        atomicAdd(p.bar_counter, 1u);
        target += gridDim.x;
        unsigned spins = 0;
        while (ld_acquire_u32(p.bar_counter) < target) {
            __nanosleep(40);
            if (++spins > (1u << 26)) {
                atomicExch(p.err_flag, 2);
                __threadfence_system();
                __trap();
            }
        }
        __threadfence();
        *released = *released + 1;
    }
    csync();
}

// per-CTA table (mean, invstd, gamma, beta), (c1 = S3/B, c2 = S4/B, -, -) of one BatchNorm block
__device__ void build_ptab(const TrainParams& p, const TBlk& b, float4* ptab, int tid, bool update_running, bool write_dgb) {
    const double invB = 1.0 / (double)p.n_rows;
    for (int f = tid; f < p.L; f += NT) {
        const double s1 = b.stat[f], s2 = b.stat[p.L + f];
        const double mean = s1 * invB;
        double var = s2 * invB - mean * mean;
        if (var < 0.0) var = 0.0;
        const float invstd = (float)(1.0 / sqrt(var + (double)p.eps));
        ptab[2 * f] = make_float4((float)mean, invstd, b.gamma[f], b.beta[f]);
        ptab[2 * f + 1] = make_float4((float)(b.stat[2 * p.L + f] * invB), (float)(b.stat[3 * p.L + f] * invB), 0.f, 0.f);
        if (update_running && b.rmean != nullptr) {
            // nn.BatchNorm1d: running = (1-m) running + m batch; running_var uses the unbiased batch variance
            const double unb = p.n_rows > 1 ? var * (double)p.n_rows / (double)(p.n_rows - 1) : var;
            b.rmean[f] = (1.f - p.momentum) * b.rmean[f] + p.momentum * (float)mean;
            b.rvar[f] = (1.f - p.momentum) * b.rvar[f] + p.momentum * (float)unb;
        }
        if (write_dgb) {
            b.dgamma[f] = (float)b.stat[3 * p.L + f];
            b.dbeta[f] = (float)b.stat[2 * p.L + f];
        }
    }
}

template <int TM>
__device__ __forceinline__ bool slot_valid(int slot, int rows_here, int& r) {
    const int grp = slot >> 4, i = slot & 15;
    r = grp * TM + i;
    return i < TM && r < rows_here;
}

// narrow head forward: outs[slot][col0 + o] = bias[o] + sum_k act[k][slot] * W[o][k]   (one warp per output column)
__device__ __forceinline__ void head_forward(const float* __restrict__ W, const float* __restrict__ bias, int N, int K,
                                             const float* act, float* outs, int col0, int warp, int lane) {
    for (int o = warp; o < N; o += NT / 32) outs[lane * OUT_LD + col0 + o] = head_column(W + (size_t)o * K, __ldg(bias + o), K, act, lane, lane, MP);
}

// aux head (after LocoModel.w2) and, in the final phase, the w_fin head + fused MultiTaskLoss and its gradient g_out
template <int TM>
__device__ __forceinline__ void fwd_heads(const TrainParams& p, bool final_phase, int prev, const float* act, float* outs,
                                          int row0, int rows_here, int tid, int warp, int lane, int nfin, float invB) {
    const int L = p.L;
    if (prev >= 0 && prev == p.aux_block) {  // w_aux head reads LocoModel.w2's output (architectures.py:60)
        head_forward(p.W_aux, p.b_aux, 1, L, act, outs, nfin, warp, lane);
        csync();
        if (tid < MP) {
            int rr;
            if (slot_valid<TM>(tid, rows_here, rr)) p.out[(size_t)(row0 + rr) * p.out_size + nfin] = outs[tid * OUT_LD + nfin];
        }
    }
    if (final_phase) {
        head_forward(p.W_fin, p.b_fin, nfin, L, act, outs, 0, warp, lane);  // architectures.py:67
        csync();
        if (tid < MP) {
            int rr;
            const bool v = slot_valid<TM>(tid, rows_here, rr);
            const size_t gr = (size_t)row0 + rr;
            float lossv[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            if (v) {
                float* o = outs + tid * OUT_LD;
                for (int k = 0; k < nfin; ++k) p.out[gr * p.out_size + k] = o[k];
                if (p.labels != nullptr) {
                    o[nfin] = p.out[gr * p.out_size + nfin];
                    const float* y = p.labels + gr * p.label_ld;
                    float gsum[OUT_LD];
#pragma unroll
                    for (int k = 0; k < OUT_LD; ++k) gsum[k] = 0.f;
                    for (int t = 0; t < p.n_tasks; ++t) {
                        const float s = (p.task_scale_dev != nullptr ? p.task_scale_dev[t] : p.task_scale[t]) * invB;
                        const int task = p.tasks[t];
                        if (task == MLB_TASK_D) {  // LaplacianLoss, losses.py:121-131
                            const float mu = o[2], si = o[3], xx = y[3];
                            const float nrm = 1.f - mu / xx, e = expf(-si);
                            lossv[t] = fabsf(nrm) * e + 0.01f + si + 2.f;
                            const float sg = nrm > 0.f ? 1.f : (nrm < 0.f ? -1.f : 0.f);
                            gsum[2] += s * sg * (-1.f / xx) * e;
                            gsum[3] += s * (1.f - fabsf(nrm) * e);
                        } else if (task == MLB_TASK_ORI) {  // nn.L1Loss over [B,2]
                            const float d7 = o[7] - y[7], d8 = o[8] - y[8];
                            lossv[t] = 0.5f * (fabsf(d7) + fabsf(d8));
                            gsum[7] += 0.5f * s * (d7 > 0.f ? 1.f : (d7 < 0.f ? -1.f : 0.f));
                            gsum[8] += 0.5f * s * (d8 > 0.f ? 1.f : (d8 < 0.f ? -1.f : 0.f));
                        } else if (task == MLB_TASK_AUX) {  // nn.BCEWithLogitsLoss, label column 10
                            const float zz = o[9], tt = y[10];
                            lossv[t] = fmaxf(zz, 0.f) - zz * tt + log1pf(expf(-fabsf(zz)));
                            gsum[9] += s * (1.f / (1.f + expf(-zz)) - tt);
                        } else {  // nn.L1Loss on one column: x, y, h, w, l (process.py:252-254, 293-304)
                            const int col = task == MLB_TASK_X ? 0 : task == MLB_TASK_Y ? 1 : task == MLB_TASK_H ? 4
                                                                     : task == MLB_TASK_W ? 5 : 6;
                            const float d = o[col] - y[col];
                            lossv[t] = fabsf(d);
                            gsum[col] += s * (d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f));
                        }
                    }
                    for (int k = 0; k < OUT_LD; ++k) p.g_out[gr * OUT_LD + k] = gsum[k];
                }
            }
            if (p.labels != nullptr) {
                for (int t = 0; t < p.n_tasks; ++t) {
                    float v2 = lossv[t];
                    for (int sft = 16; sft > 0; sft >>= 1) v2 += __shfl_xor_sync(0xffffffffu, v2, sft);
                    if (tid == 0) atomicAdd(&p.loss_acc[t], (double)v2);
                }
            }
        }
        csync();
    }
}

// ------------------------------------------------------------------------------------------------ the kernel
template <int TM>
__global__ void __launch_bounds__(MAX_THREADS, 1) loco_train_kernel(const __grid_constant__ TrainParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int L = p.L;
    const int nwarps = L >> 7;  // active consumer warps (one per 128 columns)
    constexpr int ROWS = 2 * TM;

    float* act = reinterpret_cast<float*>(smem_raw);      // [L][MP]; its head doubles as the dW A-stage / PACK transpose buffer
    const int act_floats = max(L * MP, 8 * 32 * 33);
    float* outs = act + act_floats;                        // [MP][OUT_LD]
    float* ring = outs + MP * OUT_LD;                      // [NSTAGE][KC][L]
    uint64_t* full = reinterpret_cast<uint64_t*>(ring + (size_t)NSTAGE * KC * L);
    uint64_t* empty = full + NSTAGE;
    volatile int* released = reinterpret_cast<volatile int*>(empty + NSTAGE);

    for (int i = tid; i < act_floats + MP * OUT_LD; i += blockDim.x) act[i] = 0.f;
    if (tid == 0) {
        for (int s = 0; s < NSTAGE; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], nwarps);
        }
        mbar_fence_init();
        *released = 0;
    }
    __syncthreads();

    if (warp >= 8) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");
        if (warp == 8 && lane == 0) train_producer<TM>(p, ring, act, full, empty, released);
        return;
    }
    asm volatile("setmaxnreg.inc.sync.aligned.u32 240;");
    // NOTE: every consumer thread (tid < 256) takes part in csync(); warps >= nwarps only skip the GEMM math.
    const bool gemm_warp = warp < nwarps;
    const int g = lane >> 4, c = lane & 15;
    const int n0 = warp * 128 + c * 4;
    float4* ptab = p.ptab + (size_t)blockIdx.x * L * 2;
    RingState rs = {0u, 0u, 0u};
    unsigned bar_target = 0;
    const float inv_keep = p.p_drop > 0.f ? 1.0f / (1.0f - p.p_drop) : 1.0f;
    const float invB = 1.0f / (float)p.n_rows;
    const int nfin = p.out_size - 1;
    const uint32_t seed_mix = drop_seed_mix(p.seed), drop_thr = drop_threshold(p.p_drop);
    auto col_hashes = [&](int site, uint32_t (&ch)[8]) {
#pragma unroll
        for (int j = 0; j < 8; ++j) ch[j] = drop_col_hash((uint32_t)col_of(n0, j), (uint32_t)site);
    };

    if (blockIdx.x == 0 && tid == 0) {
        unsigned long long t0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        p.phase_ns[0] = t0;
    }
    auto end_phase = [&](int ph_done) {
        grid_barrier(p, bar_target, released, tid);
        mark(p, ph_done, 3, tid);
        if (blockIdx.x == 0 && tid == 0) {
            unsigned long long t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            p.phase_ns[ph_done + 1] = t1;
        }
    };
    for (int ph = 0; ph < p.n_phases; ++ph) {
        const int type = p.phase_type[ph], bi = p.phase_blk[ph];

        if (type == PH_PACK) {
            // ---- W [L][K] -> Wt [Kpad][L] through 32x33 shared tiles (one per warp), zero accumulators
            float* tbuf = act + warp * 32 * 33;
            for (int b_i = 0; b_i < p.n_blocks; ++b_i) {
                const TBlk& b = p.blk[b_i];
                const int kt = (b.Kpad + 31) / 32, nt = L / 32;
                for (int t = blockIdx.x * 8 + warp; t < kt * nt; t += gridDim.x * 8) {
                    const int k0 = (t / nt) * 32, nb = (t % nt) * 32;
                    for (int r = 0; r < 32; ++r) {
                        const int k = k0 + lane;
                        tbuf[r * 33 + lane] = k < b.K ? b.W[(size_t)(nb + r) * b.K + k] : 0.f;
                    }
                    __syncwarp();
                    for (int r = 0; r < 32; ++r)
                        if (k0 + r < b.Kpad) b.Wt[(size_t)(k0 + r) * L + nb + lane] = tbuf[lane * 33 + r];
                    __syncwarp();
                }
                for (int f = blockIdx.x * NT + tid; f < 4 * L; f += gridDim.x * NT) b.stat[f] = 0.0;
            }
            if (blockIdx.x == 0 && tid < 8) p.loss_acc[tid] = 0.0;
            csync();
            for (int i = tid; i < 8 * 32 * 33; i += NT) act[i] = 0.f;
        } else if (type == PH_BWD_INIT) {
            for (int b_i = 0; b_i < p.n_blocks; ++b_i) {
                const TBlk& b = p.blk[b_i];
                for (int f = blockIdx.x * NT + tid; f < 2 * L; f += gridDim.x * NT) b.stat[2 * L + f] = 0.0;
                for (int f = blockIdx.x * NT + tid; f < L; f += gridDim.x * NT) b.db[f] = 0.f;
            }
            for (int f = blockIdx.x * NT + tid; f < L * p.blk[0].K; f += gridDim.x * NT) p.blk[0].dW[f] = 0.f;
            for (int b_i = 1; b_i < p.n_blocks; ++b_i) {
                float4* dw4 = reinterpret_cast<float4*>(p.blk[b_i].dW);
                for (int f = blockIdx.x * NT + tid; f < L * L / 4; f += gridDim.x * NT) dw4[f] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            for (int f = blockIdx.x * NT + tid; f < L * nfin; f += gridDim.x * NT) p.dW_fin[f] = 0.f;
            for (int f = blockIdx.x * NT + tid; f < L; f += gridDim.x * NT) p.dW_aux[f] = 0.f;
            if (blockIdx.x == 0 && tid < nfin) p.db_fin[tid] = 0.f;
            if (blockIdx.x == 0 && tid == 0) p.db_aux[0] = 0.f;
        } else if (type == PH_FWD || type == PH_FWD_FINAL) {
            // ============================================================================ forward
            const bool final_phase = type == PH_FWD_FINAL;
            const int prev = final_phase ? p.n_blocks - 1 : bi - 1;
            if (prev >= 0 && p.blk[prev].has_bn) {
                build_ptab(p, p.blk[prev], ptab, tid, p.update_running && blockIdx.x == 0, false);
                csync();
            }
            for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
                const int row0 = tile * ROWS;
                const int rows_here = min(ROWS, p.n_rows - row0);
                int r;
                const bool valid = slot_valid<TM>(lane, rows_here, r);
                const size_t grow = (size_t)row0 + r;
                // ---- prologue: the input tile of this block, k-major in `act`
                if (prev < 0) {
                    const int kpad = p.blk[0].Kpad;
                    for (int idx = tid; idx < ROWS * kpad; idx += NT) {
                        const int rr = idx / kpad, k = idx % kpad;
                        float v = 0.f;
                        if (rr < rows_here && k < p.in_size) v = __ldg(p.x + (size_t)(row0 + rr) * p.in_size + k);
                        act[k * MP + slot_of_row(rr, TM)] = v;
                    }
                } else {
                    const TBlk& pb = p.blk[prev];
                    // __restrict__ views: lets the unrolled iterations issue all their L2 loads before the first store
                    const float* __restrict__ Zp = pb.Z;
                    float* __restrict__ Ap = pb.Aout;
                    const float* __restrict__ Rp = pb.res_src >= 0 ? p.blk[pb.res_src].Aout : nullptr;
                    const float4* __restrict__ pt = ptab;
#pragma unroll 4
                    for (int k8 = warp; k8 < L / 8; k8 += 8) {
                        float h[8];
                        if (valid) {
                            if (pb.has_bn) {
                                const float4 z0 = *reinterpret_cast<const float4*>(Zp + grow * L + k8 * 8);
                                const float4 z1 = *reinterpret_cast<const float4*>(Zp + grow * L + k8 * 8 + 4);
                                const float z[8] = {z0.x, z0.y, z0.z, z0.w, z1.x, z1.y, z1.z, z1.w};
                                float res[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                                if (Rp != nullptr) {
                                    const float* ra = Rp + grow * L + k8 * 8;
                                    const float4 r0 = *reinterpret_cast<const float4*>(ra);
                                    const float4 r1 = *reinterpret_cast<const float4*>(ra + 4);
                                    res[0] = r0.x, res[1] = r0.y, res[2] = r0.z, res[3] = r0.w;
                                    res[4] = r1.x, res[5] = r1.y, res[6] = r1.z, res[7] = r1.w;
                                }
                                const uint32_t kb = keep_bits_run(p, pb.bn_index, seed_mix, drop_thr, grow, k8 * 8);
#pragma unroll
                                for (int e = 0; e < 8; ++e) {
                                    const float4 t = pt[2 * (k8 * 8 + e)];  // mean, invstd, gamma, beta
                                    const float zh = (z[e] - t.x) * t.y;
                                    float y = fmaxf(fmaf(zh, t.z, t.w), 0.f);
                                    y = (kb >> e) & 1u ? y * inv_keep : 0.f;
                                    h[e] = y + res[e];
                                }
                                float* dst = Ap + grow * L + k8 * 8;
                                *reinterpret_cast<float4*>(dst) = make_float4(h[0], h[1], h[2], h[3]);
                                *reinterpret_cast<float4*>(dst + 4) = make_float4(h[4], h[5], h[6], h[7]);
                            } else {
                                const float4 a0 = *reinterpret_cast<const float4*>(Ap + grow * L + k8 * 8);
                                const float4 a1 = *reinterpret_cast<const float4*>(Ap + grow * L + k8 * 8 + 4);
                                h[0] = a0.x, h[1] = a0.y, h[2] = a0.z, h[3] = a0.w;
                                h[4] = a1.x, h[5] = a1.y, h[6] = a1.z, h[7] = a1.w;
                            }
                        } else {
#pragma unroll
                            for (int e = 0; e < 8; ++e) h[e] = 0.f;
                        }
#pragma unroll
                        for (int e = 0; e < 8; ++e) act[(k8 * 8 + e) * MP + lane] = h[e];
                    }
                    // keep the DW phase's tail chunk clean: rows [n_rows, n_rows_pad) of every saved activation are zero
                    if (pb.has_bn && tile == p.n_tiles - 1)
                        for (int idx = tid; idx < (p.n_rows_pad - p.n_rows) * L; idx += NT) pb.Aout[(size_t)p.n_rows * L + idx] = 0.f;
                }
                csync();
                mark(p, ph, 0, tid);
                fwd_heads<TM>(p, final_phase, prev, act, outs, row0, rows_here, tid, warp, lane, nfin, invB);
                if (final_phase) continue;
                // ---- GEMM + epilogue of block bi
                const TBlk& b = p.blk[bi];
                if (gemm_warp) {
                    unsigned long long acc2[TM / 2][8];
                    acc_zero<TM>(acc2);
                    tile_gemm<TM>(acc2, b.Kpad / KC, [&](int ch, unsigned) { return act + (size_t)ch * KC * MP; }, ring, full,
                                  empty, rs, n0, g, lane, L, p.err_flag);
                    mark(p, ph, 1, tid);
                    float acc[TM][8];
                    acc_unpack<TM>(acc2, acc);
                    const float4 b0 = __ldg(reinterpret_cast<const float4*>(b.b + n0));
                    const float4 b1 = __ldg(reinterpret_cast<const float4*>(b.b + n0 + 64));
                    const float bias[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                    float s1[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s2[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                    float* dstbase = b.has_bn ? b.Z : b.Aout;
#pragma unroll
                    for (int i = 0; i < TM; ++i) {
                        const int rr = g * TM + i;
                        if (rr < rows_here) {
                            float z[8];
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                z[j] = acc[i][j] + bias[j];
                                s1[j] += z[j];
                                s2[j] = fmaf(z[j], z[j], s2[j]);
                            }
                            float* dst = dstbase + (size_t)(row0 + rr) * L + n0;
                            *reinterpret_cast<float4*>(dst) = make_float4(z[0], z[1], z[2], z[3]);
                            *reinterpret_cast<float4*>(dst + 64) = make_float4(z[4], z[5], z[6], z[7]);
                        }
                    }
                    if (b.has_bn) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            s1[j] += __shfl_xor_sync(0xffffffffu, s1[j], 16);
                            s2[j] += __shfl_xor_sync(0xffffffffu, s2[j], 16);
                            if (g == 0) {
                                atomicAdd(&b.stat[col_of(n0, j)], (double)s1[j]);
                                atomicAdd(&b.stat[L + col_of(n0, j)], (double)s2[j]);
                            }
                        }
                    } else if (tile == p.n_tiles - 1) {
                        for (int idx = lane; idx < (p.n_rows_pad - p.n_rows) * 128; idx += 32)
                            b.Aout[(size_t)p.n_rows * L + (size_t)(idx / 128) * L + warp * 128 + idx % 128] = 0.f;
                    }
                }
                csync();
                mark(p, ph, 2, tid);
            }
        } else if (type == PH_BWD_HEAD) {
            // ============================================================================ head backward
            const TBlk& lb = p.blk[p.n_blocks - 1];
            const TBlk& ab = p.blk[p.aux_block];
            const float* gsrc = p.labels != nullptr ? p.g_out : p.g_out_in;
            const int gld = p.labels != nullptr ? OUT_LD : p.out_size;
            build_ptab(p, lb, ptab, tid, false, false);
            csync();
            float dbacc = 0.f;  // tid < out_size: db_fin[tid] / db_aux
            for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
                const int row0 = tile * ROWS;
                const int rows_here = min(ROWS, p.n_rows - row0);
                for (int idx = tid; idx < ROWS * OUT_LD; idx += NT) {
                    const int rr = idx / OUT_LD, k = idx % OUT_LD;
                    outs[rr * OUT_LD + k] = (rr < rows_here && k < p.out_size) ? gsrc[(size_t)(row0 + rr) * gld + k] : 0.f;
                }
                csync();
                if (tid < p.out_size)
                    for (int rr = 0; rr < rows_here; ++rr) dbacc += outs[rr * OUT_LD + tid];
                // thread <-> up to 4 features k (coalesced rows); rows outer / features inner so that 12 independent
                // L2 loads are in flight per iteration instead of 3
                constexpr int KQ = 4;
                int kq[KQ];
                float wf[KQ][OUT_LD], accf[KQ][OUT_LD], acca[KQ], s3[KQ], s4[KQ];
                float4 tq[KQ];
#pragma unroll
                for (int q = 0; q < KQ; ++q) {
                    const int kk = tid + q * NT;
                    kq[q] = kk < L ? (kk + (int)blockIdx.x * 64) % L : -1;  // every CTA starts elsewhere (atomics spread)
                    acca[q] = s3[q] = s4[q] = 0.f;
                    tq[q] = kq[q] >= 0 ? ptab[2 * kq[q]] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int o = 0; o < OUT_LD; ++o) {
                        accf[q][o] = 0.f;
                        wf[q][o] = (kq[q] >= 0 && o < nfin) ? __ldg(p.W_fin + (size_t)o * L + kq[q]) : 0.f;
                    }
                }
                for (int rr = 0; rr < rows_here; ++rr) {
                    const size_t gr = (size_t)row0 + rr;
                    const float* go = outs + rr * OUT_LD;
                    float a9[KQ], a8[KQ], zz[KQ];
#pragma unroll
                    for (int q = 0; q < KQ; ++q) {
                        const size_t off = gr * L + (kq[q] >= 0 ? kq[q] : 0);
                        a9[q] = lb.Aout[off], a8[q] = ab.Aout[off], zz[q] = lb.Z[off];
                    }
#pragma unroll
                    for (int q = 0; q < KQ; ++q) {
                        if (kq[q] < 0) continue;
                        float G = 0.f;
#pragma unroll
                        for (int o = 0; o < OUT_LD; ++o) {
                            if (o < nfin) {
                                G = fmaf(go[o], wf[q][o], G);
                                accf[q][o] = fmaf(go[o], a9[q], accf[q][o]);
                            }
                        }
                        acca[q] = fmaf(go[nfin], a8[q], acca[q]);
                        lb.G[gr * L + kq[q]] = G;
                        const float zh = (zz[q] - tq[q].x) * tq[q].y;
                        const float y = fmaf(zh, tq[q].z, tq[q].w);
                        float gy = y > 0.f ? G : 0.f;
                        gy = keep_elem(p, lb.bn_index, (int)gr, kq[q]) ? gy * inv_keep : 0.f;
                        s3[q] += gy;
                        s4[q] = fmaf(gy, zh, s4[q]);
                    }
                }
#pragma unroll
                for (int q = 0; q < KQ; ++q) {
                    if (kq[q] < 0) continue;
                    for (int o = 0; o < nfin; ++o) atomicAdd(p.dW_fin + (size_t)o * L + kq[q], accf[q][o]);
                    atomicAdd(p.dW_aux + kq[q], acca[q]);
                    atomicAdd(&lb.stat[2 * L + kq[q]], (double)s3[q]);
                    atomicAdd(&lb.stat[3 * L + kq[q]], (double)s4[q]);
                }
                csync();
            }
            if (tid < nfin) atomicAdd(p.db_fin + tid, dbacc);
            if (tid == nfin) atomicAdd(p.db_aux, dbacc);
        } else if (type == PH_BWD) {
            // ============================================================================ backward of block bi
            const TBlk& b = p.blk[bi];
            const float* gsrc = p.labels != nullptr ? p.g_out : p.g_out_in;
            const int gld = p.labels != nullptr ? OUT_LD : p.out_size;
            build_ptab(p, b, ptab, tid, false, blockIdx.x == 0);
            csync();
            const int last = bi >= 1 ? chain_end(p, bi) : 0;
            for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
                const int row0 = tile * ROWS;
                const int rows_here = min(ROWS, p.n_rows - row0);
                int r;
                const bool valid = slot_valid<TM>(lane, rows_here, r);
                const size_t grow = (size_t)row0 + r;
                // ---- prologue: gz = gamma*invstd*(gy - mean(gy) - zhat*mean(gy*zhat)) -> Gz (global) and act (k-major)
                const float* __restrict__ Zp = b.Z;
                const float* __restrict__ Gp = b.G;
                float* __restrict__ Gzp = b.Gz;
                const float4* __restrict__ pt = ptab;
#pragma unroll 4
                for (int k8 = warp; k8 < L / 8; k8 += 8) {
                    float gz[8];
                    if (valid) {
                        const float4 z0 = *reinterpret_cast<const float4*>(Zp + grow * L + k8 * 8);
                        const float4 z1 = *reinterpret_cast<const float4*>(Zp + grow * L + k8 * 8 + 4);
                        const float4 g0 = *reinterpret_cast<const float4*>(Gp + grow * L + k8 * 8);
                        const float4 g1 = *reinterpret_cast<const float4*>(Gp + grow * L + k8 * 8 + 4);
                        const float z[8] = {z0.x, z0.y, z0.z, z0.w, z1.x, z1.y, z1.z, z1.w};
                        const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
                        const uint32_t kb = keep_bits_run(p, b.bn_index, seed_mix, drop_thr, grow, k8 * 8);
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            const float4 t = pt[2 * (k8 * 8 + e)];
                            const float4 u = pt[2 * (k8 * 8 + e) + 1];
                            const float zh = (z[e] - t.x) * t.y;
                            const float y = fmaf(zh, t.z, t.w);
                            float gy = y > 0.f ? gg[e] : 0.f;
                            gy = (kb >> e) & 1u ? gy * inv_keep : 0.f;
                            gz[e] = t.z * t.y * (gy - u.x - zh * u.y);
                        }
                        float* dst = Gzp + grow * L + k8 * 8;
                        *reinterpret_cast<float4*>(dst) = make_float4(gz[0], gz[1], gz[2], gz[3]);
                        *reinterpret_cast<float4*>(dst + 4) = make_float4(gz[4], gz[5], gz[6], gz[7]);
                    } else {
#pragma unroll
                        for (int e = 0; e < 8; ++e) gz[e] = 0.f;
                    }
#pragma unroll
                    for (int e = 0; e < 8; ++e) act[(k8 * 8 + e) * MP + lane] = gz[e];
                    // nn.Linear.bias in front of a BatchNorm: db = sum_b gz = gamma*invstd*(S3 - B*c1 - c2*sum(zhat)) == 0
                    // identically (the reference's autograd returns ~1e-9 rounding noise); db stays at the zero BWD_INIT wrote.
                }
                if (tile == p.n_tiles - 1)
                    for (int idx = tid; idx < (p.n_rows_pad - p.n_rows) * L; idx += NT) b.Gz[(size_t)p.n_rows * L + idx] = 0.f;
                csync();
                mark(p, ph, 0, tid);
                if (bi == 0) {
                    // first layer: dW0[n][k] = sum_rows gz[row][n] * x[row][k]  (K = 34 | 68), no dX needed.
                    // thread <-> feature n (coalesced re-read of the Gz rows just written), x tile broadcast from smem
                    // (ring stage 0 is idle: the producer only restarts after this phase's barrier).
                    float* xs = ring;
                    for (int idx = tid; idx < rows_here * b.K; idx += NT)
                        xs[idx] = __ldg(p.x + (size_t)row0 * p.in_size + idx);
                    csync();
                    for (int n = tid; n < L; n += NT) {
                        float gzr[ROWS];
#pragma unroll
                        for (int rr = 0; rr < ROWS; ++rr) gzr[rr] = rr < rows_here ? b.Gz[(size_t)(row0 + rr) * L + n] : 0.f;
                        for (int kk = 0; kk < b.K; ++kk) {
                            const int k = (kk + (int)blockIdx.x) % b.K;  // de-synchronise the CTAs' atomics on one address
                            float a = 0.f;
#pragma unroll
                            for (int rr = 0; rr < ROWS; ++rr) a = fmaf(gzr[rr], rr < rows_here ? xs[rr * b.K + k] : 0.f, a);
                            atomicAdd(b.dW + (size_t)n * b.K + k, a);
                        }
                    }
                    csync();
                    continue;
                }
                for (int cur = bi; cur >= last; --cur) {
                    const TBlk& pb = p.blk[cur - 1];  // the block whose output gradient this GEMM produces
                    if (gemm_warp) {
                        unsigned long long acc2[TM / 2][8];
                        acc_zero<TM>(acc2);
                        tile_gemm<TM>(acc2, L / KC, [&](int ch, unsigned) { return act + (size_t)ch * KC * MP; }, ring, full, empty,
                                      rs, n0, g, lane, L, p.err_flag);
                        mark(p, ph, 1, tid);
                        float acc[TM][8];
                        acc_unpack<TM>(acc2, acc);
                        float wa[8], mean[8], invstd[8], gam[8], bet[8];
                        uint32_t ch[8];
                        col_hashes(pb.has_bn ? pb.bn_index : 0, ch);
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const int col = col_of(n0, j);
                            wa[j] = (cur - 1 == p.aux_block) ? __ldg(p.W_aux + col) : 0.f;
                            if (pb.has_bn) {
                                const double m = pb.stat[col] * (double)invB;
                                double var = pb.stat[L + col] * (double)invB - m * m;
                                if (var < 0.0) var = 0.0;
                                mean[j] = (float)m;
                                invstd[j] = (float)(1.0 / sqrt(var + (double)p.eps));
                                gam[j] = __ldg(pb.gamma + col);
                                bet[j] = __ldg(pb.beta + col);
                            }
                        }
                        float s3[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s4[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                        // __restrict__ views (distinct workspace buffers): the loads of later rows may pass the stores of earlier ones
                        const float* __restrict__ SKp = pb.skip_to >= 0 ? p.blk[pb.skip_to].G : nullptr;
                        const float* __restrict__ Zq = pb.Z;
                        const float* __restrict__ gsr = gsrc;
                        float* __restrict__ Gq = pb.G;
                        float* __restrict__ Gzq = pb.Gz;
#pragma unroll
                        for (int i = 0; i < TM; ++i) {
                            const int rr = g * TM + i;
                            if (rr < rows_here) {
                                const size_t gr = (size_t)row0 + rr;
                                float G[8];
#pragma unroll
                                for (int j = 0; j < 8; ++j) G[j] = acc[i][j];
                                if (pb.skip_to >= 0) {  // x + y of MyLinearSimple: the skip path's gradient (architectures.py:100)
                                    const float* sk = SKp + gr * L + n0;
                                    const float4 k0 = *reinterpret_cast<const float4*>(sk);
                                    const float4 k1 = *reinterpret_cast<const float4*>(sk + 64);
                                    G[0] += k0.x, G[1] += k0.y, G[2] += k0.z, G[3] += k0.w;
                                    G[4] += k1.x, G[5] += k1.y, G[6] += k1.z, G[7] += k1.w;
                                }
                                if (cur - 1 == p.aux_block) {
                                    const float ga = gsr[gr * gld + nfin];
#pragma unroll
                                    for (int j = 0; j < 8; ++j) G[j] = fmaf(ga, wa[j], G[j]);
                                }
                                float* dst = Gq + gr * L + n0;
                                *reinterpret_cast<float4*>(dst) = make_float4(G[0], G[1], G[2], G[3]);
                                *reinterpret_cast<float4*>(dst + 64) = make_float4(G[4], G[5], G[6], G[7]);
                                if (pb.has_bn) {
                                    const float4 z0 = *reinterpret_cast<const float4*>(Zq + gr * L + n0);
                                    const float4 z1 = *reinterpret_cast<const float4*>(Zq + gr * L + n0 + 64);
                                    const float z[8] = {z0.x, z0.y, z0.z, z0.w, z1.x, z1.y, z1.z, z1.w};
                                    const uint32_t kb = keep_bits_acc(p, pb.bn_index, seed_mix, drop_thr, ch, gr, n0);
#pragma unroll
                                    for (int j = 0; j < 8; ++j) {
                                        const float zh = (z[j] - mean[j]) * invstd[j];
                                        const float y = fmaf(zh, gam[j], bet[j]);
                                        float gy = y > 0.f ? G[j] : 0.f;
                                        gy = (kb >> j) & 1u ? gy * inv_keep : 0.f;
                                        s3[j] += gy;
                                        s4[j] = fmaf(gy, zh, s4[j]);
                                    }
                                } else {
#pragma unroll
                                    for (int j = 0; j < 8; ++j) {
                                        acc[i][j] = G[j];  // no BatchNorm below (LocoModel.w2): gz == G, chained as the next A tile
                                        s3[j] += G[j];
                                    }
                                    float* dz = Gzq + gr * L + n0;
                                    *reinterpret_cast<float4*>(dz) = make_float4(G[0], G[1], G[2], G[3]);
                                    *reinterpret_cast<float4*>(dz + 64) = make_float4(G[4], G[5], G[6], G[7]);
                                }
                            } else if (!pb.has_bn) {
#pragma unroll
                                for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
                            }
                        }
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            s3[j] += __shfl_xor_sync(0xffffffffu, s3[j], 16);
                            s4[j] += __shfl_xor_sync(0xffffffffu, s4[j], 16);
                            if (g == 0) {
                                if (pb.has_bn) {
                                    atomicAdd(&pb.stat[2 * L + col_of(n0, j)], (double)s3[j]);
                                    atomicAdd(&pb.stat[3 * L + col_of(n0, j)], (double)s4[j]);
                                } else {
                                    atomicAdd(pb.db + col_of(n0, j), s3[j]);
                                }
                            }
                        }
                        if (!pb.has_bn) {
                            if (tile == p.n_tiles - 1)
                                for (int idx = lane; idx < (p.n_rows_pad - p.n_rows) * 128; idx += 32)
                                    pb.Gz[(size_t)p.n_rows * L + (size_t)(idx / 128) * L + warp * 128 + idx % 128] = 0.f;
                            csync();  // every warp has finished reading `act`
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                float* dst = act + (size_t)col_of(n0, j) * MP + g * 16;
#pragma unroll
                                for (int v = 0; v < 4; ++v) {
                                    float4 t;
                                    t.x = (v * 4 + 0 < TM) ? acc[v * 4 + 0 < TM ? v * 4 + 0 : 0][j] : 0.f;
                                    t.y = (v * 4 + 1 < TM) ? acc[v * 4 + 1 < TM ? v * 4 + 1 : 0][j] : 0.f;
                                    t.z = (v * 4 + 2 < TM) ? acc[v * 4 + 2 < TM ? v * 4 + 2 : 0][j] : 0.f;
                                    t.w = (v * 4 + 3 < TM) ? acc[v * 4 + 3 < TM ? v * 4 + 3 : 0][j] : 0.f;
                                    *reinterpret_cast<float4*>(dst + v * 4) = t;
                                }
                            }
                        }
                    } else if (!pb.has_bn) {
                        csync();
                    }
                    csync();
                }
                mark(p, ph, 2, tid);
            }
        } else if (type == PH_DW) {
            // ============================================================================ weight gradients
            // dW_i[n][k] = sum_b Gz_i[b][n] * A_{i-1}[b][k]: 32 n-rows x L columns per item, reduction streamed over b
            const int n_items = (p.n_blocks - 1) * (L / 32);
            const int nchunks = p.n_rows_pad / KC;
            const long long total = (long long)n_items * nchunks;
            const long long u0 = total * blockIdx.x / gridDim.x, u1 = total * (blockIdx.x + 1) / gridDim.x;
            for (long long u = u0; u < u1;) {
                const int item = (int)(u / nchunks), c0 = (int)(u % nchunks);
                const int c1 = (int)min((long long)nchunks, c0 + (u1 - u));
                const int b_i = 1 + item / (L / 32), nb = (item % (L / 32)) * 32;
                const bool whole = c0 == 0 && c1 == nchunks;  // this CTA owns the full reduction: plain stores
                if (gemm_warp) {
                    unsigned long long acc2[8][8];
                    acc_zero<16>(acc2);
                    tile_gemm<16>(acc2, c1 - c0, [&](int, unsigned stage) { return act + (size_t)stage * KC * 32; }, ring, full,
                                  empty, rs, n0, g, lane, L, p.err_flag);
                    float* dst = p.blk[b_i].dW + (size_t)(nb + g * 16) * L + n0;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        float lo[8], hi[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) unpack2(acc2[i][j], lo[j], hi[j]);
                        float* d0 = dst + (size_t)(2 * i) * L;
                        float* d1 = dst + (size_t)(2 * i + 1) * L;
                        if (whole) {
                            *reinterpret_cast<float4*>(d0) = make_float4(lo[0], lo[1], lo[2], lo[3]);
                            *reinterpret_cast<float4*>(d0 + 64) = make_float4(lo[4], lo[5], lo[6], lo[7]);
                            *reinterpret_cast<float4*>(d1) = make_float4(hi[0], hi[1], hi[2], hi[3]);
                            *reinterpret_cast<float4*>(d1 + 64) = make_float4(hi[4], hi[5], hi[6], hi[7]);
                        } else {
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                atomicAdd(d0 + (j & 3) + (j >> 2) * 64, lo[j]);
                                atomicAdd(d1 + (j & 3) + (j >> 2) * 64, hi[j]);
                            }
                        }
                    }
                }
                u += c1 - c0;
            }
        }
        end_phase(ph);
    }
    // ---- finalise: per-task loss means (losses.py:139 torch.mean)
    if (blockIdx.x == 0 && p.labels != nullptr && tid < p.n_tasks) p.loss_vals[tid] = (float)(p.loss_acc[tid] / (double)p.n_rows);
}

}  // namespace mlb

// ================================================================================================ host side
using namespace mlb;

struct mlb_train {
    int device, n_sms, max_rows, rows_pad, in_size, L, n_blocks;
    float *Wt[MLB_MAX_BLOCKS], *Z[MLB_MAX_BLOCKS], *A[MLB_MAX_BLOCKS], *G[MLB_MAX_BLOCKS], *Gz[MLB_MAX_BLOCKS];
    double* stat[MLB_MAX_BLOCKS];
    float* g_out;
    double* loss_acc;
    float4* ptab;
    unsigned* bar;
    int* err;
    unsigned long long* phase_ns;
    int last_n_phases;
    int last_phase_type[MAX_PHASES], last_phase_blk[MAX_PHASES];
};

static size_t train_smem_bytes(int L) {
    size_t actf = (size_t)L * MP > 8 * 32 * 33 ? (size_t)L * MP : 8 * 32 * 33;
    size_t fl = actf + MP * OUT_LD + (size_t)NSTAGE * KC * L;
    return fl * sizeof(float) + 2 * NSTAGE * sizeof(uint64_t) + 16;
}

extern "C" int mlb_train_create(int device, int max_rows, int input_size, int linear_size, int n_blocks, mlb_train_handle* out) {
    if (!out || max_rows < 2 || n_blocks < 2 || n_blocks > MLB_MAX_BLOCKS) return mlb_fail("mlb_train_create: bad argument");
    if (linear_size < 128 || linear_size > 1024 || linear_size % 128) return mlb_fail("mlb_train_create: linear_size must be a multiple of 128 in [128,1024]");
    if (input_size < 1 || input_size > 68) return mlb_fail("mlb_train_create: input_size must be in [1,68]");
    MLB_CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    MLB_CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return mlb_fail("mlb_train_create: built for sm_100a (B200) only");
    mlb_train* t = new mlb_train();
    memset(t, 0, sizeof(*t));
    t->device = device, t->n_sms = prop.multiProcessorCount, t->max_rows = max_rows, t->in_size = input_size;
    t->L = linear_size, t->n_blocks = n_blocks;
    t->rows_pad = ((max_rows + KC - 1) / KC) * KC;
    const size_t act_bytes = (size_t)t->rows_pad * linear_size * sizeof(float);
    for (int i = 0; i < n_blocks; ++i) {
        const int kpad = i == 0 ? ((input_size + KC - 1) / KC) * KC : linear_size;
        MLB_CU(cudaMalloc(&t->Wt[i], (size_t)kpad * linear_size * sizeof(float)));
        MLB_CU(cudaMalloc(&t->Z[i], act_bytes));
        MLB_CU(cudaMalloc(&t->A[i], act_bytes));
        MLB_CU(cudaMalloc(&t->G[i], act_bytes));
        MLB_CU(cudaMalloc(&t->Gz[i], act_bytes));
        MLB_CU(cudaMemset(t->Z[i], 0, act_bytes));
        MLB_CU(cudaMemset(t->A[i], 0, act_bytes));
        MLB_CU(cudaMemset(t->G[i], 0, act_bytes));
        MLB_CU(cudaMemset(t->Gz[i], 0, act_bytes));
        MLB_CU(cudaMalloc(&t->stat[i], 4 * linear_size * sizeof(double)));
        MLB_CU(cudaMemset(t->stat[i], 0, 4 * linear_size * sizeof(double)));
    }
    MLB_CU(cudaMalloc(&t->g_out, (size_t)t->rows_pad * OUT_LD * sizeof(float)));
    MLB_CU(cudaMemset(t->g_out, 0, (size_t)t->rows_pad * OUT_LD * sizeof(float)));
    MLB_CU(cudaMalloc(&t->loss_acc, 8 * sizeof(double)));
    MLB_CU(cudaMalloc(&t->ptab, (size_t)t->n_sms * linear_size * 2 * sizeof(float4)));
    MLB_CU(cudaMalloc(&t->bar, sizeof(unsigned)));
    MLB_CU(cudaMalloc(&t->err, sizeof(int)));
    MLB_CU(cudaMemset(t->err, 0, sizeof(int)));
    MLB_CU(cudaMalloc(&t->phase_ns, (MAX_PHASES + 1 + MAX_PHASES * 24) * sizeof(unsigned long long)));
    MLB_CU(cudaMemset(t->phase_ns, 0, (MAX_PHASES + 1 + MAX_PHASES * 24) * sizeof(unsigned long long)));
    *out = t;
    return 0;
}

extern "C" void mlb_train_destroy(mlb_train_handle t) {
    if (!t) return;
    cudaSetDevice(t->device);
    for (int i = 0; i < t->n_blocks; ++i) {
        cudaFree(t->Wt[i]), cudaFree(t->Z[i]), cudaFree(t->A[i]), cudaFree(t->G[i]), cudaFree(t->Gz[i]), cudaFree(t->stat[i]);
    }
    cudaFree(t->g_out), cudaFree(t->loss_acc), cudaFree(t->ptab), cudaFree(t->bar), cudaFree(t->err), cudaFree(t->phase_ns);
    delete t;
}

template <int TM>
static cudaError_t launch_train(const TrainParams& p, int grid, size_t smem, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(loco_train_kernel<TM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    void* args[] = {(void*)&p};
    return cudaLaunchCooperativeKernel((void*)loco_train_kernel<TM>, dim3(grid), dim3(MAX_THREADS), args, smem, st);
}

static int pick_tm(int n_rows, int n_ctas) {
    int best = 16;
    long best_cost = -1;
    for (int tm = 16; tm >= 8; tm -= 2) {
        const long tiles = (n_rows + 2 * tm - 1) / (2 * tm);
        const long cost = ((tiles + n_ctas - 1) / n_ctas) * tm;
        if (best_cost < 0 || cost < best_cost) best_cost = cost, best = tm;
    }
    return best;
}

// mode: 0 forward, 1 backward, 2 fused step
static int train_launch(mlb_train_handle t, const mlb_train_args* a, const mlb_train_block* blocks, void* stream, int mode) {
    if (!t || !a || !blocks) return mlb_fail("mlb_train: null argument");
    if (a->n_rows < 2 || a->n_rows > t->max_rows) return mlb_fail("mlb_train: n_rows must be in [2, max_rows] (BatchNorm needs > 1 row)");
    if (a->linear_size != t->L || a->n_blocks != t->n_blocks || a->input_size != t->in_size) return mlb_fail("mlb_train: shape differs from mlb_train_create");
    if (a->output_size < 2 || a->output_size > OUT_LD) return mlb_fail("mlb_train: bad output_size");
    if (a->aux_block < 0 || a->aux_block >= a->n_blocks - 1) return mlb_fail("mlb_train: bad aux_block");
    if (!a->x || !a->out || !a->W_aux || !a->b_aux || !a->W_fin || !a->b_fin) return mlb_fail("mlb_train: missing tensor");
    if (mode >= 1 && (!a->dW_aux || !a->db_aux || !a->dW_fin || !a->db_fin)) return mlb_fail("mlb_train: missing head gradient buffers");
    if (mode == 1 && !a->g_out) return mlb_fail("mlb_train_backward: g_out required");
    if (mode == 2 && (!a->labels || !a->loss_vals || a->n_tasks < 1 || a->n_tasks > 8)) return mlb_fail("mlb_train_step: labels / loss_vals / tasks required");
    if (a->p_dropout < 0.f || a->p_dropout >= 1.f) return mlb_fail("mlb_train: bad p_dropout");
    MLB_CU(cudaSetDevice(t->device));
    cudaStream_t st = (cudaStream_t)stream;

    TrainParams p;
    memset(&p, 0, sizeof(p));
    int bn_count = 0;
    for (int i = 0; i < a->n_blocks; ++i) {
        const mlb_train_block& s = blocks[i];
        TBlk& b = p.blk[i];
        if (s.K != (i == 0 ? a->input_size : a->linear_size)) return mlb_fail("mlb_train: block K mismatch");
        if (!s.W || !s.b || (s.has_bn && (!s.gamma || !s.beta))) return mlb_fail("mlb_train: missing block parameter");
        if (mode >= 1 && (!s.dW || !s.db || (s.has_bn && (!s.dgamma || !s.dbeta)))) return mlb_fail("mlb_train: missing block gradient buffer");
        if (i == 0 && !s.has_bn) return mlb_fail("mlb_train: the first block must have BatchNorm");
        if (s.res_src >= i) return mlb_fail("mlb_train: bad res_src");
        b.K = s.K;
        b.Kpad = ((s.K + KC - 1) / KC) * KC;
        b.has_bn = s.has_bn;
        b.res_src = s.has_bn ? s.res_src : -1;
        b.skip_to = -1;
        b.bn_index = s.has_bn ? bn_count++ : -1;
        b.W = s.W, b.b = s.b, b.gamma = s.gamma, b.beta = s.beta;
        b.rmean = s.running_mean, b.rvar = s.running_var;
        b.dW = s.dW, b.db = s.db, b.dgamma = s.dgamma, b.dbeta = s.dbeta;
        b.Wt = t->Wt[i], b.Z = t->Z[i], b.Aout = t->A[i], b.G = t->G[i], b.Gz = t->Gz[i], b.stat = t->stat[i];
    }
    for (int i = 0; i < a->n_blocks; ++i)
        if (p.blk[i].res_src >= 0) p.blk[p.blk[i].res_src].skip_to = i;
    if (!p.blk[a->n_blocks - 1].has_bn) return mlb_fail("mlb_train: the last block must have BatchNorm (LocoModel.w3)");
    if (p.blk[a->aux_block].has_bn) return mlb_fail("mlb_train: aux_block must be the BatchNorm-free block (LocoModel.w2)");
    p.n_blocks = a->n_blocks, p.aux_block = a->aux_block, p.L = a->linear_size, p.in_size = a->input_size;
    p.out_size = a->output_size, p.n_rows = a->n_rows;
    p.n_rows_pad = ((a->n_rows + KC - 1) / KC) * KC;
    int tm = a->rows_per_group ? a->rows_per_group : pick_tm(a->n_rows, t->n_sms);
    if (tm < 8 || tm > 16 || (tm & 1)) return mlb_fail("mlb_train: rows_per_group must be 0 or one of 8,10,12,14,16");
    p.n_tiles = (a->n_rows + 2 * tm - 1) / (2 * tm);
    p.p_drop = a->p_dropout, p.eps = a->bn_eps > 0.f ? a->bn_eps : 1e-5f, p.momentum = a->bn_momentum;
    p.update_running = a->update_running_stats;
    p.seed = a->drop_seed, p.drop_mask = a->drop_mask;
    p.x = a->x, p.out = a->out, p.g_out_in = a->g_out, p.g_out = t->g_out;
    p.W_aux = a->W_aux, p.b_aux = a->b_aux, p.W_fin = a->W_fin, p.b_fin = a->b_fin;
    p.dW_aux = a->dW_aux, p.db_aux = a->db_aux, p.dW_fin = a->dW_fin, p.db_fin = a->db_fin;
    if (mode == 2) {
        p.labels = a->labels, p.label_ld = a->label_ld, p.n_tasks = a->n_tasks;
        for (int i = 0; i < a->n_tasks; ++i) {
            if (a->tasks[i] < 0 || a->tasks[i] > MLB_TASK_AUX) return mlb_fail("mlb_train_step: bad task id");
            if (a->tasks[i] == MLB_TASK_AUX && (a->output_size != 10 || a->label_ld < 11)) return mlb_fail("mlb_train_step: aux task needs 10 outputs / 11 label columns");
            p.tasks[i] = a->tasks[i], p.task_scale[i] = a->task_scale[i];
        }
        p.loss_vals = a->loss_vals;
        p.task_scale_dev = a->task_scale_dev;
    }
    p.loss_acc = t->loss_acc, p.ptab = t->ptab, p.bar_counter = t->bar, p.err_flag = t->err;
    p.phase_ns = t->phase_ns;

    int np = 0;
    auto add = [&](int type, int blk) { p.phase_type[np] = type, p.phase_blk[np] = blk, np++; };
    if (mode == 0 || mode == 2) {
        add(PH_PACK, 0);
        for (int i = 0; i < a->n_blocks; ++i) add(PH_FWD, i);
        add(PH_FWD_FINAL, 0);
    }
    if (mode == 1 || mode == 2) {
        add(PH_BWD_INIT, 0);
        add(PH_BWD_HEAD, 0);
        for (int i = a->n_blocks - 1; i >= 0; --i)
            if (p.blk[i].has_bn) add(PH_BWD, i);
        add(PH_DW, 0);
    }
    p.n_phases = np;
    if (np > MAX_PHASES) return mlb_fail("mlb_train: too many phases");
    t->last_n_phases = np;
    memcpy(t->last_phase_type, p.phase_type, sizeof(int) * np);
    memcpy(t->last_phase_blk, p.phase_blk, sizeof(int) * np);

    MLB_CU(cudaMemsetAsync(t->bar, 0, sizeof(unsigned), st));
    const size_t smem = train_smem_bytes(a->linear_size);
    const int grid = t->n_sms;
    cudaError_t e;
    switch (tm) {
        case 8: e = launch_train<8>(p, grid, smem, st); break;
        case 10: e = launch_train<10>(p, grid, smem, st); break;
        case 12: e = launch_train<12>(p, grid, smem, st); break;
        case 14: e = launch_train<14>(p, grid, smem, st); break;
        default: e = launch_train<16>(p, grid, smem, st); break;
    }
    if (e != cudaSuccess) return mlb_fail(std::string("loco_train_kernel launch: ") + cudaGetErrorString(e));
    mlb_count_launch();
    return 0;
}

// per-phase wall time (ns) of the most recent launch on this handle: out_ns[i] = duration of phase i, types/blks describe it
extern "C" int mlb_train_phase_times(mlb_train_handle t, int max_n, double* out_ns, int* types, int* blks) {
    if (!t || !out_ns) return mlb_fail("mlb_train_phase_times: bad argument");
    MLB_CU(cudaSetDevice(t->device));
    MLB_CU(cudaDeviceSynchronize());
    unsigned long long ts[MAX_PHASES + 1];
    MLB_CU(cudaMemcpy(ts, t->phase_ns, sizeof(ts), cudaMemcpyDeviceToHost));
    int n = t->last_n_phases < max_n ? t->last_n_phases : max_n;
    for (int i = 0; i < n; ++i) {
        out_ns[i] = (double)(ts[i + 1] - ts[i]);
        if (types) types[i] = t->last_phase_type[i];
        if (blks) blks[i] = t->last_phase_blk[i];
    }
    return n;
}

// profiling aid: out_ns[(ph*3 + s)*8 + k] = time since the start of phase ph at which CTA s (0: first, 1: middle, 2: last
// active) passed point k (0: input tile ready, 1: GEMM done, 2: epilogue done, 3: left the grid barrier, 4 batch statistics loaded, 5 tile rows finished, 6-7 spare); 0 where unset.
extern "C" int mlb_train_subphase_times(mlb_train_handle t, int max_n, double* out_ns) {
    if (!t || !out_ns) return mlb_fail("mlb_train_subphase_times: bad argument");
    MLB_CU(cudaSetDevice(t->device));
    MLB_CU(cudaDeviceSynchronize());
    static unsigned long long ts[MAX_PHASES + 1 + MAX_PHASES * 24];
    MLB_CU(cudaMemcpy(ts, t->phase_ns, sizeof(ts), cudaMemcpyDeviceToHost));
    int n = t->last_n_phases < max_n ? t->last_n_phases : max_n;
    for (int i = 0; i < n; ++i)
        for (int q = 0; q < 24; ++q) {
            const unsigned long long v = ts[MAX_PHASES + 1 + i * 24 + q];
            out_ns[i * 24 + q] = v > ts[i] ? (double)(v - ts[i]) : 0.0;
        }
    return n;
}

extern "C" int mlb_train_forward(mlb_train_handle h, const mlb_train_args* a, const mlb_train_block* blocks, void* stream) {
    return train_launch(h, a, blocks, stream, 0);
}
extern "C" int mlb_train_backward(mlb_train_handle h, const mlb_train_args* a, const mlb_train_block* blocks, void* stream) {
    return train_launch(h, a, blocks, stream, 1);
}
extern "C" int mlb_train_step(mlb_train_handle h, const mlb_train_args* a, const mlb_train_block* blocks, void* stream) {
    return train_launch(h, a, blocks, stream, 2);
}
