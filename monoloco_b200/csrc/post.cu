// monoloco_b200 -- the steps right after the network, on the device (SURVEY.md 8(f) row N3 + row A7):
//
//   * monstereo arg-max filter          monoloco/network/process.py:307-327  (cluster_outputs / filter_outputs)
//   * Loco.post_process over MANY images monoloco/network/net.py:164-248     (bbox-centre ray, xyz_from_distance,
//                                        confidence, IoU matching utils/iou.py:6-29,44-64, left-right reorder :87-101)
//   * KITTI label rows                   monoloco/eval/generate_kitti.py:202-253 (save_txts: the 15 numbers of every line)
//
// All of it is small integer / index work plus a few fp64 scalar expressions (the reference evaluates IoU and the
// confidence in Python floats = fp64, so the device does the same: the match indices and the order are bit-exact).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/monoloco_b200.h"
#include "host_error.h"

namespace mlb {

// ------------------------------------------------------------------------------------------------
// monstereo arg-max filter: one warp per left pose.
//   pass 1: cnt[l] = #{r : aux[l][r] >= max_r aux[l][r]}   (0 if any NaN: torch.max propagates NaN -> mask all False)
//   pass 2: offset = sum(cnt[0..l)), ordered compaction of the kept rows (row-major: ties keep their order)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_max(float v) {
    for (int s = 16; s > 0; s >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, s));
    return v;
}

__global__ void stereo_count_kernel(const float* __restrict__ raw, int n_left, int n_right, int out_size,
                                    int32_t* __restrict__ cnt, float* __restrict__ best_out) {
    const int l = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (l >= n_left) return;
    const float* v = raw + (size_t)l * n_right * out_size + (out_size - 1);
    float best = -INFINITY;
    bool nan = false;
    for (int r = lane; r < n_right; r += 32) {
        const float x = v[(size_t)r * out_size];
        nan |= (x != x);
        best = fmaxf(best, x);  // fmaxf ignores NaN; NaN rows are handled through `nan`
    }
    best = warp_max(best);
    nan = __any_sync(0xffffffffu, nan);
    int c = 0;
    if (!nan)
        for (int r = lane; r < n_right; r += 32) c += v[(size_t)r * out_size] >= best;
    for (int s = 16; s > 0; s >>= 1) c += __shfl_xor_sync(0xffffffffu, c, s);
    if (lane == 0) cnt[l] = c, best_out[l] = best;
}

__global__ void stereo_scatter_kernel(const float* __restrict__ raw, const float* __restrict__ dec, const float* __restrict__ xyzc,
                                      int n_left, int n_right, int out_size, const int32_t* __restrict__ cnt,
                                      const float* __restrict__ best_in, float* __restrict__ sel_raw, float* __restrict__ sel_dec,
                                      float* __restrict__ sel_xyzc, int32_t* __restrict__ sel_idx, int32_t* __restrict__ n_sel) {
    const int l = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (l >= n_left) return;
    int off = 0;
    for (int k = lane; k < l; k += 32) off += cnt[k];
    for (int s = 16; s > 0; s >>= 1) off += __shfl_xor_sync(0xffffffffu, off, s);
    const int mine = cnt[l];
    if (l == n_left - 1 && lane == 0) *n_sel = off + mine;
    if (mine == 0) return;
    const float best = best_in[l];
    const float* v = raw + (size_t)l * n_right * out_size + (out_size - 1);
    for (int r0 = 0; r0 < n_right; r0 += 32) {
        const int r = r0 + lane;
        const bool keep = r < n_right && v[(size_t)r * out_size] >= best;
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (keep) {
            const int pos = off + __popc(m & ((1u << lane) - 1u));
            const size_t src = (size_t)l * n_right + r;
            sel_idx[pos] = (int32_t)src;
            for (int k = 0; k < out_size; ++k) sel_raw[(size_t)pos * out_size + k] = raw[src * out_size + k];
            if (dec != nullptr && sel_dec != nullptr)
                for (int k = 0; k < 8; ++k) sel_dec[(size_t)pos * 8 + k] = dec[src * 8 + k];
            if (xyzc != nullptr && sel_xyzc != nullptr)
                for (int k = 0; k < 4; ++k) sel_xyzc[(size_t)pos * 4 + k] = xyzc[src * 4 + k];
        }
        off += __popc(m);
    }
}

// ------------------------------------------------------------------------------------------------
// Loco.post_process for a batch of images: one CTA per image.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double iou64(const double* a, const double* b) {  // utils/iou.py:6-29 in fp64, same op order
    const double xi1 = fmax(a[0], b[0]), yi1 = fmax(a[1], b[1]), xi2 = fmin(a[2], b[2]), yi2 = fmin(a[3], b[3]);
    const double inter = __dmul_rn(fmax(__dsub_rn(xi2, xi1), 0.0), fmax(__dsub_rn(yi2, yi1), 0.0));
    const double a1 = __dmul_rn(__dsub_rn(a[2], a[0]), __dsub_rn(a[3], a[1]));
    const double a2 = __dmul_rn(__dsub_rn(b[2], b[0]), __dsub_rn(b[3], b[1]));
    return __ddiv_rn(inter, __dsub_rn(__dadd_rn(a1, a2), inter));
}

__global__ void __launch_bounds__(128) post_process_kernel(const mlb_post_args a) {
    extern __shared__ int sm_post[];
    const int img = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const int d0 = a.det_off[img], m = a.det_off[img + 1] - d0;
    const int g0 = a.gt_off ? a.gt_off[img] : 0, g = a.gt_off ? a.gt_off[img + 1] - g0 : 0;
    int* sorted = sm_post;                 // [max_det] detection indices by ascending confidence (stable)
    int* match = sorted + a.max_det;       // [max_det] matched gt (image-local) or -1
    int* seq = match + a.max_det;          // [max_det] position in the match list
    int* used = seq + a.max_det;           // [max_gt]
    __shared__ int s_nmatch;

    const float* kinv = a.kinv + (size_t)img * 9;
    // ---- per detection: key points, bbox-centre ray, xyz_from_distance, confidence (net.py:192-215)
    for (int j = tid; j < m; j += nt) {
        const float* kp = a.kps + (size_t)(d0 + j) * 51;
        float umin = kp[0], umax = umin, vmin = kp[17], vmax = vmin;
        for (int t = 1; t < 17; ++t) {
            umin = fminf(umin, kp[t]), umax = fmaxf(umax, kp[t]);
            vmin = fminf(vmin, kp[17 + t]), vmax = fmaxf(vmax, kp[17 + t]);
        }
        const float uc = __fadd_rn(__fdiv_rn(__fsub_rn(umax, umin), 2.f), umin);  // camera.py:82-86
        const float vc = __fadd_rn(__fdiv_rn(__fsub_rn(vmax, vmin), 2.f), vmin);
        float uh = 0.f, vh = 0.f;
        for (int t = 0; t < 5; ++t) uh = __fadd_rn(uh, kp[t]), vh = __fadd_rn(vh, kp[17 + t]);
        uh = __fdiv_rn(uh, 5.f), vh = __fdiv_rn(vh, 5.f);                          // camera.py:95-96 mean over 0:5
        const float us = __fdiv_rn(__fadd_rn(kp[5], kp[6]), 2.f), vs = __fdiv_rn(__fadd_rn(kp[22], kp[23]), 2.f);
        int32_t* uv = a.uv + (size_t)(d0 + j) * 6;   // python round() = round-half-even on the fp32 value
        uv[0] = (int32_t)rint((double)uc), uv[1] = (int32_t)rint((double)vc);
        uv[2] = (int32_t)rint((double)us), uv[3] = (int32_t)rint((double)vs);
        uv[4] = (int32_t)rint((double)uh), uv[5] = (int32_t)rint((double)vh);
        const float cx = uc * kinv[0] + vc * kinv[1] + kinv[2];  // pixel_to_camera(uv_centers, kk, 1), camera.py:23-27
        const float cy = uc * kinv[3] + vc * kinv[4] + kinv[5];
        const float cz = uc * kinv[6] + vc * kinv[7] + kinv[8];
        const float den = sqrtf(__fadd_rn(__fadd_rn(1.f, __fmul_rn(cx, cx)), __fmul_rn(cy, cy)));  // camera.py:177
        const float dd = a.dec[(size_t)(d0 + j) * 8 + 3], bi = a.dec[(size_t)(d0 + j) * 8 + 4];
        const float px = __fdiv_rn(__fmul_rn(cx, dd), den), py = __fdiv_rn(__fmul_rn(cy, dd), den),
                    pz = __fdiv_rn(__fmul_rn(cz, dd), den);
        float* xyz = a.xyz + (size_t)(d0 + j) * 3;
        xyz[0] = px, xyz[1] = py, xyz[2] = pz;
        float* ray = a.ray + (size_t)(d0 + j) * 4;
        ray[0] = cx, ray[1] = cy, ray[2] = cz, ray[3] = den;
        const double dist = sqrt(__dadd_rn(__dadd_rn(__dmul_rn((double)px, (double)px), __dmul_rn((double)py, (double)py)),
                                           __dmul_rn((double)pz, (double)pz)));     // net.py:214
        a.conf[d0 + j] = __ddiv_rn(__dmul_rn(0.035, a.boxes[(size_t)(d0 + j) * 5 + 4]), __ddiv_rn((double)bi, dist));
        match[j] = -1, seq[j] = 0;
    }
    for (int k = tid; k < g; k += nt) used[k] = 0;
    if (tid == 0) s_nmatch = 0;
    __syncthreads();

    // ---- greedy IoU matching in decreasing box confidence (utils/iou.py:44-64)
    if (g > 0 && m > 0) {
        for (int j = tid; j < m; j += nt) {   // stable rank sort by confidence (np.argsort on a handful of boxes)
            const double cj = a.boxes[(size_t)(d0 + j) * 5 + 4];
            int rank = 0;
            for (int k = 0; k < m; ++k) {
                const double ck = a.boxes[(size_t)(d0 + k) * 5 + 4];
                rank += (ck < cj) || (ck == cj && k < j);
            }
            sorted[rank] = j;
        }
        __syncthreads();
        if (tid < 32) {
            int nmatch = 0;
            for (int s = m - 1; s >= 0; --s) {
                const int j = sorted[s];
                const double* bj = a.boxes + (size_t)(d0 + j) * 5;
                double best = -1.0;
                int bidx = 0x7fffffff;
                for (int k = tid; k < g; k += 32) {
                    const double v = iou64(bj, a.gt_boxes + (size_t)(g0 + k) * 4);
                    if (v > best) best = v, bidx = k;  // first maximum within this lane's subsequence
                }
                for (int sh = 16; sh > 0; sh >>= 1) {  // np.argmax: the first index among equal maxima
                    const double ov = __shfl_xor_sync(0xffffffffu, best, sh);
                    const int oi = __shfl_xor_sync(0xffffffffu, bidx, sh);
                    if (ov > best || (ov == best && oi < bidx)) best = ov, bidx = oi;
                }
                if (best >= a.iou_min && !used[bidx]) {
                    __syncwarp();
                    if (tid == 0) used[bidx] = 1, match[j] = bidx, seq[j] = nmatch;
                    nmatch++;
                }
                __syncwarp();
            }
            if (tid == 0) s_nmatch = nmatch;
        }
        __syncthreads();
    }
    const int nmatch = s_nmatch;
    if (tid == 0) a.n_match[img] = nmatch;

    // ---- output order (net.py:187-191): matches first (left to right by box x1 when reorder, utils/iou.py:87-101, else
    // in match order), then the unmatched detections by index; xyz_real of the matches (net.py:242-247)
    for (int j = tid; j < m; j += nt) {
        int pos;
        if (match[j] >= 0) {
            if (a.reorder) {
                const double xj = a.boxes[(size_t)(d0 + j) * 5];
                pos = 0;
                for (int k = 0; k < m; ++k) {
                    if (match[k] < 0) continue;
                    const double xk = a.boxes[(size_t)(d0 + k) * 5];
                    pos += (xk < xj) || (xk == xj && k < j);
                }
            } else {
                pos = seq[j];
            }
            const float dr = (float)a.gt_d[g0 + match[j]];  // torch.tensor(python float) -> fp32 (camera.py:168-169)
            const float* ray = a.ray + (size_t)(d0 + j) * 4;
            float* xr = a.xyz_real + (size_t)(d0 + j) * 3;
            xr[0] = __fdiv_rn(__fmul_rn(ray[0], dr), ray[3]);
            xr[1] = __fdiv_rn(__fmul_rn(ray[1], dr), ray[3]);
            xr[2] = __fdiv_rn(__fmul_rn(ray[2], dr), ray[3]);
        } else {
            pos = nmatch;
            for (int k = 0; k < j; ++k) pos += match[k] < 0;
        }
        a.order[d0 + pos] = j;
        a.match_gt[d0 + j] = match[j];
    }
}

// ------------------------------------------------------------------------------------------------
// KITTI rows (generate_kitti.py:202-253, nets monoloco_pp / monstereo): per detection the 15 numbers of its txt line
//   [alpha, x1, y1, x2, y2, h, w, l, x, y, z, ry, conf, bi, epi]     (all fp64: "%f" of Python floats)
// ------------------------------------------------------------------------------------------------
__global__ void kitti_rows_kernel(int n, int out_size, double conf_scale, const double* __restrict__ boxes,
                                  const float* __restrict__ raw, const float* __restrict__ dec, const float* __restrict__ epi,
                                  double* __restrict__ rows) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* d = dec + (size_t)i * 8;
    const float* o = raw + (size_t)i * out_size;
    const double xx = d[0], yy = d[1], zz = d[2], bi = d[4];
    double* r = rows + (size_t)i * 15;
    r[0] = d[5];                                   // alpha = yaws[0]
    for (int k = 0; k < 4; ++k) r[1 + k] = boxes[(size_t)i * 5 + k];
    r[5] = o[4], r[6] = o[5], r[7] = o[6];         // h, w, l
    r[8] = xx, r[9] = yy, r[10] = zz;
    r[11] = d[6];                                  // ry = yaws[1]
    const double dist = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(xx, xx), __dmul_rn(yy, yy)), __dmul_rn(zz, zz)));
    r[12] = __ddiv_rn(__dmul_rn(conf_scale, boxes[(size_t)i * 5 + 4]), __ddiv_rn(bi, dist));
    r[13] = bi;
    r[14] = epi ? (double)epi[i] : 0.0;
}

}  // namespace mlb

using namespace mlb;

extern "C" int mlb_stereo_filter(const float* raw, const float* dec, const float* xyzc, int n_left, int n_right, int out_size,
                                 float* sel_raw, float* sel_dec, float* sel_xyzc, int32_t* sel_idx, int32_t* n_sel_dev,
                                 int32_t* cnt_scratch, float* best_scratch, void* stream) {
    if (!raw || !sel_raw || !sel_idx || !n_sel_dev || !cnt_scratch || !best_scratch || n_left < 1 || n_right < 1 || out_size < 1)
        return mlb_fail("mlb_stereo_filter: bad argument");
    const int wpb = 4, grid = (n_left + wpb - 1) / wpb;
    cudaStream_t st = (cudaStream_t)stream;
    stereo_count_kernel<<<grid, wpb * 32, 0, st>>>(raw, n_left, n_right, out_size, cnt_scratch, best_scratch);
    stereo_scatter_kernel<<<grid, wpb * 32, 0, st>>>(raw, dec, xyzc, n_left, n_right, out_size, cnt_scratch, best_scratch, sel_raw,
                                                     sel_dec, sel_xyzc, sel_idx, n_sel_dev);
    MLB_CU(cudaGetLastError());
    mlb_count_launch();
    mlb_count_launch();
    return 0;
}

extern "C" int mlb_post_process(const mlb_post_args* a, void* stream) {
    if (!a) return mlb_fail("mlb_post_process: null argument");
    if (a->n_img < 0 || a->max_det < 0 || a->max_gt < 0) return mlb_fail("mlb_post_process: negative size");
    if (a->n_img == 0) return 0;
    if (!a->det_off || !a->boxes || !a->kps || !a->kinv || !a->dec || !a->xyz || !a->ray || !a->conf || !a->uv || !a->match_gt ||
        !a->order || !a->n_match || !a->xyz_real)
        return mlb_fail("mlb_post_process: null pointer");
    if (a->gt_off && (!a->gt_boxes || !a->gt_d)) return mlb_fail("mlb_post_process: gt_off without gt_boxes / gt_d");
    const size_t smem = ((size_t)3 * a->max_det + (size_t)a->max_gt + 4) * sizeof(int);
    if (smem > 200 * 1024) return mlb_fail("mlb_post_process: too many detections / ground truths in one image");
    if (smem > 48 * 1024) MLB_CU(cudaFuncSetAttribute(post_process_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    post_process_kernel<<<a->n_img, 128, smem, (cudaStream_t)stream>>>(*a);
    MLB_CU(cudaGetLastError());
    mlb_count_launch();
    return 0;
}

extern "C" int mlb_kitti_rows(int n, int out_size, double conf_scale, const double* boxes, const float* raw, const float* dec,
                              const float* epi, double* rows, void* stream) {
    if (n == 0) return 0;
    if (n < 0 || out_size < 7 || !boxes || !raw || !dec || !rows) return mlb_fail("mlb_kitti_rows: bad argument");
    kitti_rows_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(n, out_size, conf_scale, boxes, raw, dec, epi, rows);
    MLB_CU(cudaGetLastError());
    mlb_count_launch();
    return 0;
}
