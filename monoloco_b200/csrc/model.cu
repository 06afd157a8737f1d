// The inference handle of the C ABI: mlb_create / mlb_update_weights / mlb_destroy, the per-device kernel timing that
// drives the kernel choice (calibrate), mlb_forward / mlb_forward_host and the introspection getters.  The kernels and
// their host-side state live with their families (fwd_family.cuh); plan_forward (fwd_plan.h) picks one per call.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>

#include "fwd_family.cuh"

namespace mlb {
// a rank whose shard is empty still takes part in the completion protocol of the fused all-gather
__global__ void gather_flag_only_kernel(const __grid_constant__ FwdParams p) { gather_finish(p); }
}  // namespace mlb

using namespace mlb;

struct mlb_model {
    mlb_model_desc desc;
    mlb_op ops[MLB_MAX_OPS];
    int device, n_sms;
    float* blob_dev;
    size_t n_floats;
    TileFamily tile;
    ClusterFamily cluster;
    WideFamily wide;
    Wide2Family wide2;
    TcFamily tc;
    float* res_scratch;            // residual stash of the row-tile (on request) and tensor-core kernels
    int last_kernel;               // MLB_KERNEL_* of the most recent mlb_forward launch
    // per-wave times measured on this device at mlb_create (ms): FFMA cluster wave, row-tile wave = a + b * TM, tensor-core wave
    double t_cluster_wave, t_tile_a, t_tile_b, t_tc_wave;
    bool calibrated;
    unsigned* gather_done;         // monotonic count of CTAs that finished their peer stores (fused all-gather)
    unsigned gather_done_count;    // host copy of the value it reaches after the launches issued so far
    int* err_flag_dev;             // device view of err_flag_host
    int* err_flag_host;            // mapped pinned host word: the host reads it after a sync without a copy
    float *st_in, *st_in_r, *st_raw, *st_dec, *st_xyzc, *st_x;  // staging for mlb_forward_host
    size_t st_rows, st_rows_r;
};

thread_local std::string g_mlb_err;
static std::atomic<uint64_t> g_launches{0};
void mlb_count_launch() { g_launches++; }

extern "C" const char* mlb_last_error(void) { return g_mlb_err.c_str(); }
extern "C" int mlb_abi_version(void) { return MLB_ABI_VERSION; }
extern "C" uint64_t mlb_launch_count(void) { return g_launches.load(); }

// profiling aid: point the kernels' timestamp marks at a device buffer of >= 4 * n_ops + 4 uint64 (nullptr: off).
// CTA 0 of the tile kernel stamps: [0] start, [1] input tile staged, per op i [2+4i] GEMM done, [3+4i] epilogue math done,
// [4+4i] CTA synchronised, [5+4i] activation tile rewritten; [2+4n] heads done, [3+4n] rows stored.
extern "C" int mlb_debug_fwd_marks(void* dev_buf) {
    unsigned long long* ptr = reinterpret_cast<unsigned long long*>(dev_buf);
    cudaError_t e = TileFamily::set_marks(ptr);
    if (e == cudaSuccess) e = WideFamily::set_marks(ptr);
    if (e == cudaSuccess) e = TcFamily::set_marks(ptr);
    if (e == cudaSuccess) e = Wide2Family::set_marks(ptr);
    if (e != cudaSuccess) return mlb_fail(std::string("mlb_debug_fwd_marks: ") + cudaGetErrorString(e));
    return 0;
}
extern "C" int mlb_num_sms(mlb_handle h) { return h ? h->n_sms : 0; }
extern "C" int mlb_last_kernel(mlb_handle h) { return h ? h->last_kernel : -1; }
extern "C" int mlb_tc_resident_clusters(mlb_handle h) { return (h && h->tc.available) ? h->tc.max_clusters : 0; }
extern "C" int mlb_device_error(mlb_handle h) { return h ? *reinterpret_cast<volatile int*>(h->err_flag_host) : -1; }

// Time one wave of every kernel family on THIS device (CUDA events, L2 warm, 2 launches each, the second one counts) so that
// the batch-size thresholds of mlb_forward are measured quantities instead of constants from another box.  ~10 launches.
static void calibrate(mlb_handle h) {
    const mlb_model_desc& d = h->desc;
    h->t_cluster_wave = 0.185, h->t_tile_a = 0.42, h->t_tile_b = 0.067, h->t_tc_wave = 0.33;  // round-2 B200 defaults
    if (getenv("MLB_NO_CALIBRATE")) return;
    const int max_rows = h->n_sms * 32;
    float *x = nullptr, *raw = nullptr;
    if (cudaMalloc(&x, (size_t)max_rows * d.input_size * sizeof(float)) != cudaSuccess) return;
    if (cudaMalloc(&raw, (size_t)max_rows * d.output_size * sizeof(float)) != cudaSuccess) { cudaFree(x); return; }
    cudaMemset(x, 0, (size_t)max_rows * d.input_size * sizeof(float));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0), cudaEventCreate(&e1);
    auto time_one = [&](int rows, int flags, int tm) -> double {
        mlb_forward_args a;
        memset(&a, 0, sizeof(a));
        a.input_kind = MLB_IN_X, a.flags = flags, a.n_rows = rows, a.rows_per_group = tm, a.x = x, a.out_raw = raw;
        float ms = -1.f;
        for (int rep = 0; rep < 2; ++rep) {
            cudaEventRecord(e0, 0);
            if (mlb_forward(h, &a, nullptr) != 0) return -1.0;
            cudaEventRecord(e1, 0);
            if (cudaEventSynchronize(e1) != cudaSuccess) return -1.0;
            cudaEventElapsedTime(&ms, e0, e1);
        }
        return (double)ms;
    };
    if (h->tile.available) {
        const double t8 = time_one(h->n_sms * 16, MLB_FWD_FORCE_TILE, 8), t16 = time_one(h->n_sms * 32, MLB_FWD_FORCE_TILE, 16);
        if (t8 > 0 && t16 > t8) h->t_tile_b = (t16 - t8) / 8.0, h->t_tile_a = t8 - 8.0 * h->t_tile_b;
        if (h->cluster.available) {
            const double tc = time_one(h->cluster.conc * 16, MLB_FWD_FORCE_CLUSTER, 0);
            if (tc > 0) h->t_cluster_wave = tc;
        }
    }
    if (h->tc.available) {
        const double tt = time_one(128, MLB_FWD_FORCE_TC, 0);
        if (tt > 0) h->t_tc_wave = tt;
    }
    cudaEventDestroy(e0), cudaEventDestroy(e1);
    cudaFree(x), cudaFree(raw);
    cudaGetLastError();
    h->calibrated = true;
}

// everything mlb_create allocates; on failure the caller tears the handle down with mlb_destroy
static int create_resources(mlb_model* m, const float* packed_host) {
    const int L = m->desc.linear_size, n_ops = m->desc.n_ops;
    MLB_CU(cudaMalloc(&m->blob_dev, m->n_floats * sizeof(float)));
    MLB_CU(cudaMemcpy(m->blob_dev, packed_host, m->n_floats * sizeof(float), cudaMemcpyHostToDevice));
    m->tile.setup(L, m->n_sms);
    const cudaError_t et = m->tc.setup(m->blob_dev, m->ops, n_ops, L);
    if (et != cudaSuccess) {
        if (!m->tile.available) return mlb_fail(std::string("mlb_create: tensor-core kernel set-up: ") + cudaGetErrorString(et));
        cudaGetLastError();  // the FFMA kernels cover this width: carry on without the tensor-core path
    }
    MLB_CU(m->cluster.setup(m->blob_dev, m->ops, n_ops, L));
    MLB_CU(m->wide.setup(m->blob_dev, m->ops, n_ops, L, m->n_sms));
    MLB_CU(m->wide2.setup(m->blob_dev, m->ops, n_ops, L, m->desc.output_size, m->n_sms));
    MLB_CU(cudaDeviceSynchronize());
    // up to 4 resident CTAs per SM for narrow models: the row-tile kernel's grid never exceeds it
    MLB_CU(cudaMalloc(&m->res_scratch, (size_t)m->n_sms * 4 * 128 * 256 * sizeof(float)));
    MLB_CU(mlb_zalloc(&m->gather_done, sizeof(unsigned)));
    MLB_CU(cudaHostAlloc(reinterpret_cast<void**>(&m->err_flag_host), sizeof(int), cudaHostAllocMapped));
    *m->err_flag_host = 0;
    MLB_CU(cudaHostGetDevicePointer(reinterpret_cast<void**>(&m->err_flag_dev), m->err_flag_host, 0));
    return 0;
}

extern "C" int mlb_create(const mlb_model_desc* desc, const mlb_op* ops, const float* packed_host, size_t n_floats,
                          int device, mlb_handle* out) {
    if (!desc || !ops || !packed_host || !out) return mlb_fail("mlb_create: null argument");
    if (desc->abi_version != MLB_ABI_VERSION) return mlb_fail("mlb_create: ABI version mismatch");
    if (desc->n_ops < 1 || desc->n_ops > MLB_MAX_OPS) return mlb_fail("mlb_create: n_ops out of range");
    const int L = desc->linear_size;
    if (!TileFamily::covers(L) && !TcFamily::covers(L))
        return mlb_fail("mlb_create: linear_size must be a multiple of 128 up to 1024 or a multiple of 256 up to 2048 "
                        "(monoloco_b200.packing zero-pads other widths)");
    if (desc->input_size < 1 || desc->input_size > 68) return mlb_fail("mlb_create: input_size must be in [1,68]");
    if (desc->output_size < 1 || desc->output_size > OUT_LD) return mlb_fail("mlb_create: output_size must be in [1,16]");
    for (int i = 0; i < desc->n_ops; ++i) {
        const mlb_op& op = ops[i];
        if (op.type == MLB_OP_GEMM) {
            if (op.N != L) return mlb_fail("mlb_create: GEMM op width must equal linear_size");
            if (op.Kpad % KC != 0 || op.Kpad < op.K) return mlb_fail("mlb_create: bad Kpad");
            if ((op.flags & MLB_F_IN_XIN) ? (op.Kpad > KIN_MAX) : (op.K != L)) return mlb_fail("mlb_create: bad GEMM K");
            if ((op.w_off % 4) || (op.scale_off % 4) || (op.shift_off % 4)) return mlb_fail("mlb_create: unaligned offsets");
            if ((size_t)op.w_off + (size_t)op.Kpad * L > n_floats) return mlb_fail("mlb_create: weights out of blob");
        } else if (op.type == MLB_OP_HEAD) {
            if (op.K != L || (op.K % 4)) return mlb_fail("mlb_create: HEAD K must equal linear_size");
            if (op.N < 1 || op.out_col < 0 || op.out_col + op.N > desc->output_size) return mlb_fail("mlb_create: bad HEAD columns");
            if (op.w_off % 4) return mlb_fail("mlb_create: unaligned HEAD weights");
            if ((size_t)op.w_off + (size_t)op.N * op.K > n_floats) return mlb_fail("mlb_create: head weights out of blob");
        } else {
            return mlb_fail("mlb_create: unknown op type");
        }
    }
    MLB_CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    MLB_CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return mlb_fail("mlb_create: this library is built for sm_100a (B200) only");
    mlb_model* m = new mlb_model();
    m->desc = *desc;
    memcpy(m->ops, ops, sizeof(mlb_op) * desc->n_ops);
    m->device = device;
    m->n_sms = prop.multiProcessorCount;
    m->n_floats = n_floats;
    if (create_resources(m, packed_host) != 0) {
        mlb_destroy(m);
        return -1;
    }
    calibrate(m);
    *out = m;
    return 0;
}

extern "C" int mlb_kernel_times(mlb_handle h, double out_ms[4]) {
    if (!h || !out_ms) return mlb_fail("mlb_kernel_times: null argument");
    out_ms[0] = h->t_cluster_wave, out_ms[1] = h->t_tile_a, out_ms[2] = h->t_tile_b, out_ms[3] = h->t_tc_wave;
    return h->calibrated ? 1 : 0;
}

extern "C" int mlb_update_weights(mlb_handle h, const float* packed_host, size_t n_floats, void* stream) {
    if (!h || !packed_host) return mlb_fail("mlb_update_weights: null argument");
    if (n_floats != h->n_floats) return mlb_fail("mlb_update_weights: blob size changed");
    MLB_CU(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int L = h->desc.linear_size, n_ops = h->desc.n_ops;
    MLB_CU(cudaMemcpyAsync(h->blob_dev, packed_host, n_floats * sizeof(float), cudaMemcpyHostToDevice, st));
    MLB_CU(h->cluster.repack(h->blob_dev, h->ops, n_ops, L, st));
    MLB_CU(h->wide.repack(h->blob_dev, h->ops, n_ops, L, st));
    MLB_CU(h->wide2.repack(h->blob_dev, h->ops, n_ops, L, st));
    MLB_CU(h->tc.repack(h->blob_dev, h->ops, n_ops, L, st));
    return 0;
}

extern "C" void mlb_destroy(mlb_handle h) {
    if (!h) return;
    cudaSetDevice(h->device);
    h->cluster.release(), h->wide.release(), h->wide2.release(), h->tc.release();
    cudaFree(h->blob_dev), cudaFree(h->res_scratch), cudaFree(h->gather_done), cudaFreeHost(h->err_flag_host);
    cudaFree(h->st_in), cudaFree(h->st_in_r), cudaFree(h->st_raw), cudaFree(h->st_dec), cudaFree(h->st_xyzc), cudaFree(h->st_x);
    delete h;
}

static FwdPlanInputs plan_inputs(const mlb_model* h) {
    FwdPlanInputs in;
    in.have = (unsigned)h->tile.available << MLB_KERNEL_TILE | (unsigned)h->cluster.available << MLB_KERNEL_CLUSTER |
              (unsigned)h->wide.available << MLB_KERNEL_WIDE | (unsigned)h->tc.available << MLB_KERNEL_TC |
              (unsigned)h->wide2.available << MLB_KERNEL_WIDE2;
    in.disabled = (unsigned)h->wide.disabled << MLB_KERNEL_WIDE | (unsigned)h->wide2.disabled << MLB_KERNEL_WIDE2;
    in.t_cluster_wave = h->t_cluster_wave, in.t_tile_a = h->t_tile_a, in.t_tile_b = h->t_tile_b, in.t_tc_wave = h->t_tc_wave;
    in.n_sms = h->n_sms;
    in.small_conc = h->cluster.conc;
    in.tc_clusters = h->tc.max_clusters;
    in.tile_ctas[0] = h->tile.max_ctas[0], in.tile_ctas[1] = h->tile.max_ctas[1];
    return in;
}

static const char* const kKernelName[] = {"loco_forward_kernel", "loco_forward_cluster_kernel", "loco_forward_wide_kernel",
                                          "loco_forward_tc_kernel", "loco_forward_wide2_kernel"};  // by MLB_KERNEL_*

extern "C" int mlb_forward(mlb_handle h, const mlb_forward_args* a, void* stream) {
    if (!h || !a) return mlb_fail("mlb_forward: null argument");
    if (a->n_rows < 0) return mlb_fail("mlb_forward: negative n_rows");
    if (a->n_gather < 0 || a->n_gather > MLB_MAX_PEERS) return mlb_fail("mlb_forward: n_gather out of range");
    const bool sync_gather = a->n_gather > 0 && a->gather_epoch != 0;
    if (sync_gather) {
        if (a->gather_rank < 0 || a->gather_rank >= a->n_gather) return mlb_fail("mlb_forward: gather_rank out of range");
        for (int i = 0; i < a->n_gather; ++i)
            if (!a->gather_flags[i]) return mlb_fail("mlb_forward: null gather_flags pointer");
    }
    if (a->n_rows == 0) {
        if (!sync_gather) return 0;
        // empty shard: this rank still publishes its epoch and waits for the others
        MLB_CU(cudaSetDevice(h->device));
        FwdParams pe;
        memset(&pe, 0, sizeof(pe));
        pe.n_gather = a->n_gather, pe.gather_epoch = a->gather_epoch, pe.gather_rank = a->gather_rank;
        for (int i = 0; i < a->n_gather; ++i) pe.gather_flags[i] = a->gather_flags[i];
        pe.err_flag = h->err_flag_dev;
        pe.gather_done = h->gather_done;
        pe.gather_done_target = ++h->gather_done_count;
        gather_flag_only_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(pe);
        MLB_CU(cudaGetLastError());
        g_launches++;
        return 0;
    }
    if (!a->x || !a->out_raw) return mlb_fail("mlb_forward: x and out_raw are required");
    const mlb_model_desc& d = h->desc;
    if (a->input_kind == MLB_IN_KPS && d.input_size != 34) return mlb_fail("mlb_forward: MLB_IN_KPS needs a 34-d model");
    if (a->input_kind == MLB_IN_KPS_STEREO) {
        if (d.input_size != 68) return mlb_fail("mlb_forward: MLB_IN_KPS_STEREO needs a 68-d model");
        if (!a->x_right || a->n_left < 1 || a->n_right < 1 || (long long)a->n_left * a->n_right != a->n_rows)
            return mlb_fail("mlb_forward: stereo needs x_right and n_rows == n_left * n_right");
    }
    if (a->input_kind < MLB_IN_X || a->input_kind > MLB_IN_KPS_STEREO) return mlb_fail("mlb_forward: bad input_kind");
    if ((a->flags & MLB_FWD_ZERO_CENTER) && a->input_kind != MLB_IN_KPS) return mlb_fail("mlb_forward: zero_center needs MLB_IN_KPS");
    MLB_CU(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;

    FwdParams p;
    memset(&p, 0, sizeof(p));
    p.blob = h->blob_dev;
    memcpy(p.ops, h->ops, sizeof(mlb_op) * d.n_ops);
    p.n_ops = d.n_ops, p.in_size = d.input_size, p.out_size = d.output_size, p.L = d.linear_size, p.decode_kind = d.decode_kind;
    p.input_kind = a->input_kind;
    p.flags = a->flags;
    // residual stash: Tensor Memory by default (no DRAM write-back traffic, measured 0.5-5 % faster), scratch on request
    if (a->flags & MLB_FWD_RES_SCRATCH) p.flags &= ~MLB_FWD_RES_TMEM; else p.flags |= MLB_FWD_RES_TMEM;
    p.n_rows = a->n_rows;
    p.n_right = a->n_right > 0 ? a->n_right : 1;
    p.kpad0 = h->ops[0].Kpad;
    memcpy(p.kinv, a->kinv, sizeof(p.kinv));
    p.z_met = a->z_met != 0.f ? a->z_met : 10.f;
    p.x = a->x, p.xr = a->x_right;
    p.out_raw = a->out_raw, p.out_dec = a->out_dec, p.out_xyzc = a->out_xyzc, p.out_x = a->out_x;
    p.drop_mask = a->drop_mask, p.drop_seed = a->drop_seed, p.p_drop = d.p_dropout;
    p.res_scratch = h->res_scratch;
    p.err_flag = h->err_flag_dev;
    p.n_gather = a->n_gather, p.gather_row0 = a->gather_row0;
    for (int i = 0; i < a->n_gather; ++i) {
        if (!a->gather[i]) return mlb_fail("mlb_forward: null gather pointer");
        p.gather[i] = a->gather[i];
        p.gather_flags[i] = sync_gather ? a->gather_flags[i] : nullptr;
    }
    p.gather_rank = a->gather_rank, p.gather_done = h->gather_done;
    if (sync_gather) p.gather_epoch = a->gather_epoch;

    for (;;) {
        const FwdPlan pl = plan_forward(plan_inputs(h), a->n_rows, a->flags, a->rows_per_group);
        if (pl.kernel < 0) return mlb_fail(pl.error);
        // the launch that completes the batch carries the value the done counter reaches once every arrival is in
        if (sync_gather) p.gather_done_target = h->gather_done_count + (unsigned)pl.arrivals;
        int issued = 0;
        cudaError_t e;
        switch (pl.kernel) {
            case MLB_KERNEL_TC: e = h->tc.launch(p, pl, st, &issued); break;
            case MLB_KERNEL_WIDE2: e = h->wide2.launch(p, pl, st, &issued); break;
            case MLB_KERNEL_WIDE: e = h->wide.launch(p, pl, st, &issued); break;
            case MLB_KERNEL_CLUSTER: e = h->cluster.launch(p, pl, st, &issued); break;
            default: e = h->tile.launch(p, pl, st, &issued); break;
        }
        g_launches += issued;
        if (e == cudaSuccess) {
            if (sync_gather) h->gather_done_count = p.gather_done_target;
            h->last_kernel = pl.kernel;
            return 0;
        }
        // a refused cooperative launch (e.g. MPS / partitioned SMs) of a latency kernel nobody asked for: use the other
        // kernels from now on.  Nothing ran, so no counter moved.
        const bool fall_back = issued == 0 && !(a->flags & FWD_FORCE_MASK) &&
                               (pl.kernel == MLB_KERNEL_WIDE2 || pl.kernel == MLB_KERNEL_WIDE);
        if (!fall_back) return mlb_fail(std::string(kKernelName[pl.kernel]) + " launch: " + cudaGetErrorString(e));
        cudaGetLastError();
        if (pl.kernel == MLB_KERNEL_WIDE2) h->wide2.disabled = true; else h->wide.disabled = true;
    }
}

static int ensure(float** buf, size_t floats) {
    if (*buf) cudaFree(*buf);
    *buf = nullptr;
    MLB_CU(cudaMalloc(buf, floats * sizeof(float)));
    return 0;
}

extern "C" int mlb_forward_host(mlb_handle h, const mlb_forward_args* a, void* stream) {
    if (!h || !a) return mlb_fail("mlb_forward_host: null argument");
    if (a->n_rows == 0) return 0;
    if (!a->x || !a->out_raw) return mlb_fail("mlb_forward_host: x and out_raw are required");
    MLB_CU(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const mlb_model_desc& d = h->desc;
    const size_t B = (size_t)a->n_rows;
    const bool stereo = a->input_kind == MLB_IN_KPS_STEREO;
    const size_t in_rows = stereo ? (size_t)a->n_left : B;
    const size_t in_w = a->input_kind == MLB_IN_X ? (size_t)d.input_size : 51;
    if (B > h->st_rows || in_rows > h->st_rows) {
        const size_t cap = B > in_rows ? B : in_rows;
        if (ensure(&h->st_in, cap * 68)) return -1;
        if (ensure(&h->st_raw, cap * OUT_LD)) return -1;
        if (ensure(&h->st_dec, cap * 8)) return -1;
        if (ensure(&h->st_xyzc, cap * 4)) return -1;
        if (ensure(&h->st_x, cap * 68)) return -1;
        h->st_rows = cap;
    }
    if (stereo && (size_t)a->n_right > h->st_rows_r) {
        if (ensure(&h->st_in_r, (size_t)a->n_right * 51)) return -1;
        h->st_rows_r = (size_t)a->n_right;
    }
    MLB_CU(cudaMemcpyAsync(h->st_in, a->x, in_rows * in_w * sizeof(float), cudaMemcpyHostToDevice, st));
    if (stereo) {
        if (!a->x_right) return mlb_fail("mlb_forward_host: stereo needs x_right");
        MLB_CU(cudaMemcpyAsync(h->st_in_r, a->x_right, (size_t)a->n_right * 51 * sizeof(float), cudaMemcpyHostToDevice, st));
    }
    mlb_forward_args dev = *a;
    dev.x = h->st_in;
    dev.x_right = stereo ? h->st_in_r : nullptr;
    dev.out_raw = h->st_raw;
    dev.out_dec = a->out_dec ? h->st_dec : nullptr;
    dev.out_xyzc = a->out_xyzc ? h->st_xyzc : nullptr;
    dev.out_x = a->out_x ? h->st_x : nullptr;
    dev.drop_mask = nullptr;
    dev.n_gather = 0;
    if (a->drop_mask) return mlb_fail("mlb_forward_host: drop_mask is a device-only option");
    // One image's worth of rows: the kernel stores straight into the caller's buffers when they are pinned (mapped under
    // UVA) -- a few posted PCIe writes from one CTA instead of three D2H copies.  Larger batches keep the DMA copies
    // (row-at-a-time stores would turn into ~12 small PCIe writes per detection).
    bool zero_copy = B <= 64;
    void* dptr[4] = {nullptr, nullptr, nullptr, nullptr};
    if (zero_copy) {
        void* hp[4] = {a->out_raw, a->out_dec, a->out_xyzc, a->out_x};
        for (int i = 0; i < 4 && zero_copy; ++i) {
            if (!hp[i]) continue;
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, hp[i]) != cudaSuccess || at.type != cudaMemoryTypeHost || !at.devicePointer) {
                cudaGetLastError();
                zero_copy = false;
            } else {
                dptr[i] = at.devicePointer;
            }
        }
    }
    if (zero_copy) {
        dev.out_raw = static_cast<float*>(dptr[0]);
        dev.out_dec = static_cast<float*>(dptr[1]);
        dev.out_xyzc = static_cast<float*>(dptr[2]);
        dev.out_x = static_cast<float*>(dptr[3]);
    }
    if (mlb_forward(h, &dev, stream)) return -1;
    if (!zero_copy) {
        MLB_CU(cudaMemcpyAsync(a->out_raw, h->st_raw, B * d.output_size * sizeof(float), cudaMemcpyDeviceToHost, st));
        if (a->out_dec) MLB_CU(cudaMemcpyAsync(a->out_dec, h->st_dec, B * 8 * sizeof(float), cudaMemcpyDeviceToHost, st));
        if (a->out_xyzc) MLB_CU(cudaMemcpyAsync(a->out_xyzc, h->st_xyzc, B * 4 * sizeof(float), cudaMemcpyDeviceToHost, st));
        if (a->out_x) MLB_CU(cudaMemcpyAsync(a->out_x, h->st_x, B * d.input_size * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    MLB_CU(cudaStreamSynchronize(st));
    const int err = *reinterpret_cast<volatile int*>(h->err_flag_host);
    if (err) return mlb_fail("mlb_forward_host: device error flag " + std::to_string(err));
    return 0;
}
