// Host-side state of the five forward kernel families; mlb_model (model.cu) holds one of each, and each is implemented
// next to its kernel.  setup() runs at mlb_create and sets `available` when the family covers this model on this device
// (an error return is a failed allocation, copy or attribute call); repack() rebuilds the family's weight copy from the
// blob after mlb_update_weights; release() frees what setup() allocated; launch() issues one plan_forward() plan and adds
// the kernel launches that went through to *issued.
#pragma once
#include "fwd_common.cuh"
#include "fwd_plan.h"
#include "host_error.h"

namespace mlb {

struct TileFamily {  // forward.cu: one CTA per row tile (any width the FFMA kernels cover)
    bool available;
    int threads;
    size_t smem;
    int max_ctas[2];  // resident CTAs with the residual in [0] Tensor Memory, [1] the scratch
    static bool covers(int L);
    void setup(int L, int n_sms);
    cudaError_t launch(FwdParams p, const FwdPlan& pl, cudaStream_t st, int* issued) const;
    static cudaError_t set_marks(unsigned long long* ptr);
};

struct ClusterFamily {  // forward_small.cu: an 8-CTA cluster per 16 rows (linear_size == 1024)
    bool available;
    float* slab;  // slab-major W^T copies
    long long slab_off[MLB_MAX_OPS];
    int conc;     // co-resident clusters (cudaOccupancyMaxActiveClusters)
    cudaError_t setup(const float* blob, const mlb_op* ops, int n_ops, int L);
    cudaError_t repack(const float* blob, const mlb_op* ops, int n_ops, int L, cudaStream_t st) const;
    void release();
    cudaError_t launch(FwdParams p, const FwdPlan& pl, cudaStream_t st, int* issued) const;
};

struct WideFamily {  // forward_wide.cu: the whole grid on one 32-row tile per launch
    bool available;
    bool disabled;  // a cooperative launch was refused once: only forced requests still come here
    float* slab;    // per-CTA column slabs
    long long slab_off[MLB_MAX_OPS];
    float* xg;      // [2][L][32] inter-CTA exchange tiles
    unsigned* bar;  // monotonic grid-barrier counter
    unsigned bar_count;  // host copy of the counter after the launches issued so far
    cudaError_t setup(const float* blob, const mlb_op* ops, int n_ops, int L, int n_sms);
    cudaError_t repack(const float* blob, const mlb_op* ops, int n_ops, int L, cudaStream_t st) const;
    void release();
    cudaError_t launch(FwdParams p, const FwdPlan& pl, cudaStream_t st, int* issued);
    static cudaError_t set_marks(unsigned long long* ptr);
};

struct Wide2Family {  // forward_wide2.cu: 4-CTA clusters with a K x N split, <= 16 rows
    bool available;
    bool disabled;           // as WideFamily::disabled
    float* slab;             // [cluster][K slice] slabs
    long long slab_off[MLB_MAX_OPS];
    unsigned long long* xg;  // (value, epoch) exchange pairs
    unsigned long long* hg;  // head partial pairs
    unsigned epoch;          // epochs consumed by the launches issued so far
    cudaError_t setup(const float* blob, const mlb_op* ops, int n_ops, int L, int out_size, int n_sms);
    cudaError_t repack(const float* blob, const mlb_op* ops, int n_ops, int L, cudaStream_t st) const;
    void release();
    cudaError_t launch(FwdParams p, const FwdPlan& pl, cudaStream_t st, int* issued);
    static cudaError_t set_marks(unsigned long long* ptr);
};

struct TcFamily {  // forward_tc.cu: error-compensated TF32 on the tensor cores, persistent clusters over 128-row tiles
    bool available;
    float* wplanes[MLB_MAX_OPS];  // hi / lo weight planes per GEMM
    int n_kb[MLB_MAX_OPS];
    float* ws;                    // one workspace slot per co-resident cluster
    size_t slot_floats;
    int max_clusters;
    int nct;                      // CTAs per cluster = L / 256
    static bool covers(int L);
    // a failed set-up frees what it allocated; the caller decides whether the FFMA kernels can carry on alone
    cudaError_t setup(const float* blob, const mlb_op* ops, int n_ops, int L);
    cudaError_t repack(const float* blob, const mlb_op* ops, int n_ops, int L, cudaStream_t st) const;
    void release();
    cudaError_t launch(FwdParams p, const FwdPlan& pl, cudaStream_t st, int* issued) const;
    static cudaError_t set_marks(unsigned long long* ptr);
};

}  // namespace mlb
