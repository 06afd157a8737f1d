#!/usr/bin/env python
"""
bench.py -- monoloco hot path on B200:  detections/s of the fused forward (pre-process -> LocoModel -> decode).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference] [--dump-outputs DIR]

What it reports (DESIGN.md §6):
  * one step = one pass of the hot path over one batch of synthetic 17-keypoint detections
    (BASELINE.json configs[1]: LocoModel mono 34->9, 3 stages x 1024, batch 4096 per GPU, fp32);
  * `value`  = whole-job detections/s with inputs resident in HBM, timed with CUDA events on the launching stream,
               L2 flushed (256 MiB memset) before every timed step, max over ranks;
  * `e2e`    = same metric through the public host-buffer call (pinned host memory; H2D + kernel(+ all-gather) + D2H
               per step): `mlb_forward_host` at N = 1, `ShardedLoco.forward_host` at N > 1;
  * `roofline` (binding bound first), `cpu_baseline`, `clocks`, `gpu_launches` as specified.
  * --dump-outputs DIR: after the timed steps, the arrays the last timed step handed its caller, as DIR/<name>.npy in
    float32 (`raw` [B,9] and `dec` [B,8] at N = 1, the gathered `rows` [N*B,20] at N > 1, `raw` for --impl reference).
    Inputs are seeded, so two builds run with the same arguments can be compared file for file.
  * --impl reference: the reference's CPU implementation of the path (oracle/torch_port.py = the same torch-eager
    op sequence as the reference nn.Module) timed on the host cores.
Multi-GPU: launched by torch.distributed.run; detections shard over ranks (weak scaling, 4096 per GPU); the step is ONE
kernel launch per rank whose epilogue stores the output rows into every rank's gather buffer over NVLink and whose
last CTA completes the all-gather with a flag protocol on the same peer memory (--gather nccl: NCCL all-gather A/B).
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "detections/sec LocoModel(34->9, 3x1024) fused forward @ batch 4096 per GPU"
UNIT = "detections/s"
DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(path, arrays):
    """Write {name: tensor or array} as path/<name>.npy in float32.  All arrays share the row dimension; when they come to
    more than DUMP_BYTES, the same fixed, seeded sample of rows is kept from each and its row numbers go to row_index.npy
    (float64), so that two runs with the same arguments write the same rows."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)).astype(np.float32)
              for k, v in arrays.items()}
    n = next(iter(arrays.values())).shape[0]
    row_bytes = sum(a[:1].nbytes for a in arrays.values())
    if n * row_bytes > DUMP_BYTES:
        k = (DUMP_BYTES - 4096) // (row_bytes + 8)   # 4 KiB for the .npy headers, 8 B per row for its index
        idx = np.sort(np.random.RandomState(0).choice(n, k, replace=False))
        arrays = {name: a[idx] for name, a in arrays.items()}
        arrays['row_index'] = idx.astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), a)


def profile_json(name):
    path = os.path.join(ROOT, 'profiles', name)
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return {}


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d.get('hbm_gbs', 6650.0), 'measured (MEASURED_PEAKS.json)', d
    return 6650.0, 'fallback (B200_PROFILING.md)', {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md): one persistent
    `nvidia-smi -lms 20` process, started before and killed after the region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '20'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.15)  # first sample lands before the timed region starts
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is None:
            return
        time.sleep(0.05)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ''
        self.rows = [[c.strip() for c in ln.split(',')] for ln in out.strip().splitlines() if ln.strip()]

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def best_cpu_threads(fn, reps=5, budget_s=25.0):
    """The reference's CPU path is torch eager; on a many-core shared host `all threads` is often NOT its fastest
    setting.  Policy (fixed, so that two boxes pick the same way): candidates 8/16/32/64/all cores, one warm-up call
    then the MEDIAN of `reps` timed calls each; a candidate whose first timed call is > 3x the best median so far is
    dropped after that call.  Returns (best thread count, {threads: median seconds})."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu})
    table, best, best_t = {}, cands[0], None
    t_all = time.perf_counter()
    for c in cands:
        torch.set_num_threads(c)
        fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
            if best_t is not None and ts[0] > 3.0 * best_t:
                break
        med = float(np.median(ts))
        table[str(c)] = med
        if best_t is None or med < best_t:
            best, best_t = c, med
        if time.perf_counter() - t_all > budget_s:
            break
    torch.set_num_threads(best)
    return best, table


def cpu_reference_rate(sd, x_np, budget_s=10.0, min_reps=5):
    """detections/s of the reference's CPU path (torch eager, best host thread count) on a bounded sample."""
    from oracle import torch_port as T  # the one place bench.py executes oracle/: the timed CPU baseline
    tsd = T.to_torch(sd)
    x = torch.from_numpy(x_np)
    with torch.no_grad():
        _, table = best_cpu_threads(lambda: T.model_forward(tsd, x))
        for _ in range(2):
            T.model_forward(tsd, x)
        times = []
        t_all = time.perf_counter()
        while len(times) < min_reps or (time.perf_counter() - t_all < budget_s and len(times) < 200):
            t0 = time.perf_counter()
            T.model_forward(tsd, x)
            times.append(time.perf_counter() - t0)
    med = float(np.median(times))
    return x_np.shape[0] / med, len(times), med, table


# ------------------------------------------------------------------------------------------------------------------
# torch-eager CUDA comparator: the only GPU implementation the reference has (trainer.py:81-82, predict.py:117-121 pick
# cuda when available; BASELINE.md §3).  The reference nn.Module's op sequence (architectures.py:48-71, 88-102) through
# torch.nn.functional on the same state_dict: cuBLAS SGEMM with TF32 off (torch default) + aten elementwise kernels.
# ------------------------------------------------------------------------------------------------------------------
def _eager_forward(sd, x, training=False, p=0.0):
    F = torch.nn.functional

    def block(y, lin, bn, relu=True):
        y = F.linear(y, sd[lin + '.weight'], sd[lin + '.bias'])
        if bn is not None:
            y = F.batch_norm(y, sd[bn + '.running_mean'], sd[bn + '.running_var'], sd[bn + '.weight'], sd[bn + '.bias'],
                             training=training, momentum=0.1, eps=1e-5)
        if relu:
            y = F.relu(y)
            if training and p > 0:
                y = F.dropout(y, p, True)
        return y

    y = block(x, 'w1', 'batch_norm1')
    i = 0
    while 'linear_stages.%d.w1.weight' % i in sd:
        s = 'linear_stages.%d' % i
        y = y + block(block(y, s + '.w1', s + '.batch_norm1'), s + '.w2', s + '.batch_norm2')
        i += 1
    if 'w_fin.weight' not in sd:
        return F.linear(y, sd['w2.weight'], sd['w2.bias'])
    y = F.linear(y, sd['w2.weight'], sd['w2.bias'])
    aux = F.linear(y, sd['w_aux.weight'], sd['w_aux.bias'])
    y = block(y, 'w3', 'batch_norm3')
    return torch.cat((F.linear(y, sd['w_fin.weight'], sd['w_fin.bias']), aux), dim=1)


def _eager_loss(out, lab):
    """MultiTaskLoss over ('d','x','y','h','w','l','ori') with unit lambdas (losses.py:59-73, 121-131)."""
    mu, si, g = out[:, 2:3], out[:, 3:4], lab[:, 3:4]
    loss = (torch.abs(1 - mu / g) * torch.exp(-si) + 0.01 + si + 2).mean()
    for oc, gc in ((slice(0, 1), slice(0, 1)), (slice(1, 2), slice(1, 2)), (slice(4, 5), slice(4, 5)),
                   (slice(5, 6), slice(5, 6)), (slice(6, 7), slice(6, 7)), (slice(7, 9), slice(7, 9))):
        loss = loss + torch.nn.functional.l1_loss(out[:, oc], lab[:, gc])
    return loss


def timed(fn, n, dev, flush=None):
    """Mean / min ms over n device-timed calls (CUDA events on the current stream).  flush: a buffer larger than L2
    that is rewritten before every call (cold-cache timing); events bracket only the call."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize(dev)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    for e0, e1 in ev:
        if flush is not None:
            flush.zero_()
        e0.record()
        fn()
        e1.record()
    torch.cuda.synchronize(dev)
    ts = [e0.elapsed_time(e1) for e0, e1 in ev]
    return float(np.mean(ts)), float(np.min(ts))


def extras(eng, sd, dev, flush, ffma_peak):
    """Side measurements outside the timed region (the other BASELINE.json configs and the verdict's comparators),
    device-timed.  Every entry says whether L2 was warm or flushed."""
    from monoloco_b200 import synthetic, packing, engine as E, _lib as L_
    out = {}
    kk = synthetic.KITTI_K
    fpd = packing.flops_per_detection(sd)
    hbm_peak = peaks()[0]
    try:
        # ---- forward latency by batch (L2 warm, back to back): which kernel runs and its share of the FFMA peak
        lat = {}
        for b in (1, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 65536):
            x = torch.from_numpy(synthetic.make_keypoints(b, seed=2)).to(dev)
            ms, _ = timed(lambda: eng.forward(x, kk=kk, kind=L_.IN_KPS), 20 if b <= 4096 else 3, dev)
            lat[str(b)] = {"ms": ms, "kernel": eng.last_kernel()[1], "tflops": fpd * b / ms / 1e9,
                           "vs_fp32_ffma_peak": (fpd * b / ms / 1e9 / ffma_peak) if ffma_peak else None}
        out["forward_ms_by_batch"] = lat
        # ---- one image's worth of detections (<= 32 rows) is the weight-streaming regime (SURVEY 8(d): B <= ~19): the
        # whole-grid kernel against the HBM copy peak on the bytes it has to touch, L2 flushed (cold) and warm
        wbytes = eng.packed.blob.size * 4
        x16 = torch.from_numpy(synthetic.make_keypoints(16, seed=2)).to(dev)
        cold, cold_min = timed(lambda: eng.forward(x16, kk=kk, kind=L_.IN_KPS), 20, dev, flush=flush)
        warm = lat["16"]["ms"]
        out["small_batch_roofline"] = {
            "rows": 16, "kernel": eng.last_kernel()[1], "bound": "hbm", "weight_bytes": wbytes,
            "cold_ms": cold, "cold_min_ms": cold_min, "cold_GBps": wbytes / (cold * 1e-3) / 1e9,
            "cold_frac_of_hbm_copy_peak": wbytes / (cold * 1e-3) / 1e9 / hbm_peak,
            "warm_ms": warm, "warm_GBps": wbytes / (warm * 1e-3) / 1e9,
            "warm_frac_of_hbm_copy_peak": wbytes / (warm * 1e-3) / 1e9 / hbm_peak, "peak_GBps": hbm_peak}
        # ---- BASELINE.json's literal metric: MonolocoModel(34, 9, 1024) forward at batch 4096 (architectures.py:105-145)
        msd = synthetic.make_state_dict('monoloco', 34, 9, 1024, 3, 1)
        meng = E.LocoEngine(msd, device=dev)
        x4k = torch.from_numpy(synthetic.make_keypoints(4096, seed=2)).to(dev)
        ms, _ = timed(lambda: meng.forward(x4k, kk=kk, kind=L_.IN_KPS), 10, dev, flush=flush)
        mf = packing.flops_per_detection(msd)
        out["monoloco_model_l1024_b4096"] = {"ms": ms, "detections_per_s": 4096 / (ms * 1e-3), "l2": "flushed",
                                             "kernel": meng.last_kernel()[1], "tflops": mf * 4096 / ms / 1e9,
                                             "vs_fp32_ffma_peak": (mf * 4096 / ms / 1e9 / ffma_peak) if ffma_peak else None}
        meng.close()
        # ---- configs[2]: stereo 64 x 64 pairs + arg-max filter + xyz_from_distance
        seng = E.LocoEngine(synthetic.make_state_dict('loco', 68, 10, 1024, 3, 2), device=dev)
        le, ri = synthetic.make_keypoints(64, seed=3, right=True)
        le, ri = torch.from_numpy(le).to(dev), torch.from_numpy(ri).to(dev)

        def stereo():
            o = seng.forward(le, x_right=ri, kk=kk, kind=L_.IN_KPS_STEREO, want_xyzc=True)
            seng.stereo_filter(o['raw'], o['dec'], 64, 64, xyzc=o['xyzc'], trim=False)
        out["stereo_64x64_pairs_plus_filter_ms"] = timed(stereo, 10, dev)[0]
        seng.close()
        # ---- N2: MC-dropout epistemic path, 50 passes x 16 detections + Laplace sampling + std (net.py:135-161)
        out["epistemic_n50_m16_ms"] = timed(lambda: eng.epistemic_std(x16, 50, kind=L_.IN_KPS, kk=kk), 10, dev)[0]
        # ---- configs[3]: the one-launch training step at batch 4096
        from monoloco_b200.network.architectures import LocoModel
        from monoloco_b200.train import train_step
        m = LocoModel(34, 9, 1024, p_dropout=0.2, num_stage=3)
        m.load_state_dict({k: torch.from_numpy(np.array(v)) for k, v in sd.items()})
        m.to(dev).train()
        xt = torch.from_numpy(synthetic.make_inputs(4096, 34, seed=3)).to(dev)
        yt = torch.from_numpy(synthetic.make_labels(4096, seed=4)).to(dev)
        tasks = ('d', 'x', 'y', 'h', 'w', 'l', 'ori')
        ms, _ = timed(lambda: train_step(m, xt, yt, tasks), 5, dev)
        tr = profile_json('train_traffic.json')
        out["train_step_b4096"] = {
            "ms": ms, "what": "forward + MultiTaskLoss + backward + dW, one cooperative launch, fp32",
            "roofline": {"bound": "fp32", "achieved": 3 * fpd * 4096 / ms / 1e9, "peak": ffma_peak, "unit": "TFLOP/s",
                         "frac": (3 * fpd * 4096 / ms / 1e9 / ffma_peak) if ffma_peak else None,
                         "algorithmic_flops": 3 * fpd * 4096, "traffic": tr.get('traffic_bytes'),
                         "algorithmic_bytes": tr.get('algorithmic_bytes'), "traffic_source": tr.get('source')}}
        del m
        # ---- the reference's own GPU path: torch-eager CUDA (cuBLAS SGEMM, TF32 off), same weights / shapes
        assert not torch.backends.cuda.matmul.allow_tf32
        dsd = {k: torch.as_tensor(np.array(v)).to(dev) for k, v in sd.items()}
        xin = torch.from_numpy(synthetic.make_inputs(4096, 34, seed=0)).to(dev)
        with torch.no_grad():
            ef, _ = timed(lambda: _eager_forward(dsd, xin), 10, dev, flush=flush)
        ours_x, _ = timed(lambda: eng.forward(xin, kind=L_.IN_X), 10, dev, flush=flush)
        gsd = {k: (v.clone().requires_grad_(True) if (v.is_floating_point() and 'running' not in k) else v.clone())
               for k, v in dsd.items()}

        def eager_train():
            for v in gsd.values():
                v.grad = None
            _eager_loss(_eager_forward(gsd, xt, training=True, p=0.2), yt).backward()
        et, _ = timed(eager_train, 5, dev)
        out["torch_eager_cuda"] = {
            "what": "reference op sequence through torch.nn.functional on the same B200 (cuBLAS SGEMM fp32, TF32 off)",
            "forward_b4096_ms": ef, "forward_b4096_ours_same_input_ms": ours_x, "forward_speedup": ef / ours_x,
            "train_step_b4096_ms": et, "train_step_ours_ms": ms, "train_speedup": et / ms,
            "l2": "flushed before every forward; train steps back to back"}
    except Exception as exc:  # side measurements must never break the contract line
        out["error"] = repr(exc)
    return out


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path, timed on the host cores."""
    if rank != 0:
        return
    from monoloco_b200 import synthetic
    from oracle import loco_oracle as O
    from oracle import torch_port as T
    sd = synthetic.make_state_dict('loco', 34, 9, 1024, 3, 0)
    B = args.batch
    kps = synthetic.make_keypoints(B, seed=0)
    tsd = T.to_torch(sd)
    times = []
    with torch.no_grad():
        x0 = torch.from_numpy(O.preprocess_monoloco(kps, synthetic.KITTI_K))
        _, table = best_cpu_threads(lambda: T.model_forward(tsd, x0))
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            x = O.preprocess_monoloco(kps, synthetic.KITTI_K)           # process.py:47-67
            out = T.model_forward(tsd, torch.from_numpy(x))            # architectures.py:48-71
            O.extract_outputs(out.numpy())                             # process.py:231-278
            if i >= args.warmup:
                times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {'raw': out})
    ms = 1e3 * float(np.mean(times))
    val = B / (ms * 1e-3)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "ms_per_step_median": 1e3 * float(np.median(times)),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "LocoModel mono 34->9 L=1024 x3 stages, pre-process + forward + decode, batch %d, CPU" % B,
                       "batch_per_step": B},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                             "host_cpus": os.cpu_count(), "thread_candidates_median_s": table,
                             "sample": "%d steps x %d detections, torch-eager CPU restatement (oracle/torch_port.py), thread "
                                       "count = best median of 5 over 8/16/32/64/all" % (args.steps, B)},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def step_stats(per_step):
    a = np.asarray(per_step, dtype=np.float64)
    return {"median": float(np.median(a)), "p95": float(np.percentile(a, 95)), "max": float(a.max()),
            "min": float(a.min()), "slowest_step": int(a.argmax())}


def gather_sample_check(rows, world, B, seeds, sd, n_per_rank=16):
    """Gathered rows against the oracle on a sample (first / last rows of every rank's shard)."""
    from oracle import loco_oracle as O  # checker only; outside every timed region
    from monoloco_b200 import synthetic, _lib as L_
    worst, ok_all, n = 0.0, True, 0
    for r in range(world):
        kps = synthetic.make_keypoints(B, seed=seeds[r])
        idx = np.unique(np.concatenate([np.arange(min(n_per_rank, B)), np.arange(max(B - n_per_rank, 0), B)]))
        ref_raw = O.loco_model_forward(sd, O.preprocess_monoloco(kps[idx], synthetic.KITTI_K))
        ref = O.extract_outputs(ref_raw)
        got = rows[r * B + idx].cpu().numpy()
        ok, w = O.close(got[:, :9], ref_raw)
        ok2, w2 = O.close(got[:, L_.GATHER_DEC:L_.GATHER_DEC + 4], ref['xyzd'], col_scale=False)
        ok_all &= bool(ok and ok2)
        worst = max(worst, float(w), float(w2))
        n += len(idx)
    return {"rows_checked": n, "ok": ok_all, "worst_err_over_tol": worst}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--batch', type=int, default=4096, help='detections per GPU per step')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='skip the side measurements')
    ap.add_argument('--rows-per-group', type=int, default=0)
    ap.add_argument('--gather', default='fused', choices=['fused', 'nccl'],
                    help='multi-GPU output all-gather: fused peer stores + device-side flags, or NCCL')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help="write the last timed step's outputs to DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))

    if args.impl == 'reference':
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    from monoloco_b200 import synthetic, engine, packing, _lib as L_

    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    B = args.batch
    sd = synthetic.make_state_dict('loco', 34, 9, 1024, 3, 0)
    eng = engine.LocoEngine(sd, device=dev)
    lib = L_.lib()
    kk = synthetic.KITTI_K
    kps_host = torch.from_numpy(synthetic.make_keypoints(B, seed=rank)).pin_memory()
    kps = kps_host.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    st = torch.cuda.current_stream(dev)
    sharded = None
    if world > 1:
        from monoloco_b200 import distributed as D
        sharded = D.ShardedLoco(eng, world * B, mode=args.gather)

    def step():
        if sharded is not None:
            return sharded.forward(kps, kk, rows_per_group=args.rows_per_group)  # forward + all-gather of [N*B, 20] rows
        return eng.forward(kps, kk=kk, kind=L_.IN_KPS, rows_per_group=args.rows_per_group)

    for _ in range(args.warmup):
        flush.zero_()
        step()
    torch.cuda.synchronize(dev)

    # ---------------- timed region: K steps, device-timed, L2 flushed before each.  The barrier + synchronize sit INSIDE
    # the sampler block, after its process start-up, so no rank's entry skew is billed to step 0.
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    with ClockSampler(local_rank) as clocks:
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        # the sampler start-up + barrier left the GPU idle for ~0.2 s: two more untimed steps, queued directly in front of the
        # timed ones, so that step 0 is not billed for the wake-up (it was 1.5 x the median in every run)
        for _ in range(2):
            flush.zero_()
            step()
        launches0 = lib.mlb_launch_count()
        for e0, e1 in ev:
            flush.zero_()
            e0.record(st)
            out = step()
            e1.record(st)
        torch.cuda.synchronize(dev)
        launches = lib.mlb_launch_count() - launches0
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)
    eng.check_error()
    eng.last_kernel_of_step = eng.last_kernel()
    # before the all-reduce below: at N > 1 the rows are a view of a gather buffer that every rank's next step overwrites
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out if sharded is None else {'rows': out})
    per_step = torch.tensor([e0.elapsed_time(e1) for e0, e1 in ev], dtype=torch.float64, device=dev)
    total = per_step.sum().reshape(1)
    if world > 1:
        dist.all_reduce(total, op=dist.ReduceOp.MAX)      # the contract's number: max over ranks of the K-step time
        dist.all_reduce(per_step, op=dist.ReduceOp.MAX)   # per-step distribution: slowest rank of every step
    ms_per_step = float(total.item()) / args.steps
    value = world * B / (ms_per_step * 1e-3)
    stats = step_stats(per_step.cpu().numpy())

    # ---------------- e2e through the public host-buffer call (pinned host memory in, pinned host memory out)
    if sharded is None:
        out_host = {'raw': torch.empty((B, 9)).pin_memory(), 'dec': torch.empty((B, 8)).pin_memory()}
        e2e_call = lambda: eng.forward_host(kps_host, kk=kk, kind=L_.IN_KPS, out=out_host)  # noqa: E731
        h2d, d2h = B * 51 * 4, B * 17 * 4
        e2e_what = "mlb_forward_host: H2D keypoints + fused forward + D2H raw/decoded rows + sync"
    else:
        rows_host = torch.empty((world * B, L_.GATHER_LD), dtype=torch.float32).pin_memory()
        e2e_call = lambda: sharded.forward_host(kps_host, kk, out_rows_host=rows_host)  # noqa: E731
        h2d, d2h = B * 51 * 4, world * B * L_.GATHER_LD * 4
        e2e_what = ("ShardedLoco.forward_host per rank: H2D local keypoints + fused forward + all-gather + D2H of the "
                    "whole gathered [N*B,20] tensor + sync")
    for _ in range(3):
        e2e_call()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_call()
    torch.cuda.synchronize(dev)
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    if world > 1:
        t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = world * B / (e2e_ms * 1e-3)

    multi = {}
    if world > 1:
        # gathered bytes against the oracle on a sample, from one more (untimed) step
        rows = step()
        torch.cuda.synchronize(dev)
        eng.check_error()
        if rank == 0:
            multi["gather_check"] = gather_sample_check(rows, world, B, list(range(world)), sd)
        dist.barrier()
        # BASELINE configs[4]: 1 M detections over 8 GPUs = 131072 rows per GPU (weak scaling at the other N)
        B4 = 131072
        from monoloco_b200 import distributed as D
        sh4 = D.ShardedLoco(eng, world * B4, mode=args.gather)
        k4 = torch.from_numpy(synthetic.make_keypoints(B4, seed=1000 + rank)).to(dev)
        for _ in range(2):
            sh4.forward(k4, kk)
        torch.cuda.synchronize(dev)
        dist.barrier()
        torch.cuda.synchronize(dev)
        n4 = 5
        ev4 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n4)]
        for e0, e1 in ev4:
            flush.zero_()
            e0.record(st)
            rows4 = sh4.forward(k4, kk)
            e1.record(st)
        torch.cuda.synchronize(dev)
        eng.check_error()
        t4 = torch.tensor([sum(e0.elapsed_time(e1) for e0, e1 in ev4)], dtype=torch.float64, device=dev)
        dist.all_reduce(t4, op=dist.ReduceOp.MAX)
        ms4 = float(t4.item()) / n4
        if rank == 0:
            multi["config4_131072_per_gpu"] = {
                "rows_per_gpu": B4, "global_rows": world * B4, "ms_per_step": ms4, "steps": n4,
                "value": world * B4 / (ms4 * 1e-3), "unit": UNIT,
                "gather_check": gather_sample_check(rows4, world, B4, [1000 + r for r in range(world)], sd)}
        dist.barrier()
        sh4.close()

    if rank == 0:
        hbm_peak, peak_src, pk = peaks()
        w_bytes = eng.packed.blob.size * 4
        io_bytes = 204 + 36 + 32          # raw kps in + raw out + decoded out (SURVEY.md §8d)
        alg_bytes = w_bytes + B * io_bytes
        flops = packing.flops_per_detection(sd) * B
        # single-GPU kernel time: at world == 1 the step is exactly one launch of loco_forward_kernel
        achieved_gbs = alg_bytes / (ms_per_step * 1e-3) / 1e9
        ffma_peak = engine.probe_ffma_tflops(local_rank)
        achieved_tf = flops / (ms_per_step * 1e-3) / 1e12
        tr = profile_json('forward_traffic.json')
        kid, kname = eng.last_kernel_of_step
        if kid == 3:
            # tensor-core kernel: every fp32 product is three TF32 MMAs (hi.hi, lo.hi, hi.lo) -> executed tensor flops =
            # 3 x algorithmic; TF32 dense peak = half the bf16 peak the driver measured (K = 8 vs 16 per instruction)
            bf16_peak = float(pk.get('bf16_tflops', 2250.0 * 0.75))
            tf32_peak = bf16_peak / 2.0
            roof = {"bound": "tensor", "kernel": kname, "achieved": 3.0 * achieved_tf, "peak": tf32_peak, "unit": "TFLOP/s",
                    "frac": 3.0 * achieved_tf / tf32_peak,
                    "what": "executed TF32 tensor-core flops (3 MMAs per fp32 product: a_hi.w_hi, a_lo.w_hi, a_hi.w_lo) / kernel time",
                    "peak_source": "TF32 dense = bf16 dense / 2; bf16 %.1f TFLOP/s %s" % (bf16_peak, 'measured (MEASURED_PEAKS.json, burst)' if 'bf16_tflops' in pk else 'fallback'),
                    "algorithmic_flops": flops, "algorithmic_tflops": achieved_tf,
                    "algorithmic_frac_of_tf32_peak": achieved_tf / tf32_peak,
                    "algorithmic_vs_fp32_ffma_peak": achieved_tf / ffma_peak if ffma_peak else None,
                    "fp32_ffma_peak": ffma_peak,
                    "traffic": tr.get('traffic_bytes') if B == 4096 else None, "traffic_source": tr.get('source'),
                    "algorithmic_bytes": alg_bytes}
        else:
            roof = {"bound": "fp32", "kernel": kname, "achieved": achieved_tf, "peak": ffma_peak, "unit": "TFLOP/s",
                    "frac": achieved_tf / ffma_peak if ffma_peak else None,
                    "peak_source": "measured in-run by mlb_probe_ffma (pure FFMA kernel; 148 SM x 128 lanes x 2 x clock)",
                    "algorithmic_flops": flops,
                    "traffic": tr.get('traffic_bytes') if B == 4096 else None, "traffic_source": tr.get('source'),
                    "algorithmic_bytes": alg_bytes}
        roof["hbm"] = {"bound": "hbm", "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s",
                       "frac": achieved_gbs / hbm_peak, "peak_source": peak_src,
                       "note": "not the binding bound at this batch (weights are read once, 34.9 MB per launch); see "
                               "extras.small_batch_roofline for the <= 32-row regime where it is"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "ms_per_step_stats": stats,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "LocoModel mono 34->9 L=1024 x3 stages: raw keypoints [B,3,17] -> fused pre-process + "
                                   "forward + decode, batch %d per GPU" % B,
                       "batch_per_gpu": B, "global_batch": world * B, "parallelism": "dp%d" % world,
                       "l2": "flushed before every timed step (256 MiB memset)",
                       "collective": ("none" if world == 1 else
                                      ("one launch per step: kernel-epilogue peer stores over NVLink (cudaIpc) + device-side "
                                       "release/acquire flag protocol, no NCCL in the data plane" if args.gather == 'fused'
                                       else "NCCL all_gather_into_tensor") + " of [N*B,20] fp32 rows per step")},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms, "what": e2e_what},
            "gpu_launches": int(launches),
            "clocks": clocks.summary(),
            # binding bound first (the kernel that ran decides: tensor cores at this batch); the HBM figure the metric
            # string asks for is nested beside it
            "roofline": roof,
        }
        line["kernel_selection"] = eng.kernel_times()
        line.update(multi)
        if not args.no_extras and world == 1:
            line["extras"] = extras(eng, sd, dev, flush, ffma_peak)
        if not args.no_cpu_baseline and world == 1:   # reported on rank 0 at N = 1 only
            x = np.ascontiguousarray(synthetic.make_inputs(B, 34, seed=0))
            rate, reps, med, table = cpu_reference_rate(sd, x)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                                    "host_cpus": os.cpu_count(), "thread_candidates_median_s": table,
                                    "sample": "%d x batch-%d model forwards (oracle/torch_port.py), median %.1f ms; thread "
                                              "count = best median of 5 over 8/16/32/64/all" % (reps, B, med * 1e3)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        if sharded is not None:
            sharded.close()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
