#!/usr/bin/env python
"""bench.py -- BASELINE.json metric on BASELINE.json configs[1]:
   Faster-RCNN 2FC + Relation + LearnNMS, ResNet-101, synthetic 1000x600 image, N=300 ROIs, 16 heads, one image per GPU.

A "step" = one image through trunk (torch/cuDNN, library plumbing) + the hot path (hand-written CUDA behind the C ABI:
proposal -> ROI pool -> fc_new_1 -> relation#1 -> fc_new_2 -> relation#2 -> cls/bbox -> learn_nms).
  value      images/sec, inputs resident in HBM, CUDA events, barrier+sync both sides, max over ranks
  e2e        same through the public API with the image in pinned HOST memory (H2D inside the timed region) and the
             detections (sorted boxes + final scores) copied back to the host every step
  hot_path   the same step without the trunk (trunk outputs resident) + relation-module microseconds
  roofline   the fused relation kernel (relation_fused_kernel: geometry + pair FC + QK^T + softmax + P.V' in one launch)
             timed alone as a captured graph at N=M=300, d=1024, H=16: achieved = 4*N*M*d FLOP / duration against the
             measured bf16 peak (MEASURED_PEAKS.json); algorithmic bytes by SURVEY 8(d)
  sweep      BASELINE.json configs[4]: N in {100,300,1000,3000} x d in {256,1024} x H in {4,16} (all 16 on the tcgen05 kernels)
  train      the training form of configs[1]: fwd+bwd as ONE CUDA-graph replay, one flat gradient bucket, ONE NCCL SUM allreduce,
             SGD (1 image per rank per step); allreduce timed alone and in the step, bus GB/s, elementwise sum check
  configs    configs[2] Deformable Faster (test-time images/sec) and configs[3] FPN (test-time images/sec + the data-parallel
             training step with 2 images per GPU accumulated before the one allreduce)
  cpu_baseline  the numpy/C oracle of the hot path (oracle/pipeline_np.py) on this host, one image
  --impl reference   the CPU arm: torch-CPU fp32 trunk + oracle hot path, same metric/config (rank 0 only)
  --dump-outputs DIR what the last timed step returned (either arm), as DIR/<name>.npy

bench.py measures the library as __graft_entry__.build() left it and writes nothing in the tree, which may be read-only: it
compiles nothing, and stops with an error when the library is missing or older than its sources (run build() first).

Multi-GPU (torchrun): images are independent at test time -> N replicas, one image per rank per step, no data-path
collective (the reference's only exchange is the gradient allreduce of training; DESIGN.md section "multi-GPU").
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np   # noqa: E402
import torch         # noqa: E402

WORKLOAD = 'faster_rcnn_2fc_relation_learnnms_r101_600x1000_n300_h16'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--precision', default=None, choices=[None, 'f16', 'fp32'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-sweep', action='store_true', help='skip the relation-module roofline sweep (configs[4])')
    ap.add_argument('--no-train', action='store_true', help='skip the data-parallel training blocks (gradient allreduce)')
    ap.add_argument('--no-configs', action='store_true', help='skip the configs[2] (Deformable) and configs[3] (FPN) blocks')
    ap.add_argument('--extras-budget', type=float, default=float(os.environ.get('RELNET_EXTRAS_BUDGET_S', '120')),
                    help='seconds the optional blocks (configs[2]/[3], training steps) may take after the headline measurement; past '
                         'it every rank stops and rank 0 prints the line without them')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last timed step returned to its caller as DIR/<name>.npy '
                         '(float32, float64 for integer outputs; rank 0).  Inputs and weights are seeded, so two builds '
                         'run with the same arguments can be compared output for output')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    return args


DUMP_LIMIT = 64 << 20


def dump_outputs(outdir, outputs):
    """outputs: {name: torch tensor or numpy array} -> outdir/<name>.npy; floating point as float32 (float64 kept), integers
    as float64 (exact).  The detection outputs of one image are a few MB, far below DUMP_LIMIT."""
    arrs = {}
    for k, v in outputs.items():
        t = torch.as_tensor(v).detach().cpu()
        arrs[k] = (t.double() if t.dtype == torch.float64 or not t.is_floating_point() else t.float()).numpy()
    total = sum(a.nbytes for a in arrs.values())
    if total > DUMP_LIMIT:
        raise RuntimeError('--dump-outputs: %d bytes exceed the %d byte limit' % (total, DUMP_LIMIT))
    os.makedirs(outdir, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(outdir, k + '.npy'), a)


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d['hbm_gbs'], tflops=d['bf16_tflops'], tflops_sustained=d.get('bf16_tflops_sustained'),
                    source='MEASURED_PEAKS.json (of measured)')
    return dict(hbm_gbs=6650.0, tflops=1590.0, tflops_sustained=1400.0, source='B200_PROFILING.md fallback (of fallback)')


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled DURING the timed region: NVML (a few ms per sample, so even a 35 ms region gets
    several) with the nvidia-smi query of the profiling recipe as the fallback."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
    NAMES = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.source = index, [], False, 'nvidia-smi'
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = (pynvml, pynvml.nvmlDeviceGetHandleByIndex(index))
            self.source = 'nvml'
        except Exception:
            self.nvml = None

    def sample_nvml(self):
        nv, h = self.nvml
        sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        flags = [bool(r & nv.nvmlClocksThrottleReasonHwSlowdown), bool(r & nv.nvmlClocksThrottleReasonHwThermalSlowdown),
                 bool(r & nv.nvmlClocksThrottleReasonSwThermalSlowdown), bool(r & nv.nvmlClocksThrottleReasonSwPowerCap)]
        return [str(sm), str(mx)] + ['Active' if f else 'Not Active' for f in flags]

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self.rows.append(self.sample_nvml())
                    time.sleep(0.004)
                    continue
            except Exception:
                self.nvml, self.source = None, 'nvidia-smi'          # fall back for the rest of the run
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(',')]
                if len(f) >= 6:
                    self.rows.append(f)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        sm = sorted(float(r[0]) for r in self.rows)
        reasons = [n for i, n in enumerate(self.NAMES) if any(r[2 + i].lower().startswith('active') for r in self.rows)]
        return dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=float(self.rows[0][1]), reasons=reasons, samples=len(self.rows),
                    source=self.source)


def make_inputs(seed=0):
    g = torch.Generator().manual_seed(seed)
    image = torch.randn((1, 3, 600, 1000), generator=g) * 50.0          # post mean-subtraction scale (SURVEY 8d)
    im_info = torch.tensor([[600.0, 1000.0, 1.0]])
    return image, im_info


def timed(fn, steps, warmup, dist_on, after=None):
    """W untimed steps, then exactly K steps between barrier+synchronize, CUDA events, ms for all K steps (max ranks).
    after: called once after the K steps and before the closing event (multi-stream pipelines: drain every in-flight
    image, so all of their copies are inside the timed region)."""
    import torch.distributed as dist
    for _ in range(warmup):
        fn()
    if after:
        after()
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    if after:
        after()
        torch.cuda.synchronize()      # every stream of the pipeline is idle: the closing event is stamped after all of them
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if dist_on:
        from relnet_b200 import replicas
        dist.barrier()
        ms = replicas.max_over_ranks(ms, device='cuda')
    return ms


def count_launches(fn):
    """kernel launches of one step, split into ours (librelnet_b200.so) and library (cuDNN/cuBLAS/torch) by name."""
    try:
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        ours = lib = 0
        names = {}
        for ev in prof.events():
            if ev.device_type is not None and 'cuda' in str(ev.device_type).lower() and ev.name and 'Memcpy' not in ev.name \
                    and 'Memset' not in ev.name:
                if 'rn::' in ev.name or 'rn_' in ev.name:
                    ours += 1
                    names[ev.name.split('(')[0][:60]] = names.get(ev.name.split('(')[0][:60], 0) + 1
                else:
                    lib += 1
        return ours, lib, names
    except Exception as e:      # profiler unavailable: fall back to the static count of the C ABI call graph
        return None, None, {'error': str(e)}


def _graph_time_us(fn, flush, reps=15):
    """one stage as a captured graph (no host gaps, tensor-map encode outside), 256 MB L2 flush between replays,
    CUDA events, median"""
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for _ in range(3):
            fn()
        s.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            fn()
    torch.cuda.synchronize()
    ts = []
    for i in range(reps):
        flush.fill_(i & 1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); g.replay(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


def _relation_point(ops, synth, device, flush, N, d, H, reps):
    """module and N x M stage microseconds of one (N, d, H) point; the tcgen05 path when it covers the shape"""
    c = synth.make_relation_case(N * 31 + d + H, N, d, H)
    t = [torch.from_numpy(c[k]).to(device) for k in ('X', 'boxes', 'Wq', 'bq', 'Wk', 'bk', 'Wg', 'bg', 'Wout', 'bout')]
    tc = ops.relation_tc_supported(d, d, H)
    rec = dict(N=N, d=d, H=H, dk=d // H, F_tc_gflop=round(4.0 * N * N * d / 1e9, 4))
    if tc:
        ws = torch.empty(ops.relation_workspace_bytes(N, N, d, d, d, H) + 4096, dtype=torch.uint8, device=device)
        kw = dict(group=H, residual_relu=True, precision='f16', workspace=ws)
        ops.relation(*t, **kw)
        rec['path'] = 'tcgen05 fused (geometry + attention, one launch)' if ops.relation_fused_active() else 'tcgen05 unfused'
        rec['module_us'] = round(_graph_time_us(lambda: ops.relation(*t, **kw), flush, reps), 2)
        rec['nm_us'] = round(_graph_time_us(lambda: ops.relation(*t, stage_mask=6, **kw), flush, reps), 2)
        rec['proj_us'] = round(_graph_time_us(lambda: ops.relation(*t, stage_mask=1, **kw), flush, reps), 2)
    else:
        kw = dict(group=H, residual_relu=True, precision='fp32')
        ops.relation(*t, **kw)
        rec['path'] = 'fp32 kernels + library GEMMs (d_k = %d > 64: not covered by the tcgen05 kernels)' % (d // H)
        rec['module_us'] = round(_graph_time_us(lambda: ops.relation(*t, **kw), flush, reps), 2)
        rec['nm_us'] = None
    return rec


def relation_kernel_roofline(ops, pk, device, sweep=True):
    """The fused relation kernel (relation_fused.cu: pair geometry + pair FC + QK^T + softmax + P.V', ONE launch) at the
    headline size N = M = 300, d = 1024, H = 16, timed as a captured graph of that one stage with an L2 flush between
    replays.  achieved = SURVEY 8(d) algorithmic FLOPs 4 N M d / duration against the measured bf16 peak; algorithmic bytes
    by SURVEY 8(d): s (N d + 2 M d) + 16 max(N, M) + 4 (E H + H) + s N d, s = 2.  Also the configs[4] sweep."""
    from relnet_b200 import synth
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)     # > 126 MB L2
    N = M = 300; d = 1024; H = 16; E = 64
    head = _relation_point(ops, synth, device, flush, N, d, H, 25)
    flops = 4.0 * N * M * d
    alg_bytes = int(2 * (N * d + 2 * M * d) + 16 * max(N, M) + 4 * (E * H + H) + 2 * N * d)
    achieved = flops / (head['nm_us'] * 1e-6) / 1e12
    traffic = None          # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this kernel
    try:
        r0 = json.load(open(os.path.join(ROOT, 'profiles', 'r02_ncu_relation_fused_n300.json')))
        traffic = int(r0['dram__bytes_read.sum'] + r0['dram__bytes_write.sum'])
    except Exception:
        pass
    roof = dict(bound='tensor', kernel='relation_fused_kernel (geometry + pair FC + QK^T + softmax + P.V\', one cooperative launch)',
                achieved=round(achieved, 3), peak=pk['tflops'], unit='TFLOP/s', frac=round(achieved / pk['tflops'], 5),
                traffic=traffic, algorithmic_bytes=alg_bytes, algorithmic_flops=flops, duration_us=head['nm_us'],
                timing='captured graph of the one stage, 256 MB L2 flush between replays, CUDA events, median of 25',
                peak_source=pk['source'],
                note='N=M=300: 0.37 GFLOP is ~0.25 us of tensor time; the kernel is latency / SFU bound (per pair 2 log + 16 '
                     'sincos + H exp2 on the XU pipe), see sweep for N up to 3000')
    # companion figure: the unit that actually binds this formulation.  Per pair 2 lg2 + 2 coordinates x 8 frequencies x (sin,
    # cos) (the two size coordinates are separable: per-box tables, no MUFU per pair) and one ex2 per (pair, head), against the
    # XU pipe's 16 results / clk / SM at the SM clock the sampler saw
    def xu_bound(n, h, us, mhz):
        ops_ = float(n) * n * (34 + h)
        peak = 16.0 * 148 * mhz * 1e6
        return dict(N=n, H=h, mufu_ops=ops_, xu_floor_us=round(ops_ / peak * 1e6, 2), measured_us=us,
                    frac_of_xu_peak=round(ops_ / peak / (us * 1e-6), 4))
    roof['xu'] = dict(note='MUFU (XU pipe) floor of the same launch: the contraction alone would take 4NMd / tensor peak',
                      tensor_floor_us=round(flops / (pk['tflops'] * 1e12) * 1e6, 3), at_N300=xu_bound(N, H, head['nm_us'], 1965.0))
    times = dict(module=head['module_us'], nm_stage=head['nm_us'], proj=head['proj_us'])
    sw = None
    if sweep:
        sw = []
        try:
            for n in (100, 300, 1000, 3000):
                for dd in (256, 1024):
                    for hh in (4, 16):
                        rec = head if (n, dd, hh) == (N, d, H) else _relation_point(ops, synth, device, flush, n, dd, hh, 9)
                        if rec.get('nm_us'):
                            ach = rec['F_tc_gflop'] * 1e9 / (rec['nm_us'] * 1e-6) / 1e12
                            rec['nm_tflops'] = round(ach, 2)
                            rec['nm_frac_of_measured_bf16_peak'] = round(ach / pk['tflops'], 4)
                        sw.append(rec)
            big = [r for r in sw if (r['N'], r['d'], r['H']) == (3000, 1024, 16) and r.get('nm_us')]
            if big:
                roof['xu']['at_N3000'] = xu_bound(3000, 16, big[0]['nm_us'], 1965.0)
                traffic3k = None
                try:
                    r3 = json.load(open(os.path.join(ROOT, 'profiles', 'r02_ncu_relation_fused_n3000.json')))
                    traffic3k = int(r3['dram__bytes_read.sum'] + r3['dram__bytes_write.sum'])
                except Exception:
                    pass
                roof['at_N3000'] = dict(duration_us=big[0]['nm_us'], achieved=big[0]['nm_tflops'], frac=big[0]['nm_frac_of_measured_bf16_peak'],
                                        algorithmic_bytes=int(2 * (3000 * 1024 * 3) + 16 * 3000 + 4 * (64 * 16 + 16) + 2 * 3000 * 1024),
                                        traffic=traffic3k)
        except Exception as e:      # the sweep adds keys; the headline roofline above never depends on it
            sw.append({'failed': (str(e).splitlines()[0][:200] if str(e) else type(e).__name__)})
    del flush
    return roof, times, sw


def train_block(args, ts, images, im_info, device, world, rank, dist_on, mode, report=None):
    """Training form of a config: fwd + bwd of `len(images)` images per rank (trunk res3+ by torch/cuDNN autograd, the hot path
    through the C-ABI forward / backward pairs), ONE flat gradient bucket, ONE NCCL SUM allreduce per step, SGD update.
    Reports ms/step (max over ranks), the allreduce's own milliseconds and bus bandwidth, the bucket size.
    Order: the EAGER step is measured first, with the collective's cost and the sum check, and handed to `report` (rank 0 puts
    it into the bench line at once); only then the step is captured as a CUDA graph and measured again."""
    from relnet_b200 import replicas
    from relnet_b200.train import bus_gbs
    import torch.distributed as dist
    K, W = max(3, min(args.steps, 8)), 3
    nbytes = ts.bucket.flat.numel() * 4

    def timed_steps(k):
        torch.cuda.synchronize()
        if dist_on:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        evs = []
        e0.record()
        for _ in range(k):
            evs.append(ts.step(images, im_info))
        e1.record()
        torch.cuda.synchronize()
        ms_ = replicas.max_over_ranks(e0.elapsed_time(e1) / k, device)
        ar_ = replicas.max_over_ranks(sorted(a.elapsed_time(b) for a, b in evs)[len(evs) // 2], device)
        return ms_, ar_

    # ---- eager
    for _ in range(W):
        ts.step(images, im_info)
    eager_ms, eager_ar = timed_steps(max(3, K // 2))
    # the exchange is a SUM: allreduce the bucket of ONE backward and compare it, element by element, with the sum of the
    # ranks' own copies of that same bucket (gathered separately) -- independent of step-to-step atomics / ordering noise
    ts.bucket.zero_()
    for im in images:
        ts.forward_backward(im, im_info)
    ncheck = min(ts.bucket.flat.numel(), 8 << 20)                 # the last 8 Mi elements of the bucket (head + late trunk layers)
    local = ts.bucket.flat[-ncheck:].clone()
    if dist_on:
        parts = [torch.empty_like(local) for _ in range(world)]
        dist.all_gather(parts, local)
        want = torch.zeros_like(local, dtype=torch.float64)
        for q in parts:
            want += q.double()
        del parts
    else:
        want = local.double()
    ts.bucket.allreduce()
    chk = float((ts.bucket.flat[-ncheck:].double() - want).abs().max() / want.abs().max().clamp_min(1e-30))
    del want, local
    # the collective on its own (ranks aligned by a barrier first): what the exchange costs without the arrival skew of the
    # backward that the in-step figure includes
    ms_alone = 0.0
    if dist_on:
        al = []
        for _ in range(5):
            dist.barrier()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); ts.bucket.allreduce(); b.record()
            torch.cuda.synchronize()
            al.append(a.elapsed_time(b))
        ms_alone = replicas.max_over_ranks(sorted(al)[len(al) // 2], device)
    res = dict(mode=mode, images_per_sec=round(world * len(images) / (eager_ms / 1e3), 2), images_per_rank_per_step=len(images),
               ms_per_step=round(eager_ms, 3), allreduce_ms_in_step=round(eager_ar, 4), allreduce_ms=round(ms_alone, 4),
               allreduce_bus_gbs=round(bus_gbs(nbytes, ms_alone, world), 1),
               bucket_mb=round(nbytes / 1e6, 1), collectives_per_step=1 if dist_on else 0, reduce_op='sum (rescale_grad = 1.0)',
               reduced_vs_sum_of_ranks_rel=chk, steps=K, warmup=W, rois=ts.last.get('rois'),
               contractions='forward (general kernels) and backward of the relation / learn-NMS ops on the tcgen05 tf32 GEMM '
                            '(gemm_tf32.cu); no cuBLAS in the hot path',
               launch='eager (torch autograd drives the library trunk and the C-ABI fwd/bwd pairs); allreduce after backward, not overlapped',
               eager_ms_per_step=round(eager_ms, 3),
               losses={k: (round(v, 4) if isinstance(v, float) else v) for k, v in ts.last.items() if k != 'rois'})
    if report:
        report(dict(res))
    # ---- the accumulate phase (zero + fwd + bwd of every micro-batch) as ONE CUDA graph; the allreduce + SGD update follow the replay
    ok, why = 1.0, ''
    try:
        ts.capture(images, im_info)
        torch.cuda.synchronize()
    except Exception as e:           # stay measurable: keep the eager result and say why
        ok, why = 0.0, ' (graph capture failed on this rank: %s)' % (str(e).splitlines()[0][:160] if str(e) else type(e).__name__)
        torch.cuda.synchronize()
    if dist_on:                      # one decision for the whole job: every rank replays the graph, or none does
        flag = torch.tensor([ok], device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if float(flag.item()) < 1.0 and ok == 1.0:
            why = ' (graph capture failed on another rank)'
        ok = float(flag.item())
    if ok < 1.0:
        ts.graph = None
        res['launch'] += why
        return res
    for _ in range(W):
        ts.step(images, im_info)
    ms, ms_ar = timed_steps(K)
    res.update(images_per_sec=round(world * len(images) / (ms / 1e3), 2), ms_per_step=round(ms, 3), allreduce_ms_in_step=round(ms_ar, 4),
               launch='one CUDA-graph replay for the whole forward + backward (library trunk autograd + the C-ABI fwd/bwd pairs), then '
                      'the NCCL allreduce and the SGD update; allreduce after backward, not overlapped')
    return res


def config2_block(args, prec, device, world, dist_on, image32_d, im_info):
    """BASELINE.json configs[2]: Deformable Faster-RCNN 2FC + Relation + LearnNMS, one image per GPU, same timing as the headline
    (resident inputs, one CUDA-graph replay per image)."""
    from relnet_b200.pipeline import DeformableRelationHead, Detector, GraphedStep, init_head_params
    from relnet_b200.trunk import make_trunk
    trunk = make_trunk(device, torch.bfloat16).enable_dcn()
    head = DeformableRelationHead(init_head_params(0, device), precision=prec)
    det = Detector(trunk, head, im_info, dcn=True)
    g = GraphedStep(det, [image32_d])
    steps = max(5, min(args.steps, 30))
    ms = timed(lambda: g(image32_d), steps, 3, dist_on)
    c4 = trunk.c4(image32_d)
    g5 = GraphedStep(lambda c: trunk.c5feat_dcn(c), [c4])
    ms5 = timed(lambda: g5(c4), steps, 3, dist_on)
    return dict(workload='deformable_faster_rcnn_2fc_relation_learnnms_r101_600x1000_n300_h16', images_per_sec=round(world * steps / (ms / 1e3), 2),
                ms_per_step=round(ms / steps, 4), steps=steps, res5_dcn_conv_new_1_ms=round(ms5 / steps, 4),
                note='res5: 3 deformable convs (our channels-last sampler + tcgen05 GEMM, offset convs N(0,0.01)); head: '
                     'DeformablePSROIPooling x2 with the offset FC between (our kernels); rest as configs[1]')


def config3_block(args, prec, device, world, rank, dist_on, train=True, report=None):
    """BASELINE.json configs[3]: FPN 2FC + Relation + LearnNMS.  test: one 608 x 1024 image per GPU, 1000 given rois over four
    pyramid levels, n = 150 (replicas).  train: the data-parallel step -- 2 images per GPU per step accumulated locally, ONE
    NCCL SUM allreduce of the whole gradient bucket (batch 16 on 8 GPUs)."""
    from relnet_b200.pipeline import FPNDetector, FPNRelationHead, GraphedStep, init_head_params
    from relnet_b200.train import FPNTrainStep
    from relnet_b200.trunk import make_fpn_trunk
    g = torch.Generator().manual_seed(1000 + rank)
    image = (torch.randn((1, 3, 608, 1024), generator=g) * 50.0).to(device)
    im_info = torch.tensor([[608.0, 1024.0, 1.0]], device=device)
    trunk = make_fpn_trunk(device, torch.bfloat16)
    head = FPNRelationHead(init_head_params(0, device), precision=prec)
    import numpy as np
    rng = np.random.default_rng(5)
    sz = np.exp(rng.uniform(np.log(16.0), np.log(0.95 * 608), 1000)); ar = np.exp(rng.uniform(np.log(0.5), np.log(2.0), 1000))
    w = np.minimum(sz * np.sqrt(ar), 1022); h = np.minimum(sz / np.sqrt(ar), 606)
    x1 = rng.uniform(0, 1, 1000) * (1023 - w); y1 = rng.uniform(0, 1, 1000) * (607 - h)
    rois = torch.tensor(np.stack([np.zeros(1000), x1, y1, x1 + w, y1 + h], 1), dtype=torch.float32, device=device)
    det = FPNDetector(trunk, head, im_info, rois)
    gs = GraphedStep(det, [image])
    steps = max(5, min(args.steps, 30))
    ms = timed(lambda: gs(image), steps, 3, dist_on)
    feats = trunk(image)
    gh = GraphedStep(lambda *f: head.detect(det.rois_sorted, det.counts, list(f), im_info), list(feats))
    msh = timed(lambda: gh(*feats), steps, 3, dist_on)
    out = dict(workload='fpn_2fc_relation_learnnms_r101_608x1024_n1000_h16_first150',
               test=dict(images_per_sec=round(world * steps / (ms / 1e3), 2), ms_per_step=round(ms / steps, 4), steps=steps,
                         head_ms_per_image=round(msh / steps, 4), rois_per_level=det.counts))
    if report:
        report(dict(out))
    if train:
        del gs, gh, det, head, trunk, feats
        torch.cuda.empty_cache()
        ts = FPNTrainStep(make_fpn_trunk(device, torch.bfloat16), device, num_rois=1000, micro_batches=2, lr=0.0)
        images = [image, (torch.randn((1, 3, 608, 1024), generator=g) * 50.0).to(device)]
        def rep(partial):
            out['train'] = partial
            if report:
                report(dict(out))
        out['train'] = train_block(args, ts, images, im_info, device, world, rank, dist_on,
                                   'configs[3] data-parallel training step: 2 images / GPU / step (batch %d), N = 1000 + G rois, '
                                   'first_n = 150' % (2 * world), report=rep)
        del ts
        torch.cuda.empty_cache()
    return out


def cpu_threads():
    """Host threads for the CPU arm: 16 was the fastest of {8,16,32,64,128} for the torch-CPU trunk on the 128-core B200
    host (128 threads: 30 s/image from oversubscription; tools/cpu_threads_probe.py), and OpenBLAS behaves alike."""
    n = min(16, os.cpu_count() or 1)
    torch.set_num_threads(n)
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=n)
    except Exception:
        pass
    return n


def cpu_baseline(steps=1):
    from oracle import pipeline_np, proposal_np as P
    ncores = cpu_threads()
    from relnet_b200.pipeline import init_head_params
    prm = {k: v.numpy() for k, v in init_head_params(0, 'cpu').items()}
    cls_prob, bbox_pred, info = P.make_proposal_case(0)
    feat = np.maximum(np.random.default_rng(0).standard_normal((1, 256, 38, 63)), 0).astype(np.float32)
    t0 = time.perf_counter()
    for _ in range(steps):
        pipeline_np.head_forward(prm, cls_prob, bbox_pred, feat, info)
    dt = (time.perf_counter() - t0) / steps
    return dict(value=round(1.0 / dt, 4), unit='images/sec', cores=ncores, kind='port',
                sample='hot path only (proposal..learn_nms) of %d image(s), numpy float32 + C oracle; trunk excluded' % steps,
                seconds_per_image=round(dt, 3))


def run_reference(args):
    """CPU arm: torch-CPU fp32 trunk + numpy/C oracle hot path, one image per step, rank 0 only."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from oracle import pipeline_np
    from relnet_b200.pipeline import init_head_params
    from relnet_b200.trunk import make_trunk
    ncores = cpu_threads()
    trunk = make_trunk('cpu', torch.float32)
    prm = {k: v.numpy() for k, v in init_head_params(0, 'cpu').items()}
    image, im_info = make_inputs()
    steps = args.steps; warm = min(args.warmup, 1)       # ~5 s per image on 8 cores

    def step():
        prob, bbox, feat = trunk(image)
        return pipeline_np.head_forward(prm, prob.numpy(), bbox.numpy(), feat.numpy(), im_info.numpy())
    for _ in range(warm):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = step()
    dt = (time.perf_counter() - t0) / steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    v = round(1.0 / dt, 4)
    sample = 'full step (torch-CPU fp32 trunk + numpy/C oracle hot path), %d timed image(s)' % steps
    emit({
        'impl': 'reference', 'metric': 'images/sec', 'value': v, 'unit': 'images/sec', 'n_gpus': args.gpus, 'steps': steps,
        'warmup': warm, 'ms_per_step': round(dt * 1e3, 2), 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'global_batch': 1, 'parallelism': 'cpu'},
        'cpu_baseline': {'value': v, 'unit': 'images/sec', 'cores': ncores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': v, 'unit': 'images/sec', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}})


def require_built():
    """The tree is measured as build() left it, and may be read-only: nothing is compiled here."""
    from relnet_b200 import build
    if not build.current():
        raise RuntimeError('%s is missing or older than its sources: run __graft_entry__.build() first' % build.LIB)


_REAL_STDOUT = None


def emit(obj):
    """the ONE JSON line, on the process's original stdout"""
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(obj) + '\n')
    out.flush()


def main():
    # stdout carries exactly one JSON line: library chatter (e.g. NCCL's "NCCL version ..." banner, make output) is sent
    # to stderr by pointing fd 1 at fd 2 for the whole run and keeping a private handle on the original stdout
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)
    args = parse()
    if args.impl == 'reference':
        return run_reference(args)
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py --impl ours needs a CUDA device (no CPU path in the product)'
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    dist_on = world > 1
    if dist_on:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=device)
    require_built()
    import relnet_b200
    from relnet_b200 import ops
    from relnet_b200.pipeline import RelationHead, init_head_params
    from relnet_b200.trunk import make_trunk

    prec = args.precision or ops.default_precision()
    # cuDNN heuristics by default: the autotuner (RELNET_CUDNN_BENCHMARK=1) times every candidate once and its picks varied
    # from process to process (trunk 0.81 .. 0.90 ms, 851 .. 885 img/s over five runs); the heuristic picks are
    # reproducible (0.867 ms, 876 / 877 img/s on two runs) -- a one-shot measurement should not depend on tuner luck
    torch.backends.cudnn.benchmark = os.environ.get('RELNET_CUDNN_BENCHMARK', '0') == '1'
    # ramp the clocks before anything is timed or tuned
    _a = torch.randn(4096, 4096, device=device, dtype=torch.bfloat16)
    for _ in range(200):
        _a = (_a @ _a).clamp_(-1, 1)
    torch.cuda.synchronize()
    del _a
    trunk = make_trunk(device, torch.bfloat16)
    head = RelationHead(init_head_params(0, device), precision=prec)
    image_h, im_info_h = make_inputs(seed=rank)
    image_pin = image_h.pin_memory()
    image_d = image_h.to(device=device, dtype=torch.bfloat16).contiguous(memory_format=torch.channels_last)
    im_info = im_info_h.to(device)
    out_pin = {'b': torch.empty((100, 80, 4), dtype=torch.float32).pin_memory(),
               's': torch.empty((100, 80), dtype=torch.float32).pin_memory()}

    from relnet_b200.pipeline import GraphedStep, Detector

    full_step = Detector(trunk, head, im_info)   # fp32 NCHW image -> detections; proposal chain || res5 on two streams

    image32_d = image_h.to(device)
    eager_ms = timed(lambda: full_step(image32_d), max(5, args.steps // 2), 3, dist_on)    # un-graphed, for reference
    graphed = GraphedStep(full_step, [image32_d])       # the public fast path: one CUDA-graph replay per image

    def step_resident():
        return graphed(image32_d)

    def step_e2e():
        o = graphed(image_pin)                  # H2D of the pinned host image into the graph's static input, replay
        out_pin['b'].copy_(o['learn_nms_sorted_bbox'], non_blocking=True)
        out_pin['s'].copy_(o['nms_final_score_output'], non_blocking=True)
        torch.cuda.current_stream().synchronize()          # the caller holds the detections on the host
        return o

    from relnet_b200.pipeline import StreamingDetector
    streamer = StreamingDetector(trunk, head, im_info, image32_d, depth=2)
    pending = []

    def step_e2e_stream():
        # the throughput API: image i's H2D / D2H overlap image i-1 / i+1's compute; every image still pays both copies
        pending.append(streamer.submit(image_pin))
        if len(pending) == streamer.depth:
            streamer.collect(pending.pop(0))

    def drain():
        while pending:
            streamer.collect(pending.pop(0))

    trunk_out = trunk(image32_d)
    hot_graph = GraphedStep(lambda a, b, c: head.forward(a, b, c, im_info), list(trunk_out))
    trunk_graph = GraphedStep(lambda im: trunk(im), [image32_d])

    def step_hot():
        return hot_graph(*trunk_out)

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms = timed(step_resident, args.steps, args.warmup, dist_on)
    if sampler:
        sampler.stop_flag = True
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, graphed.out)     # the graph's output buffers: what its last replay returned
    ms_e2e_sync = timed(step_e2e, args.steps, max(3, args.warmup // 2), dist_on)
    ms_e2e = timed(step_e2e_stream, args.steps, max(3, args.warmup // 2), dist_on, after=drain)
    ms_hot = timed(step_hot, args.steps, 3, dist_on)
    ms_trunk = timed(lambda: trunk_graph(image32_d), args.steps, 3, dist_on)

    t_headline = time.time()                 # every rank leaves the last timed() together (barrier + max-reduce inside)
    del streamer, graphed, hot_graph, trunk_graph
    torch.cuda.empty_cache()

    # ---- rank 0: everything the contract line needs, BEFORE the optional blocks (they only add keys to it)
    line = None
    if rank == 0:
        pk = peaks()
        ours, lib, names = count_launches(lambda: full_step(image32_d))
        roof, rel_times, sweep = (None, {}, None)
        if ops.device_info()['sm100'] and prec == 'f16':
            try:
                roof, rel_times, sweep = relation_kernel_roofline(ops, pk, device, sweep=not args.no_sweep)
            except Exception as e:      # reported in the line; the headline value does not depend on the single-kernel timing
                roof = {'failed': (str(e).splitlines()[0][:200] if str(e) else type(e).__name__)}
                torch.cuda.synchronize()
        line = {
            'metric': 'images/sec', 'value': round(world * args.steps / (ms / 1e3), 3), 'unit': 'images/sec',
            'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': round(ms / args.steps, 4),
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f16' if prec == 'f16' else 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'global_batch': world, 'parallelism': 'replicas x%d (1 image/GPU)' % world, 'launch': 'one CUDA-graph replay per image',
                       'trunk': 'ResNet-101 convolutions on cuDNN (bf16 channels_last, fused conv+bias+relu calls; library, out of scope) with our '
                                'space-to-depth stem input, max-pool and RPN-head (bf16 tcgen05 GEMM) kernels around them',
                       'hot_path_precision': prec, 'l2': 'inputs (7.2 MB image) + 180 MB of trunk activations per step '
                       'exceed the 126 MB L2; relation kernel timed with an explicit 256 MB L2 flush'},
            'e2e': {'value': round(world * args.steps / (ms_e2e / 1e3), 3), 'unit': 'images/sec',
                    'h2d_bytes_per_step': int(image_pin.numel() * 4), 'd2h_bytes_per_step': int(100 * 80 * 5 * 4),
                    'api': 'pipeline.StreamingDetector (2 slots in flight: each image pays its own H2D + D2H, overlapped with '
                           'the neighbouring images\' compute)',
                    'one_image_at_a_time': round(world * args.steps / (ms_e2e_sync / 1e3), 3)},
            'gpu_launches': (ours or 0) * args.steps, 'gpu_launches_per_step': ours, 'library_launches_per_step': lib,
            'hot_path': {'ms_per_image': round(ms_hot / args.steps, 4), 'images_per_sec': round(args.steps / (ms_hot / 1e3), 2),
                         'trunk_ms_per_image': round(ms_trunk / args.steps, 4),
                         'eager_ms_per_step_no_graph': round(eager_ms / max(5, args.steps // 2), 4),
                         'relation_module_us': {k: round(v, 2) for k, v in rel_times.items()},
                         'proposals_kept_before_pad': int(ops.proposal(trunk_out[0], trunk_out[1], im_info, return_num_kept=True, **head.cfg)[2].item())},
            'clocks': sampler.summary() if sampler else None,
            'roofline': roof,
            'train': None,
            'configs': {'2_deformable_faster': None, '3_fpn': None},
            'sweep': sweep,
        }
        if not args.no_cpu_baseline and world == 1:          # the contract asks for it on rank 0 at N=1 only
            line['cpu_baseline'] = cpu_baseline()
        line['kernels'] = names

    # ---- optional blocks: configs[2] / configs[3] and the data-parallel training steps (the one collective of the path).  They run
    # under a deadline counted from the end of the headline measurement: if it passes (a slow or stuck collective, host contention
    # with 8 processes ...) every rank stops there and rank 0 prints the line it already has -- the headline never depends on them.
    done = threading.Event()
    emit_lock = threading.Lock()

    def bail():
        with emit_lock:
            if not done.is_set():
                done.set()
                if rank == 0 and line is not None:
                    line['extras'] = 'stopped at the %.0f s deadline (--extras-budget); blocks finished until then are in the line' % args.extras_budget
                    emit(line)
        os._exit(0)
    # every rank leaves at (nearly) the same moment, rank 0 a little earlier so that its line is out before any peer can notice a
    # missing process
    t_deadline = t_headline + args.extras_budget + (0.0 if rank == 0 else 1.5)
    timer = threading.Timer(max(5.0, t_deadline - time.time()), bail)
    timer.daemon = True
    timer.start()

    def put(key, sub, val):
        if line is not None:
            if sub is None:
                line[key] = val
            else:
                line[key][sub] = val

    def guarded(fn):
        try:
            return fn()
        except Exception as e:       # a failed optional block is reported, not fatal (collectives stay symmetric inside the blocks)
            msg = (str(e).splitlines()[0][:200] if str(e) else type(e).__name__)
            try:
                torch.cuda.synchronize()
            except Exception as e2:  # a sticky device error: nothing further can run on this rank, the line still goes out
                raise RuntimeError('%s; device unusable afterwards (%s)' % (msg, str(e2).splitlines()[0][:120] if str(e2) else type(e2).__name__))
            return {'failed': msg}
    # cheap replica block first, then the training step of configs[1] (the one collective of the path; its eager result enters the
    # line before graph capture is attempted), then configs[3]
    try:
        if not args.no_configs and prec == 'f16':
            put('configs', '2_deformable_faster', guarded(lambda: config2_block(args, prec, device, world, dist_on, image32_d, im_info)))
            torch.cuda.empty_cache()
        if not args.no_train:
            def cfg1_train():
                from relnet_b200.train import TrainStep
                ts = TrainStep(make_trunk(device, torch.bfloat16, seed=0), device, micro_batches=1, lr=0.0)
                timg, _ = make_inputs(seed=100 + rank)
                return train_block(args, ts, [timg.to(device)], im_info, device, world, rank, dist_on,
                                   'configs[1] data-parallel training step, 1 image / GPU / step', report=lambda r: put('train', None, r))
            put('train', None, guarded(cfg1_train))
            torch.cuda.empty_cache()
        if not args.no_configs and prec == 'f16':
            put('configs', '3_fpn', guarded(lambda: config3_block(args, prec, device, world, rank, dist_on, train=not args.no_train,
                                                                    report=lambda r: put('configs', '3_fpn', r))))
            torch.cuda.empty_cache()
    except BaseException as e:       # whatever escapes the optional blocks on any rank must not cost the job its headline line:
        # this rank stops here; rank 0 prints what it has, the others leave with status 0 (peers still inside a collective are
        # released by their own deadline)
        sys.stderr.write('bench.py: optional blocks aborted on rank %d: %s\n' % (rank, (str(e).splitlines()[0][:300] if str(e) else type(e).__name__)))
        if line is not None:
            line['extras'] = 'aborted: %s' % (str(e).splitlines()[0][:200] if str(e) else type(e).__name__)
        with emit_lock:
            if not done.is_set():
                done.set()
                if rank == 0 and line is not None:
                    emit(line)
        sys.stdout.flush(); sys.stderr.flush()
        if dist_on:                  # leave together with the peers (at the deadline), not before them: a process that disappears
            time.sleep(max(0.0, t_deadline - time.time()) + 5.0)     # while the others sit in a collective turns a reported failure into a job abort
        os._exit(0)
    with emit_lock:                  # exactly once: either this or bail() prints the line
        timer.cancel()
        if not done.is_set():
            done.set()
            if rank == 0:
                emit(line)
    if dist_on:
        import torch.distributed as dist
        try:
            dist.barrier()
            dist.destroy_process_group()
        except Exception:
            pass


if __name__ == '__main__':
    main()
