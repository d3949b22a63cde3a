#!/usr/bin/env python
"""
bench.py - BASELINE.json metric: line-images/s (48 px height) of the rpred hot path on N B200s.

Workload (config.workload "cfg2"): VGSL [1,48,0,1 Cr3,3,32 Mp2,2 Cr3,3,64 Mp2,2 S1(1x0)1,3 Lbx256 O1c200], random-init
weights (reference init distributions), one step = ONE batch of 64 synthetic 48x800 lines through
`kb_recognize` (net -> softmax -> arg-max -> CTC collapse -> label tuples on the host).

  value  lines/s with the line batches already resident in HBM, K steps through the asynchronous pipeline (kb_recognize_async / kb_wait:
         `--inflight` batches in flight on ONE handle from ONE host thread), decoded labels returned to the host.
  serial the same K steps one synchronous kb_recognize at a time, per-stage CUDA events on (the source of `roofline`).
  e2e    the pipeline with pinned HOST buffers: H2D of the 64x48x800 fp32 batch and D2H of the label block are inside the timed region
         (e2e_u8: uint8 lines, a quarter of the bytes; scale / invert / pad on the device).
  roofline      the dominant kernel stage of the serial step, timed with CUDA events on the launching stream inside the timed region
                (kb_set_timing), against MEASURED_PEAKS.json; per-stage fractions beside it.
  cfg5 / cfg3   side measurements (BASELINE configs[4] and [2]) in the same line.
  cpu_baseline  the oracle (torch-CPU restatement of the reference, `kind: "port"`; the reference is a Python package
                whose dependencies are not installed on the GPU box) on all host cores, bounded sample.
  --impl reference   times that same CPU implementation as its own arm.

N > 1 (torchrun): line batches shard embarrassingly - every rank runs its own replica on its own shard (weak
scaling, fixed 64 lines per step per GPU); weights are broadcast once from rank 0 over NCCL before the timed
region and the decoded label blocks of all steps are gathered to rank 0 once at its end.
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

import numpy as np
import torch

CFG2 = '[1,48,0,1 Cr3,3,32 Mp2,2 Cr3,3,64 Mp2,2 S1(1x0)1,3 Lbx256 O1c200]'
BATCH, HEIGHT, WIDTH, NCLS = 64, 48, 800, 200
CPU_NOTE = ''
METRIC = 'line-images/sec (48px height)'
UNIT = 'lines/s'


# ---------------------------------------------------------------------------------------------------------
# algorithmic work per line (SURVEY.md 8d; DESIGN.md "roofline accounting")
# ---------------------------------------------------------------------------------------------------------
def stage_work(W=WIDTH):
    w2, T = W // 2, (W // 2) // 2
    f = 4  # fp32 bytes
    return {  # stage -> (FLOPs per line, algorithmic HBM bytes per line = unique input + output of the stage)
        'C_0': (2 * 48 * W * 32 * 9, f * (48 * W + 48 * W * 32)),
        'Mp_1': (0, f * (48 * W * 32 + 24 * w2 * 32)),
        'C_2': (2 * 24 * w2 * 64 * 288, f * (24 * w2 * 32 + 24 * w2 * 64)),
        'Mp_3': (0, f * (24 * w2 * 64 + 12 * T * 64)),
        'S_4': (0, f * 2 * 768 * T),
        'L_5.xproj': (2 * T * 768 * 2048, f * (768 * T + 2048 * T)),
        'L_5.rec': (2 * T * 2 * 1024 * 256, f * (2048 * T + 512 * T)),
        'O_6': (2 * T * 512 * 200, f * (512 * T + 200 * T)),
        'decode': (0, f * (200 * T) + 16 * T),
        # fused groups: same FLOPs, only the group's external input and output touch HBM (4 bytes per element: one fp32 tensor or,
        # equivalently, the two fp16 operand planes the tensor-core consumer reads)
        'C_0+Mp_1': (2 * 48 * W * 32 * 9, f * (48 * W + 24 * w2 * 32)),
        'C_2+Mp_3+S_4': (2 * 24 * w2 * 64 * 288, f * (24 * w2 * 32 + 768 * T)),
    }


def per_stage_roofline(per_stage_ms, work, pk, batch):
    """stage -> achieved TFLOP/s and GB/s on the algorithmic work of `stage_work`, and both as fractions of the measured peaks
    (SURVEY 8d: report both fractions per kernel; the binding one is the larger)."""
    out = {}
    for k, ms in per_stage_ms.items():
        if k not in work or ms <= 0:
            continue
        fl, by = work[k][0] * batch, work[k][1] * batch
        tf, gbs = fl / (ms * 1e-3) / 1e12, by / (ms * 1e-3) / 1e9
        out[k] = {'ms': round(ms, 4), 'tflops': round(tf, 2), 'gbs': round(gbs, 1), 'tensor_frac': round(tf / pk['tf_sustained'], 4),
                  'hbm_frac': round(gbs / pk['hbm_gbs'], 4)}
    return out


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return {'hbm_gbs': d['hbm_gbs'], 'tf_burst': d['bf16_tflops'], 'tf_sustained': d['bf16_tflops_sustained'], 'src': 'measured'}
    return {'hbm_gbs': 6650.0, 'tf_burst': 1590.0, 'tf_sustained': 1400.0, 'src': 'fallback'}


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region (B200_PROFILING.md).  In-process NVML polling every 10 ms (nvidia_ml_py):
    an `nvidia-smi -lms` child, as used first, kept the driver busy enough to stretch the serial multi-GPU steps by ~0.15 ms;
    nvidia-smi stays as the fallback when NVML cannot be loaded."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
    BITS = {'sw_power_cap': 0x4, 'hw_slowdown': 0x8, 'sw_thermal_slowdown': 0x20, 'hw_thermal_slowdown': 0x40}

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.nvml, self.h, self.samples, self.stop_flag = None, None, [], False

    def _nvml_index(self):
        cvd = os.environ.get('CUDA_VISIBLE_DEVICES', '')
        try:
            ids = [int(x) for x in cvd.split(',') if x.strip() != '']
            return ids[self.index] if ids else self.index
        except (ValueError, IndexError):
            return self.index

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._nvml_index())
            self.nvml = pynvml
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100',
                                          '-i', str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)
                mx = n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)
                rs = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((float(sm), float(mx), int(rs)))
            except Exception:
                pass
            time.sleep(0.01)

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.th.join(timeout=1)
            sm = [s_[0] for s_ in self.samples]; mx = [s_[1] for s_ in self.samples]
            reasons = sorted(k for k, bit in self.BITS.items() if any(s_[2] & bit for s_ in self.samples))
            return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons,
                    'samples': len(sm), 'source': 'nvml'}
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm), 'source': 'nvidia-smi'}


def make_batches(count, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.rand(BATCH, 1, HEIGHT, WIDTH, generator=g) for _ in range(count)]


def oracle_model(seed=0):
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import vgsl_oracle as vo
    om = vo.OracleModel(CFG2)
    w = om.init_like_reference(seed)
    return vo, om, w


def usable_cpus():
    """Cores this process may actually use: affinity mask capped by the cgroup CPU quota (a 128-thread pool on a
    quota-limited container is 50x slower than the right size)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ('/sys/fs/cgroup/cpu.max', '/sys/fs/cgroup/cpu/cpu.cfs_quota_us'):
        try:
            txt = open(path).read().split()
            if path.endswith('cpu.max'):
                if txt[0] != 'max':
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                per = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
                if q > 0:
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except Exception:
            continue
    return max(1, n)


def pick_threads(vo, om):
    """Gives the CPU arm its best shot: tries a few intra-op thread counts on a small sample and keeps the fastest."""
    n = usable_cpus()
    cands = sorted({c for c in (n, n // 2, 64, 32, 16, 8) if 1 <= c <= n}, reverse=True)
    g = torch.Generator().manual_seed(5)
    x = torch.rand(16, 1, HEIGHT, 400, generator=g)
    lens = torch.full((16,), 400, dtype=torch.long)
    best, best_t, tried = cands[-1], float('inf'), {}
    t_start = time.perf_counter()
    for c in cands:
        torch.set_num_threads(c)
        vo.rec_predict(om, x[:4], lens[:4])                    # thread-pool warm-up
        t0 = time.perf_counter()
        vo.rec_predict(om, x, lens)
        dt = time.perf_counter() - t0
        tried[c] = round(dt, 3)
        if dt < best_t:
            best, best_t = c, dt
        if time.perf_counter() - t_start > 40:
            break
    return best, n, tried


def time_cpu(steps, warmup, threads=None):
    """The reference's CPU path for one step: nn(x, lens) + softmax + greedy_decoder on a batch of 64 (rpred.py:225-228)."""
    vo, om, _ = oracle_model()
    global CPU_NOTE
    if threads is None:
        threads, avail, tried = pick_threads(vo, om)
        CPU_NOTE = f'usable cores {avail} (os.cpu_count {os.cpu_count()}); thread-count probe s/16-line sample {tried}'
    torch.set_num_threads(threads)
    xs = make_batches(2, 100)
    lens = torch.full((BATCH,), WIDTH, dtype=torch.long)
    for i in range(warmup):
        vo.rec_predict(om, xs[i % 2], lens)
    t0 = time.perf_counter()
    for i in range(steps):
        vo.rec_predict(om, xs[i % 2], lens)
    dt = time.perf_counter() - t0
    return BATCH * steps / dt, dt / steps * 1e3, threads


def cpu_model_name():
    try:
        for ln in open('/proc/cpuinfo'):
            if ln.startswith('model name'):
                return ln.split(':', 1)[1].strip()
    except Exception:
        pass
    return 'unknown'


def run_reference_arm(args, rank):
    if rank != 0:
        return
    lps, ms, threads = time_cpu(args.steps, args.warmup)
    line = {'impl': 'reference', 'metric': METRIC, 'value': lps, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': 'cfg2', 'spec': CFG2, 'batch_per_gpu': BATCH, 'global_batch': BATCH * args.gpus, 'line': f'{HEIGHT}x{WIDTH}'},
            'notes': {'device': 'host CPU (rank 0 only)'},
            'cpu_baseline': {'value': lps, 'unit': UNIT, 'cores': threads, 'kind': 'port', 'cpu': cpu_model_name(),
                             'sample': f'{args.steps} batches of {BATCH} lines {HEIGHT}x{WIDTH} after {args.warmup} warm-up; '
                                       'torch-CPU restatement of the reference path (oracle/vgsl_oracle.py), fp32; ' + CPU_NOTE},
            'e2e': {'value': lps, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


BLLA = ('[1,1800,0,3 Cr7,7,64,2,2 Gn32 Cr3,3,128,2,2 Gn32 Cr3,3,128 Gn32 Cr3,3,256 Gn32 Cr3,3,256 Gn32 '
        'Lbx32 Lby32 Cr1,1,32 Gn32 Lby32 Lbx32 O2l4]')


def run_cfg3(args):
    """BASELINE configs[2]: blla.mlmodel architecture, 2400x3200 pages (-> 3x1800x1350 net input), batch 8, 1 GPU:
    nn -> nearest upsample to the input size -> sigmoid (`kb_segment`).  Reports pages/s next to the oracle on the CPU."""
    import __graft_entry__ as ge
    ge.build()
    import kraken_b200 as kb
    from kraken_b200.blla import segmentation_heatmap
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import vgsl_oracle as vo
    N, H, W = args.pages, 1800, 1350
    om = vo.OracleModel(BLLA)
    w = om.init_like_reference(3)
    m = kb.TorchVGSLModel(vgsl=BLLA, model_type=['segmentation'])
    m.load_state_dict(w)
    m.to('cuda:0')
    g = torch.Generator().manual_seed(3)
    pages = [torch.rand(N, 3, H, W, generator=g).cuda() for _ in range(2)]
    for i in range(max(2, args.warmup)):
        segmentation_heatmap(m, pages[i % 2], (H, W))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    m.reset_launch_count()
    e0.record()
    for i in range(args.steps):
        hm = segmentation_heatmap(m, pages[i % 2], (H, W))
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    launches = int(m.launch_count)
    # end to end through the public call with HOST tensors (pinned pages in, heat maps out to host memory), strictly serial
    hpages = [p_.cpu().pin_memory() for p_ in pages]
    segmentation_heatmap(m, hpages[0], (H, W))
    sampler = ClockSampler(0)
    sampler.start()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(args.steps):
        hm_host = segmentation_heatmap(m, hpages[i % 2], (H, W))
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    clocks = sampler.stop()
    # per-stage times from a separate pass (the stage timers put event pairs around every layer)
    stage = {}
    m.set_timing(True)
    for i in range(args.steps):
        segmentation_heatmap(m, pages[i % 2], (H, W))
        for k, v in m.last_timing():
            stage[k] = stage.get(k, 0.0) + v
    m.set_timing(False)
    cpu = None
    if not args.no_cpu_baseline:
        torch.set_num_threads(usable_cpus())
        x1 = pages[0][:1].cpu()
        vo.seg_heatmap(om, x1, (H, W))
        t0 = time.perf_counter()
        for _ in range(2):
            vo.seg_heatmap(om, x1, (H, W))          # the reference never batches pages (spred.py:268)
        cpu = {'value': 2 / (time.perf_counter() - t0), 'unit': 'pages/s', 'cores': usable_cpus(), 'kind': 'port', 'cpu': cpu_model_name(),
               'sample': '2 pages 3x1800x1350 after 1 warm-up, oracle seg_heatmap (nn + interpolate + sigmoid), batch 1'}
    flops = 390.9e9 * N
    line = {'metric': 'pages/sec (blla forward, 2400x3200 pages)', 'value': N / (ms / 1e3), 'unit': 'pages/s', 'n_gpus': 1, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic', 'config': {'workload': 'cfg3', 'spec': BLLA, 'batch': N, 'page': f'3x{H}x{W}', 'heatmap': f'4x{H}x{W}'},
            'e2e': {'value': N / (e2e_ms / 1e3), 'unit': 'pages/s', 'ms_per_step': e2e_ms, 'h2d_bytes_per_step': N * 3 * H * W * 4,
                    'd2h_bytes_per_step': int(hm_host.numel()) * 4, 'api': 'kraken_b200.blla.segmentation_heatmap -> kb_segment, host pages in, host heat maps out'},
            'clocks': clocks,
            'gpu_launches': launches, 'stages_ms': {k: round(v / args.steps, 3) for k, v in stage.items()},
            'whole_step_tflops_fp32_equiv': flops / (ms / 1e3) / 1e12, 'cpu_baseline': cpu,
            'heatmap_range': [float(hm.min()), float(hm.max())]}
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, blocks):
    """Writes the label blocks one step of the timed path returned (`TorchSeqRecognizer.collect`: counts, labels, starts, ends,
    confs) as DIR/<name>.npy, integers as float64 and confidences as float32.  The engine leaves the slots past a line's count
    unwritten, so they are zeroed: two runs on the same inputs then compare element for element."""
    os.makedirs(out_dir, exist_ok=True)
    valid = np.arange(blocks['labels'].shape[1])[None, :] < blocks['counts'][:, None]
    for name, a in blocks.items():
        if a.ndim == 2:
            a = np.where(valid, a, 0)
        np.save(os.path.join(out_dir, name + '.npy'), a.astype(np.float32 if name == 'confs' else np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None, help='timed steps (default: 200 on the GPU arm, 20 CPU batches on the reference arm)')
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--cpu-steps', type=int, default=6)
    ap.add_argument('--inflight', type=int, default=6, help='pipeline slots (batches in flight from the one host thread) of the e2e arm')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-numa-bind', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the cfg3 / cfg5 side measurements')
    ap.add_argument('--workload', default='cfg2', choices=['cfg2', 'cfg3'])
    ap.add_argument('--pages', type=int, default=8)
    ap.add_argument('--cfg5-lines', type=int, default=100000)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the label blocks of the last timed `value` step (rank 0) to DIR/<name>.npy (cfg2 GPU arm only)')
    args = ap.parse_args()
    if args.dump_outputs is not None and (args.impl != 'b200' or args.workload != 'cfg2'):
        ap.error('--dump-outputs applies to the cfg2 workload of the GPU arm')
    if args.steps is not None and args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    if args.steps is None:
        args.steps = 200 if (args.impl == 'b200' and args.workload == 'cfg2') else 20
    # a hung kernel or a lost pipeline ticket must not sit on the GPU box until its time limit: dump every thread's stack and exit
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get('KB_BENCH_WATCHDOG', '1200')), exit=True)

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference_arm(args, rank)
        return
    if args.workload == 'cfg3':
        if rank == 0:
            run_cfg3(args)
        return

    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    import torch.distributed as dist
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group('nccl', device_id=torch.device(f'cuda:{local}'))
        dist.barrier()
    import kraken_b200 as kb
    from kraken_b200.dist import ResultBlocks, bind_to_gpu_numa, recognize_sharded_blocks
    dev = f'cuda:{local}'
    # bind this rank (its threads and the pinned staging buffers it is about to first-touch) to the cores of its GPU's NUMA node:
    # round 1 lost 40 % of the 8-GPU end-to-end rate to ranks feeding their GPU across the socket interconnect
    numa_cores = bind_to_gpu_numa(local) if not args.no_numa_bind else None
    torch.cuda.set_device(local)

    # ---- weights: rank 0 initialises, one NCCL broadcast of the packed blob, every rank loads its replica
    m = kb.TorchVGSLModel(vgsl=CFG2, model_type=['recognition'])
    if rank == 0:
        _, _, w = oracle_model(0)                        # same seeded weights the parity tests use
        m.load_state_dict(w)
    if world > 1:
        from kraken_b200.dist import broadcast_state_dict
        m.load_state_dict(broadcast_state_dict(m.state_dict(), src=0, device=torch.device(dev)))
    rec = kb.TorchSeqRecognizer(m, device=dev)
    lens = torch.full((BATCH,), WIDTH, dtype=torch.long)
    # end-to-end arm: ONE engine handle with DEPTH pipeline slots (own stream + workspace each, one copy of the weights) fed by ONE
    # host thread through kb_recognize_async / kb_wait: the H2D copy, the kernels and the D2H read-back of consecutive batches overlap,
    # and the thread sleeps on a blocking CUDA event while it waits - how a serving loop would run it
    DEPTH = max(1, min(args.inflight, 16))
    rec.set_pipeline_depth(DEPTH)

    NB = 4                                               # distinct input batches rotated through the steps
    host = [b.pin_memory() for b in make_batches(NB, 1000 + rank)]
    devb = [b.to(dev) for b in host]
    # the same kind of lines as uint8 crops (SURVEY 8f rank 1): scale / invert / pad run on the device inside kb_recognize_u8
    host_u8 = [(b * 255).to(torch.uint8).pin_memory() for b in host]
    inv255 = np.full(BATCH, 255, np.int16)
    T = WIDTH // 4

    def step(x, out=None):
        return rec._recognize_raw(x, lens, want_probs=False, out=out)     # the ABI's own output blocks (labels, starts, ends, confs, counts)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # result blocks of a run in ONE pinned int32 buffer (kraken_b200.dist.ResultBlocks): every engine call writes its output blocks
    # straight into its slice, the run's single gather to rank 0 ships the buffer as it is (no host-side repacking)
    blocks = {}

    def run_blocks(steps):
        if steps not in blocks:
            blocks[steps] = ResultBlocks(steps, BATCH, T)
        return blocks[steps]

    def run_pipelined(batches, steps, u8=False):
        rb = run_blocks(steps)
        pend = []
        for i in range(steps):
            if len(pend) == DEPTH:
                j, t = pend.pop(0)
                rec.collect(t, out=rb.views(j))
            pend.append((i, rec.submit(batches[i % NB], lens, inv255 if u8 else None)))
        while pend:
            j, t = pend.pop(0)
            rec.collect(t, out=rb.views(j))
        return rb

    def timed(batches, steps, on_step=None, pipelined=False, u8=False):
        run_blocks(steps)                                  # the pinned result buffer of a run is allocated outside its timed region
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if pipelined:
            rb = run_pipelined(batches, steps, u8)
        else:
            rb = run_blocks(steps)
            for i in range(steps):
                step(batches[i % NB], rb.views(i))
                if on_step is not None:
                    on_step()
        if world > 1:
            got = rb.gather(0, torch.device(dev))          # the single gather of the run's decoded label sequences to rank 0 over NCCL
            if rank == 0:
                assert len(got) == world and got[0].shape[0] == steps
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), rb

    for i in range(args.warmup):
        step(devb[i % NB]); step(host[i % NB])
    run_pipelined(host, 2 * DEPTH)
    run_pipelined(host_u8, 2 * DEPTH, u8=True)
    run_pipelined(devb, 2 * DEPTH)
    if world > 1:
        run_blocks(args.steps).gather(0, torch.device(dev))      # warm the NCCL gather up at the payload size of the timed runs
        ms_warm = torch.zeros(1, device=dev); dist.all_reduce(ms_warm, op=dist.ReduceOp.MAX)

    # ---- timed region 1 (strictly serial, one synchronous kb_recognize per step): per-stage CUDA-event timing on the launching stream
    m.set_timing(True)
    stage_ms = {}

    def on_step():
        for name, ms in m.last_timing():
            stage_ms[name] = stage_ms.get(name, 0.0) + ms

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    m.reset_launch_count()
    ms_serial, _ = timed(devb, args.steps, on_step)
    launches_serial = m.launch_count
    m.set_timing(False)
    # ---- timed region 2: `value` - the same K steps, inputs resident in HBM, through the asynchronous pipeline (one host thread)
    m.reset_launch_count()
    ms_total, rb_value = timed(devb, args.steps, pipelined=True)
    launches = m.launch_count
    # the e2e regions below write into the same result buffer: keep what the last `value` step returned
    last_value = {k: v.copy() for k, v in rb_value.views(args.steps - 1).items()}
    # ---- timed region 3: end to end through the public API with pinned host buffers
    ms_e2e_serial, _ = timed(host, args.steps)
    ms_e2e, _ = timed(host, args.steps, pipelined=True)
    ms_e2e_u8, _ = timed(host_u8, args.steps, pipelined=True, u8=True)
    clocks = sampler.stop() if rank == 0 else None
    decoded_last = int(rb_value.views(args.steps - 1)['counts'].sum())

    # ---- cfg5 (BASELINE configs[4]): 100 000 synthetic 48 x 1200 lines sharded over the ranks (strong scaling), lines generated on the
    # device per shard, through kraken_b200.dist.recognize_sharded_blocks: asynchronous pipeline per rank + ONE gather at the end
    cfg5 = None
    if not args.no_extra:
        W5, T5, TOTAL5 = 1200, 300, args.cfg5_lines
        nb_total = (TOTAL5 + BATCH - 1) // BATCH
        nb_mine = (nb_total + world - 1) // world            # every rank runs the same number of batches (the last ones may be surplus)
        g5 = torch.Generator(device=dev).manual_seed(2 + rank)
        dev5 = [torch.rand(BATCH, 1, HEIGHT, W5, generator=g5, device=dev) for _ in range(NB)]
        lens5 = torch.full((BATCH,), W5, dtype=torch.long)
        my5 = [(dev5[i % NB], lens5) for i in range(nb_mine)]
        rb5 = ResultBlocks(nb_mine, BATCH, T5)
        recognize_sharded_blocks(rec, my5[:2 * DEPTH], T5, depth=DEPTH, device=torch.device(dev) if world > 1 else None, blocks=ResultBlocks(2 * DEPTH, BATCH, T5))
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        recognize_sharded_blocks(rec, my5, T5, depth=DEPTH, device=torch.device(dev) if world > 1 else None, blocks=rb5)
        e1.record()
        barrier()
        ms5 = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms5, op=dist.ReduceOp.MAX)
        ms5 = float(ms5.item())
        lines5 = nb_mine * world * BATCH
        cfg5 = {'workload': 'cfg5', 'lines': lines5, 'line': f'{HEIGHT}x{W5}', 'scaling': 'strong', 'ms_total': ms5, 'value': lines5 / (ms5 / 1e3), 'unit': UNIT,
                'batches_per_rank': nb_mine, 'in_flight': DEPTH, 'decoded_labels_last_batch': int(rb5.views(nb_mine - 1)['counts'].sum()),
                'api': 'kraken_b200.dist.recognize_sharded_blocks: device-resident shard -> kb_recognize_async/kb_wait -> one NCCL gather of the label blocks'}
        del dev5, my5, rb5

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    if args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, last_value)

    pk = peaks()
    work = stage_work()
    T_ = T
    ms_step = ms_total / args.steps
    value = world * BATCH * args.steps / (ms_total / 1e3)
    e2e = world * BATCH * args.steps / (ms_e2e / 1e3)
    per_stage = {k: v / args.steps for k, v in stage_ms.items()}
    dom = max((k for k in per_stage if k in work), key=lambda k: per_stage[k])
    flops, byts = work[dom][0] * BATCH, work[dom][1] * BATCH
    t_tensor, t_hbm = flops / (pk['tf_sustained'] * 1e12), byts / (pk['hbm_gbs'] * 1e9)
    dur = per_stage[dom] / 1e3
    if t_tensor >= t_hbm:
        roof = {'bound': 'tensor', 'achieved': flops / dur / 1e12, 'peak': pk['tf_sustained'], 'unit': 'TFLOP/s'}
    else:
        roof = {'bound': 'hbm', 'achieved': byts / dur / 1e9, 'peak': pk['hbm_gbs'], 'unit': 'GB/s'}
    # measured DRAM bytes per launch of that kernel from the committed `ncu --set full` capture of this same command (profiles/); null if
    # the capture is missing
    traffic = None
    for tf_name in ('r02_ncu_dram_bytes_per_launch.json', 'r01d_ncu_dram_bytes_per_launch.json'):
        try:
            with open(os.path.join(ROOT, 'profiles', tf_name)) as fh:
                tj = json.load(fh)
            kmap = {'L_5.rec': ('k_lstm_rec_tc<8>', 0), 'L_5.xproj': ('k_gemm_tc<', 0), 'O_6': ('k_gemm_tc<', 1),
                    'C_2+Mp_3+S_4': ('k_conv_tc', 0), 'C_0+Mp_1': ('k_conv1_', 0)}
            if dom in kmap:
                hits = [v for k_, v in tj.items() if kmap[dom][0] in k_]
                if hits:
                    traffic = float(hits[0][min(kmap[dom][1], len(hits[0]) - 1)])
                    break
        except (OSError, ValueError, IndexError, KeyError, TypeError):
            continue
    roof.update({'frac': roof['achieved'] / roof['peak'], 'traffic': traffic, 'kernel': dom, 'kernel_ms': per_stage[dom],
                 'share_of_serial_step': per_stage[dom] / (ms_serial / args.steps),
                 'peak_source': pk['src'] + (' (sustained bf16 GEMM)' if roof['bound'] == 'tensor' else ' (copy bandwidth)'),
                 'algorithmic_per_launch': {'flops': flops, 'bytes': byts},
                 'timed': 'per-stage CUDA events on the launching stream inside the strictly serial timed region (kb_set_timing)',
                 'stages_ms': {k: round(v, 4) for k, v in per_stage.items()},
                 'per_stage': per_stage_roofline(per_stage, work, pk, BATCH)})
    tot_f = sum(work[k][0] for k in per_stage if k in work) * BATCH          # only the stages that actually ran (fused groups replace their members)
    tot_b = (4 * 48 * WIDTH + 2 * 4 * 768 * T_ + 2 * 4 * 2048 * T_ + 2 * 4 * 512 * T_ + 8 * T_) * BATCH

    def whole(ms):
        return {'tensor_frac': tot_f / (ms / 1e3) / (pk['tf_sustained'] * 1e12), 'hbm_frac': tot_b / (ms / 1e3) / (pk['hbm_gbs'] * 1e9)}
    roof['whole_step'] = {'serial': whole(ms_serial / args.steps), 'pipelined_value': whole(ms_step * world), 'pipelined_e2e': whole(ms_e2e / args.steps * world),
                          'algorithmic_per_step': {'flops': tot_f, 'bytes': tot_b}}
    if cfg5 is not None:
        f5 = (2 * 48 * 1200 * 32 * 9 + 2 * 24 * 600 * 64 * 288 + 300 * (2 * 2 * 1024 * 768 + 2 * 2 * 1024 * 256 + 2 * 200 * 512))
        b5 = 4 * 48 * 1200 + 2 * 4 * 768 * 300 + 2 * 4 * 2048 * 300 + 2 * 4 * 512 * 300 + 8 * 300
        lps_gpu = cfg5['value'] / world
        cfg5['roofline'] = {'tensor_frac': lps_gpu * f5 / (pk['tf_sustained'] * 1e12), 'hbm_frac': lps_gpu * b5 / (pk['hbm_gbs'] * 1e9),
                            'algorithmic_per_line': {'flops': f5, 'bytes': b5}, 'note': 'whole path per GPU against the measured peaks (SURVEY 8d)'}

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        lps, cms, threads = time_cpu(args.cpu_steps, 2)
        cpu = {'value': lps, 'unit': UNIT, 'cores': threads, 'kind': 'port', 'cpu': cpu_model_name(),
               'sample': f'{args.cpu_steps} batches of {BATCH} lines {HEIGHT}x{WIDTH} after 2 warm-up ({cms:.0f} ms/batch); '
                         'oracle/vgsl_oracle.py = torch-CPU restatement of rpred.py:225-228 + ctc_decoder.py, fp32; ' + CPU_NOTE}
    cfg3 = None
    if world == 1 and not args.no_extra:
        cfg3 = cfg3_brief(args)

    d2h = BATCH * T_ * 16 + BATCH * 4
    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic',
            'config': {'workload': 'cfg2', 'spec': CFG2, 'batch_per_gpu': BATCH, 'global_batch': BATCH * world, 'line': f'{HEIGHT}x{WIDTH}'},
            'notes': {'parallelism': f'replicas x{world} (independent line shards, 1 weight broadcast + 1 result gather)',
                       'value_is': f'{args.steps} steps per GPU, line batches resident in HBM, submitted through kb_recognize_async / kb_wait with {DEPTH} batches '
                                   'in flight from one host thread per GPU (serial.* = one synchronous kb_recognize per step)',
                       'l2': f'{NB} rotating input batches; ~0.3 GB of activations per step > 126 MB L2',
                       'numa_cores': None if numa_cores is None else f'{numa_cores[0]}..{numa_cores[-1]} ({len(numa_cores)} cores)'},
            'serial': {'value': world * BATCH * args.steps / (ms_serial / 1e3), 'ms_per_step': ms_serial / args.steps, 'gpu_launches': int(launches_serial),
                       'sum_of_stages_ms': round(sum(per_stage.values()), 4),
                       'note': 'one synchronous kb_recognize per step with per-stage event timing on; the gap to the sum of the stages is the host turn-around between calls'},
            'e2e': {'value': e2e, 'unit': UNIT, 'ms_per_step': ms_e2e / args.steps, 'in_flight': DEPTH, 'host_threads': 1,
                    'serial_value': world * BATCH * args.steps / (ms_e2e_serial / 1e3),
                    'h2d_bytes_per_step': BATCH * HEIGHT * WIDTH * 4, 'd2h_bytes_per_step': d2h,
                    'h2d_gbs_per_rank': BATCH * HEIGHT * WIDTH * 4 / (ms_e2e / args.steps / 1e3) / 1e9,
                    'api': 'TorchSeqRecognizer.submit/collect -> kb_recognize_async/kb_wait on one handle, pinned host lines in, label blocks out; '
                           'serial_value = TorchSeqRecognizer._recognize_raw -> kb_recognize one call at a time'},
            'e2e_u8': {'value': world * BATCH * args.steps / (ms_e2e_u8 / 1e3), 'unit': UNIT, 'ms_per_step': ms_e2e_u8 / args.steps,
                       'in_flight': DEPTH, 'host_threads': 1, 'h2d_bytes_per_step': BATCH * HEIGHT * WIDTH + BATCH * 6, 'd2h_bytes_per_step': d2h,
                       'api': 'TorchSeqRecognizer.submit(uint8 lines) -> kb_recognize_async(KB_DTYPE_U8): pinned uint8 lines in; ToDtype(scale) + tensor_invert + padding on the device'},
            'gpu_launches': int(launches), 'clocks': clocks, 'roofline': roof, 'cpu_baseline': cpu, 'cfg5': cfg5, 'cfg3': cfg3,
            'decoded_labels_last_step': decoded_last}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def cfg3_brief(args):
    """BASELINE configs[2] next to the headline: blla architecture on 8 pages 3x1800x1350 -> 4x1800x1350 heat maps (kb_segment), device-timed
    and end to end with pinned host pages in / pinned host heat maps out.  `python bench.py --workload cfg3` has the long form."""
    import kraken_b200 as kb
    from kraken_b200.blla import segmentation_heatmap
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import vgsl_oracle as vo
    N, H, W = 8, 1800, 1350
    om = vo.OracleModel(BLLA)
    m3 = kb.TorchVGSLModel(vgsl=BLLA, model_type=['segmentation'])
    m3.load_state_dict(om.init_like_reference(3))
    m3.to('cuda:0')
    g = torch.Generator().manual_seed(3)
    hpages = [torch.rand(N, 3, H, W, generator=g).pin_memory() for _ in range(2)]
    pages = [p_.cuda() for p_ in hpages]
    for i in range(3):
        segmentation_heatmap(m3, pages[i % 2], (H, W))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = 5
    e0.record()
    for i in range(steps):
        segmentation_heatmap(m3, pages[i % 2], (H, W))
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    segmentation_heatmap(m3, hpages[0], (H, W))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        hm = segmentation_heatmap(m3, hpages[i % 2], (H, W))
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / steps
    pk = peaks()
    return {'workload': 'cfg3', 'metric': 'pages/sec (blla forward, 2400x3200 pages -> 3x1800x1350)', 'batch': N, 'value': N / (ms / 1e3), 'unit': 'pages/s',
            'ms_per_step': ms, 'e2e': {'value': N / (e2e_ms / 1e3), 'ms_per_step': e2e_ms, 'h2d_bytes_per_step': N * 3 * H * W * 4,
                                       'd2h_bytes_per_step': int(hm.numel()) * 4, 'pinned_output': bool(hm.is_pinned())},
            'roofline': {'tensor_frac': N / (ms / 1e3) * 390.9e9 / (pk['tf_sustained'] * 1e12), 'hbm_frac': N / (ms / 1e3) * 1.628e9 / (pk['hbm_gbs'] * 1e9),
                         'note': 'whole forward: 390.9 GFLOP and 1.628 GB algorithmic per page (SURVEY 8d)'},
            'weights': 'seeded (reference init); parity of this size with the real blla.mlmodel weights: tests/test_gpu_configs.py'}


if __name__ == '__main__':
    main()
