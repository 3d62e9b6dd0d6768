#!/usr/bin/env python
"""bench.py -- panoramas/sec of HorizonNet('resnet50', rnn).forward at 512x1024, batch 32 per GPU.

    python bench.py --gpus N --steps K --warmup W           # our CUDA path (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N ...           # the reference's CPU implementation (oracle port)
    python bench.py ... --dump-outputs DIR                  # also save the last timed step's outputs (DIR/bon.npy, cor.npy)

One "step" = one forward over one batch of 32 synthetic panoramas per GPU (BASELINE.json configs[1];
N>1 = configs[3]: data-parallel shards + one NCCL all-gather of the outputs per step).
Prints ONE JSON line (rank 0).  Timing: W warm-up steps, then exactly K steps bracketed by
barrier + cuda synchronize, CUDA events on the launching stream, max over ranks.  The inputs rotate
between two 201 MB batches and every step streams >9 GB of activations, so nothing survives in the
126 MB L2 between steps ("inputs larger than L2").

Timed regions of the default run (all on the device, CUDA events):
  1. headline `value`: K steps through `HorizonNet.forward_pipelined` (C ABI hn_model_forward_async): back-to-back
     batches, the encoder of batch i+1 overlapping the bi-LSTM of batch i on internal streams, flushed at the end;
  2. the same K steps through plain `forward` (one stream, no overlap) with per-launch CUDA events inside the library:
     stage split, the conv roofline (`roofline`), the LSTM figure and `serial_ms_per_step`;
  3. `e2e`: host buffers in / host buffers out through hn_model_submit_host / hn_model_collect_host;
  4. secondary kernels (`roofline.secondary`): pano_stretch over 10k panoramas (BASELINE configs[2]), LSTM;
  5. comparators (aux): stock PyTorch eager (cuDNN) on the same GPU, TF32 on and off, and the CPU baselines.
"""
import argparse
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True        # the benchmark runs from a built tree and writes nothing into it
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BATCH = 32
GFLOP_PER_PANO = 142.90            # BASELINE.md section 2 (algorithmic, all convs + LSTM + head)
WORKLOAD = 'batch-32 synthetic 512x1024 panoramas, resnet50_rnn forward (BASELINE configs[1])'
PS_BYTES_PER_PANO = 12582912       # pano_stretch: 6,291,456 B read + 6,291,456 B written (SURVEY 8d)
KGRID = (0.5, 0.75, 1.0, 1.25, 1.5, 1.75, 2.0)


def _peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return {'hbm_gbs': p['hbm_gbs'], 'tf': p.get('bf16_tflops_sustained', p['bf16_tflops']),
                'tf_burst': p['bf16_tflops'], 'src': 'measured'}
    return {'hbm_gbs': 6650.0, 'tf': 1400.0, 'tf_burst': 1590.0, 'src': 'fallback'}


def host_threads():
    """Threads the CPU legs may use: the CPUs this process is allowed to run on, capped at the physical core count and
    at the cgroup CPU quota (a 1-GPU lease of a big host gets a slice of its cores; asking torch for os.cpu_count()
    threads there oversubscribes the slice and measured 35x slower in round 1)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    info = {'affinity': n, 'logical': os.cpu_count()}
    try:
        import psutil
        phys = psutil.cpu_count(logical=False)
        if phys:
            info['physical'] = phys
            n = min(n, phys)
    except Exception:
        pass
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()
        if quota != 'max':
            q = max(1, int(math.floor(float(quota) / float(period))))
            info['cgroup_quota'] = q
            n = min(n, q)
    except Exception:
        try:
            q = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())
            p = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if q > 0 and p > 0:
                info['cgroup_quota'] = max(1, q // p)
                n = min(n, info['cgroup_quota'])
        except Exception:
            pass
    info['used'] = max(1, n)
    return info


def _median(v):
    s = sorted(v)
    return s[len(s) // 2] if len(s) % 2 else 0.5 * (s[len(s) // 2 - 1] + s[len(s) // 2])


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU with NVML during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = threading.Event()
        self.sm = []
        self.reasons = set()
        self.sm_max = None
        self.power = []

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                nv.nvmlClocksThrottleReasonHwSlowdown: 'hw_slowdown',
                nv.nvmlClocksThrottleReasonHwThermalSlowdown: 'hw_thermal_slowdown',
                nv.nvmlClocksThrottleReasonSwThermalSlowdown: 'sw_thermal_slowdown',
                nv.nvmlClocksThrottleReasonSwPowerCap: 'sw_power_cap',
                nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: 'hw_power_brake',
            }
            while not self.stop_flag.is_set():
                self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                except Exception:
                    pass
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
                time.sleep(0.02)
        except Exception as e:              # NVML missing: report that, never fake numbers
            self.reasons.add(f'nvml_unavailable:{type(e).__name__}')

    def summary(self):
        sm = sorted(self.sm)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': self.sm_max,
                'power_w_max': max(self.power) if self.power else None, 'samples': len(sm),
                'reasons': sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------ CPU legs
def _cpu_forward_times(batch, reps, max_seconds, warmup=1):
    """Per-call seconds of the CPU oracle forward (restatement of the reference's model.py:254-281) at `batch`."""
    import torch
    from oracle import horizonnet_ref
    from horizonnet_b200.weights import synthetic_state_dict, synthetic_panoramas
    sd = synthetic_state_dict(0, 'random')
    x = synthetic_panoramas(batch, seed=11)
    times = []
    with torch.no_grad():
        for _ in range(warmup):
            horizonnet_ref.forward(sd, x)
        t_start = time.perf_counter()
        for _ in range(reps):
            t0 = time.perf_counter()
            horizonnet_ref.forward(sd, x)
            times.append(time.perf_counter() - t0)
            if time.perf_counter() - t_start > max_seconds and len(times) >= 3:
                break
    return times


def _ps_worker(args):
    """One pano_stretch on one CPU thread (reference misc/panostretch.py:81-117: numpy trig + scipy map_coordinates)."""
    import numpy as np
    from oracle import panostretch_ref
    seed, kx, ky = args
    os.environ['OMP_NUM_THREADS'] = '1'
    img = np.random.RandomState(seed).rand(512, 1024, 3).astype(np.float32)
    corners = np.array([[158, 186], [158, 329], [353, 185], [353, 330]], np.float32)
    t0 = time.perf_counter()
    panostretch_ref.pano_stretch(img, corners, kx, ky, use_scipy=True)
    return time.perf_counter() - t0


def cpu_pano_stretch_baseline(n_single=50, n_pool=64, workers=8):
    """SURVEY 8d: single-thread ms/img over >= 50 (kx,ky) samples, plus an 8-process pool mirroring the DataLoader's
    num_workers=8 (train.py:97), extrapolated to the 10k-pano job."""
    import multiprocessing as mp
    pairs = [(a, b) for a in KGRID for b in KGRID]
    single = [_ps_worker((i, *pairs[i % 49])) for i in range(n_single)]
    ms_img = _median(single) * 1e3
    out = {'single_thread_ms_per_img': round(ms_img, 2), 'single_thread_panos_per_s': round(1e3 / ms_img, 2),
           'samples': n_single, 'kind': 'port (oracle/panostretch_ref.py coordinates + scipy.ndimage.map_coordinates)'}
    try:
        ctx = mp.get_context('fork')
        with ctx.Pool(workers) as pool:
            pool.map(_ps_worker, [(1000 + i, *pairs[i % 49]) for i in range(workers)])      # warm the workers
            t0 = time.perf_counter()
            pool.map(_ps_worker, [(i, *pairs[i % 49]) for i in range(n_pool)], chunksize=1)
            dt = time.perf_counter() - t0
        rate = n_pool / dt
        out.update({'pool_workers': workers, 'pool_panos_per_s': round(rate, 2),
                    'pool_seconds_per_10k_extrapolated': round(10000 / rate, 1), 'pool_samples': n_pool})
    except Exception as e:
        out['pool_error'] = str(e)
    return out


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (the oracle port:
    /root/reference cannot travel to the GPU box and has no compiled code).  Each step is a bounded sample of the
    batch-32 workload: ONE panorama forward; `value` = 1 / median step time.  A batch-8 leg (median of >= 5) is
    reported beside it (SURVEY 8d asks for bs1 and bs8)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import torch
    ht = host_threads()
    # torchrun exports OMP_NUM_THREADS=1 to its workers; this arm is the only rank doing work
    torch.set_num_threads(ht['used'])
    t1 = _cpu_forward_times(1, args.steps, 1e9, warmup=max(1, min(args.warmup, 2)))
    med1 = _median(t1)
    value = 1.0 / med1
    t8 = _cpu_forward_times(8, 5, 90.0, warmup=1) if not args.quick_cpu else []
    med8 = _median(t8) if t8 else None
    cores = torch.get_num_threads()
    sample = ('1 panorama per step (bounded sample of the batch-32 workload), fp32 CPU torch ops, median of '
              f'{len(t1)} steps; threads used {cores}')
    emit_json({
        'impl': 'reference', 'metric': 'panoramas/sec', 'value': round(value, 4), 'unit': 'panoramas/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': round(med1 * 1e3, 2),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'sample': sample},
        'cpu_baseline': {'value': round(value, 4), 'unit': 'panoramas/s', 'cores': cores, 'kind': 'port', 'sample': sample,
                         'bs1_ms_median': round(med1 * 1e3, 2), 'bs1_ms_min': round(min(t1) * 1e3, 2),
                         'bs1_ms_max': round(max(t1) * 1e3, 2),
                         'bs8_panos_per_s': round(8.0 / med8, 4) if med8 else None,
                         'bs8_ms_median': round(med8 * 1e3, 2) if med8 else None, 'bs8_reps': len(t8),
                         'host_threads': ht},
        'e2e': {'value': round(value, 4), 'unit': 'panoramas/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    })


# ------------------------------------------------------------------------------------------------ GPU comparators
def gpu_eager_comparator(sd, x_dev, ours_bon, ours_cor, steps=5):
    """Stock PyTorch eager on the same GPU (BASELINE.md section 3 / SURVEY 2b: the bar a user would otherwise get from
    `model.HorizonNet(...).cuda()`): cuDNN convolutions + cuDNN nn.LSTM, the functional restatement in
    oracle/horizonnet_ref.py for everything around the LSTM.  Timed with CUDA events at bs32, TF32 allowed (torch's conv
    default) and disallowed; errors against the CPU fp32 oracle on two panoramas of the batch."""
    import torch
    from oracle import horizonnet_ref as R
    dev = x_dev.device
    sdd = {k: v.to(dev) for k, v in sd.items()}
    lstm = torch.nn.LSTM(1024, 512, num_layers=2, bidirectional=True).to(dev).eval()
    with torch.no_grad():
        for name, p in lstm.named_parameters():
            p.copy_(sdd['bi_rnn.' + name])
    lstm.flatten_parameters()

    def fwd(x):
        mean = x.new_tensor(R.X_MEAN).view(1, 3, 1, 1)
        std = x.new_tensor(R.X_STD).view(1, 3, 1, 1)
        feats = R.encoder((x[:, :3] - mean) / std, sdd)
        red = [R.global_height_conv(f, sdd, s, 256).reshape(x.shape[0], -1, 256) for s, f in enumerate(feats)]
        seq = torch.cat(red, dim=1).permute(2, 0, 1).contiguous()
        out, _ = lstm(seq)
        out = out @ sdd['linear.weight'].t() + sdd['linear.bias']
        out = out.view(out.shape[0], out.shape[1], 3, 4).permute(1, 2, 0, 3).contiguous().view(out.shape[1], 3, -1)
        return out[:, 1:], out[:, :1]

    rows = [0, x_dev.shape[0] - 1]
    with torch.no_grad():
        rb, rc = R.forward(sd, x_dev[rows].cpu())                      # CPU fp32 oracle (the parity reference)
    res = {'rows_checked': rows,
           'ours_max_abs_err': round(max(float((ours_bon[rows].cpu() - rb).abs().max()),
                                         float((ours_cor[rows].cpu() - rc).abs().max())), 9)}
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    try:
        torch.backends.cudnn.benchmark = True
        for label, tf32 in (('tf32', True), ('fp32', False)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            with torch.no_grad():
                for _ in range(3):
                    bon, cor = fwd(x_dev)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    bon, cor = fwd(x_dev)
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            err = max(float((bon[rows].cpu() - rb).abs().max()), float((cor[rows].cpu() - rc).abs().max()))
            res[label] = {'panos_per_s': round(x_dev.shape[0] / (ms * 1e-3), 1), 'ms_per_step': round(ms, 3),
                          'max_abs_err_vs_cpu_oracle': round(err, 9), 'meets_1e-4': bool(err < 1e-4)}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
    res['what'] = ('stock PyTorch eager on this GPU: cuDNN convs + cuDNN nn.LSTM, bs32, CUDA events, %d steps after 3 '
                   'warm-ups (cudnn.benchmark on)' % steps)
    return res


def pano_stretch_10k(dev, peaks):
    """BASELINE configs[2]: 10,000 synthetic 512x1024x3 panoramas, the 49-pair kx/ky grid cycled; 64 distinct images
    on the device are cycled to bound memory (805 MB in + out per call > L2).  CUDA events around the whole job."""
    import torch
    from horizonnet_b200.misc.panostretch import pano_stretch_batch
    n_img, total = 64, 10000
    gen = torch.Generator(device=dev).manual_seed(0)
    imgs = torch.rand(n_img, 512, 1024, 3, device=dev, generator=gen)
    out = torch.empty_like(imgs)
    pairs = [(a, b) for a in KGRID for b in KGRID]
    calls = []
    done = 0
    while done < total:
        n = min(n_img, total - done)
        calls.append((n, [pairs[(done + i) % 49][0] for i in range(n)], [pairs[(done + i) % 49][1] for i in range(n)]))
        done += n
    for c in calls[:3]:
        pano_stretch_batch(imgs[:c[0]], c[1], c[2], out=out[:c[0]])
    torch.cuda.synchronize()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for n, kx, ky in calls:
        pano_stretch_batch(imgs[:n], kx, ky, out=out[:n])
    a1.record()
    torch.cuda.synchronize()
    ms = a0.elapsed_time(a1)
    gbs = total * PS_BYTES_PER_PANO / (ms * 1e-3) / 1e9
    return {'kernel': 'stretch_kernel (pano_stretch, BASELINE configs[2])', 'bound': 'hbm', 'achieved': round(gbs, 1),
            'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': round(gbs / peaks['hbm_gbs'], 4),
            'peak_source': peaks['src'] + ' HBM copy bandwidth',
            'panos_per_s': round(total / (ms * 1e-3), 1), 'panos': total, 'ms_total': round(ms, 2),
            'launches': len(calls), 'avg_launch_ms': round(ms / len(calls), 4),
            'bytes_per_pano': PS_BYTES_PER_PANO,
            'sample': '10,000 panos = 64 distinct device images cycled (805 MB in+out per launch > L2), 49-pair kx/ky grid cycled'}


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as entry
    from horizonnet_b200 import _lib
    from horizonnet_b200.model import HorizonNet
    from horizonnet_b200.parallel import OutputGatherer
    from horizonnet_b200.weights import synthetic_state_dict, synthetic_panoramas

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device -- this framework has no CPU path (use --impl reference)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    if rank == 0:
        entry.build()
    if world > 1:
        dist.barrier()
    lib = _lib.lib()

    sd = synthetic_state_dict(0, 'random')
    net = HorizonNet('resnet50', True).eval()
    net.load_state_dict(sd, strict=True)
    net.use_tensor_cores(not args.fp32)
    net = net.to(dev)
    # two distinct input batches per rank, rotated (seeded per rank: SURVEY 8d config 4)
    xs = [synthetic_panoramas(BATCH, seed=1000 + rank + 100 * i).to(dev) for i in range(2)]
    gather = OutputGatherer() if world > 1 else None

    def run_steps(n, pipelined):
        """n steps; with N>1 every step's outputs are all-gathered (one step behind the forward in pipelined mode, so
        that the collective never waits for the recurrence that is still in flight)."""
        pending = None
        last = None
        for i in range(n):
            with torch.no_grad():
                out = net.forward_pipelined(xs[i & 1]) if pipelined else net(xs[i & 1])
            if world > 1:
                if pipelined:
                    if pending is not None:
                        last = gather(*pending)          # outputs of step i-1: complete on this stream by contract
                    pending = out
                else:
                    last = gather(*out)
            else:
                last = out
        if pipelined:
            net.flush()
            if world > 1 and pending is not None:
                last = gather(*pending)
        return last

    for mode in (True, False):
        run_steps(max(args.warmup, 3), mode)
    torch.cuda.synchronize()

    def timed(pipelined, profile):
        net.set_profile(profile)
        net.read_profile(reset=True)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        sampler = ClockSampler(local)
        sampler.start()
        time.sleep(0.05)
        l0 = lib.hn_kernel_launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        last = run_steps(args.steps, pipelined)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        sampler.stop_flag.set()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        launches = torch.tensor([lib.hn_kernel_launches() - l0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(launches, op=dist.ReduceOp.SUM)
        net.check()
        prof = net.read_profile(reset=True) if profile else None
        net.set_profile(False)
        sampler.join(timeout=2)
        return float(ms.item()), int(launches.item()), prof, sampler.summary(), last

    total_ms, launches, _, clocks, last_pipe = timed(True, False)          # 1. headline
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_pipe)
    serial_ms, _, prof, clocks_serial, last_serial = timed(False, True)    # 2. serial + per-launch events
    value = world * BATCH * args.steps / (total_ms * 1e-3)

    # N>1 self-check (SURVEY 8d config 4): the gathered result holds, bit for bit, what a single GPU computes for
    # every shard: rank 0 recomputes the LAST rank's final batch locally and compares it with its slice of the gather
    selfcheck = None
    if world > 1:
        idx = (args.steps - 1) & 1
        with torch.no_grad():
            xo = synthetic_panoramas(BATCH, seed=1000 + (world - 1) + 100 * idx).to(dev)
            ob, oc = net(xo)
            mb, mc = net(xs[idx])
        lo = (world - 1) * BATCH
        ok = bool(torch.equal(last_pipe[0][lo:lo + BATCH], ob) and torch.equal(last_pipe[1][lo:lo + BATCH], oc) and
                  torch.equal(last_pipe[0][rank * BATCH:(rank + 1) * BATCH], mb) and
                  torch.equal(last_serial[0][rank * BATCH:(rank + 1) * BATCH], mb) and
                  torch.equal(last_serial[1][rank * BATCH:(rank + 1) * BATCH], mc))
        okt = torch.tensor([1.0 if ok else 0.0], device=dev)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        selfcheck = {'gathered_equals_single_gpu_bitwise': bool(okt.item() == 1.0),
                     'what': 'every rank: own shard of the NCCL gather (pipelined and serial loops) == its local forward; plus the last '
                             "rank's shard recomputed locally from its seed"}
        if not selfcheck['gathered_equals_single_gpu_bitwise']:
            raise SystemExit('bench.py: the gathered outputs differ from the single-GPU result')
    else:
        with torch.no_grad():
            sb, sc = net(xs[(args.steps - 1) & 1])
        if not (torch.equal(sb, last_pipe[0]) and torch.equal(sc, last_pipe[1])):
            raise SystemExit('bench.py: pipelined forward differs from the plain forward')

    # ---- 3. end-to-end through the C ABI with HOST buffers (H2D + forward + D2H inside the calls)
    xh = [synthetic_panoramas(BATCH, seed=2000 + rank + 100 * i).pin_memory() for i in range(2)]
    e2e_steps = max(3, min(args.steps, 10))
    net.forward_host(xh[0], device=local)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    net.submit_host(xh[0], device=local)                 # pipelined host API: upload + encoder of batch i+1 overlap batch i
    for i in range(e2e_steps):
        if i + 1 < e2e_steps:
            net.submit_host(xh[(i + 1) & 1], device=local)
        hb, hc = net.collect_host(device=local)
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * BATCH * e2e_steps / float(e2e_s.item())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = _peaks()
    # ---- roofline of the dominant kernel family: the implicit-GEMM convolution kernels (serial region, per-launch events)
    conv_cls = ('encoder_convs', 'height_reduction_convs', 'lstm_input_projection')
    conv_ms = sum(prof[c][0] for c in conv_cls)
    conv_flops = sum(prof[c][1] for c in conv_cls)
    conv_n = sum(prof[c][2] for c in conv_cls)
    achieved = conv_flops / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
    stage_ms = {k: round(v[0] / args.steps, 4) for k, v in prof.items()}
    traffic = None
    try:
        import glob
        files = sorted(glob.glob(os.path.join(ROOT, 'profiles', 'r*_conv_tc_traffic.json')))
        if files and not args.fp32:
            traffic = json.load(open(files[-1]))['dram_bytes_per_launch_avg']
    except Exception:
        traffic = None
    roofline = {
        'kernel': 'conv implicit-GEMM family (%s)' % ('conv_igemm_f32, fp32 CUDA cores' if args.fp32 else 'conv_tc_kernel / gemm_tc_kernel, tcgen05 split-fp16 x3 products'),
        'bound': 'tensor', 'achieved': round(achieved, 3), 'peak': peaks['tf'], 'unit': 'TFLOP/s',
        'frac': round(achieved / peaks['tf'], 5), 'peak_source': peaks['src'] + ' bf16 dense, sustained',
        'traffic': traffic, 'traffic_source': 'dram__bytes_read+write per launch, averaged over the conv-family launches of one bs32 forward (ncu per-launch capture, latest profiles/r*_conv_tc_traffic.json)' if traffic else None,
        'launches_per_step': conv_n / args.steps,
        'avg_launch_ms': round(conv_ms / max(conv_n, 1), 5),
        'algorithmic_gflop_per_step': round(conv_flops / args.steps / 1e9, 2),
        'share_of_step': round(conv_ms / serial_ms, 4),
        'issued_over_algorithmic': 1 if args.fp32 else 3,
        'measured_in': 'the serial timed region (plain forward, one stream, per-launch CUDA events inside the library)',
        'note': 'achieved = algorithmic conv FLOPs (2*M*N*K, single product) / summed CUDA-event time of the conv launches; the tensor pipe issues 3x that (hi*hi + hi*lo + lo*hi)',
        'secondary': [],
    }
    lstm_ms = prof['lstm_recurrence'][0] / args.steps
    roofline['secondary'].append({
        'kernel': 'lstm_cluster_kernel (bi-LSTM recurrence, 2 launches per step)', 'bound': 'hbm',
        'achieved': round(151.4e6 / (lstm_ms * 1e-3) / 1e9, 2) if lstm_ms > 0 else None, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
        'frac': round(151.4e6 / (lstm_ms * 1e-3) / 1e9 / peaks['hbm_gbs'], 5) if lstm_ms > 0 else None,
        'ms_per_step': round(lstm_ms, 4), 'us_per_recurrence_step': round(lstm_ms * 1e3 / 512, 3),
        'note': 'algorithmic 151.4 MB per batch of 32 (SURVEY 8d); the recurrence is latency-bound (512 dependent steps on 64 SMs), so '
                'the HBM fraction is reported because BASELINE asks for it; in the headline loop it overlaps the next batch\'s encoder'})

    aux = {'stage_ms_per_step_serial': stage_ms}
    try:
        roofline['secondary'].append(pano_stretch_10k(dev, peaks))
    except Exception as e:
        roofline['secondary'].append({'kernel': 'stretch_kernel', 'error': str(e)})
    # ---- auxiliary: single-panorama inference with device-side TTA (flip + 2 rotations = 4 views), "next" row f2
    try:
        from horizonnet_b200.inference import tta_forward
        xi = synthetic_panoramas(1, seed=77)
        for _ in range(2):
            tta_forward(net, xi, flip=True, rotate=[0.25, 0.5])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        reps = 10
        for _ in range(reps):
            tta_forward(net, xi, flip=True, rotate=[0.25, 0.5])     # host tensor in, numpy out: includes H2D + D2H
        dt = (time.perf_counter() - t0) / reps
        aux['tta_single_image'] = {'images_per_s': round(1.0 / dt, 2), 'ms_per_image': round(dt * 1e3, 3), 'views': 4,
                                   'api': 'horizonnet_b200.inference.tta_forward (hn_model_infer_tta), host in / host out'}
    except Exception as e:
        aux['tta_single_image'] = {'error': str(e)}
    # ---- auxiliary: the on-device augmentation pipeline ("next" row f3) and the rotatePanorama gather (f4), if built
    try:
        from horizonnet_b200 import augment as _aug
        aux.update(_aug.bench_aux(dev, peaks))
    except Exception as e:
        aux['augment'] = {'error': str(e)}

    # ---- auxiliary: the training step ("next" row f1, BASELINE configs[4] shape per GPU: batch 8, L1 + BCE, Adam)
    if world == 1:
        try:
            aux['train_step'] = train_step_aux(dev)
        except Exception as e:
            aux['train_step'] = {'error': '%s: %s' % (type(e).__name__, e)}
        torch.cuda.empty_cache()

    # ---- comparators (N=1 only): stock PyTorch eager on this GPU; the CPU oracle on this host's cores
    cpu = None
    if world == 1 and not args.no_comparators:
        try:
            with torch.no_grad():
                ob, oc = net(xs[0])
            aux['gpu_eager'] = gpu_eager_comparator(sd, xs[0], ob, oc)
        except Exception as e:
            aux['gpu_eager'] = {'error': '%s: %s' % (type(e).__name__, e)}
        torch.cuda.empty_cache()
    if world == 1 and not args.no_cpu_baseline:
        ht = host_threads()
        torch.set_num_threads(ht['used'])
        t1 = _cpu_forward_times(1, 9, 14.0)
        t8 = _cpu_forward_times(8, 3, 30.0, warmup=0) if not args.quick_cpu else []
        med1 = _median(t1)
        cpu = {'value': round(1.0 / med1, 4), 'unit': 'panoramas/s', 'cores': torch.get_num_threads(), 'kind': 'port',
               'sample': f'median of {len(t1)} single-panorama forwards of the same random-init resnet50_rnn '
                         '(oracle/horizonnet_ref.py, torch CPU fp32) after 1 warm-up',
               'bs1_ms_median': round(med1 * 1e3, 2), 'host_threads': ht}
        if t8:
            cpu['bs8_panos_per_s'] = round(8.0 / _median(t8), 4)
            cpu['bs8_reps'] = len(t8)
        try:
            cpu['train_step'] = cpu_train_step_baseline()
        except Exception as e:
            cpu['train_step'] = {'error': str(e)}
        try:
            cpu['pano_stretch'] = cpu_pano_stretch_baseline()
        except Exception as e:
            cpu['pano_stretch'] = {'error': str(e)}

    line = {
        'metric': 'panoramas/sec', 'value': round(value, 3), 'unit': 'panoramas/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': round(total_ms / args.steps, 4),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32' if args.fp32 else 'f16x2-split (hi+lo fp16 planes, 3 tcgen05 products, fp32 accumulate; fp32-equivalent)',
        'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'global_batch': BATCH * world, 'parallelism': f'dp{world}',
                   'weights': 'random-init (synthetic_state_dict seed 0, randomised BN statistics)',
                   'l2': 'inputs larger than L2 (2 rotating 201 MB batches, >9 GB activations per step)',
                   'schedule': 'back-to-back batches through hn_model_forward_async: encoder of batch i+1 overlaps the bi-LSTM of batch i '
                               '(two internal streams), flushed inside the timed region; serial_ms_per_step is the one-stream latency',
                   'collective': 'all_gather_into_tensor of bon [32,2,1024] + cor [32,1,1024] fp32 per rank per step (NCCL)' if world > 1 else 'none',
                   'selfcheck': selfcheck},
        'clocks': clocks,
        'serial_ms_per_step': round(serial_ms / args.steps, 4),
        'serial_panos_per_s': round(world * BATCH * args.steps / (serial_ms * 1e-3), 2),
        'e2e': {'value': round(e2e_value, 3), 'unit': 'panoramas/s', 'steps': e2e_steps,
                'h2d_bytes_per_step': BATCH * 3 * 512 * 1024 * 4 * world, 'd2h_bytes_per_step': BATCH * 3 * 1024 * 4 * world,
                'api': 'hn_model_submit_host / hn_model_collect_host (pinned host buffers; every step uploads its 201 MB input and reads its outputs back; upload + encoder of batch i+1 overlap batch i)'},
        'gpu_launches': launches,
        'roofline': roofline,
        'cpu_baseline': cpu,
        'tflops_algorithmic': round(value * GFLOP_PER_PANO / 1e3, 2),
        'aux': aux,
    }
    emit_json(line)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(path, outputs):
    """--dump-outputs: the (bon, cor) the headline path returned in its last timed step -- with N>1 the all-gathered
    result -- as float32 path/bon.npy [B,2,1024] and path/cor.npy [B,1,1024] (393 KB per 32 panoramas).  Weights and
    inputs are seeded, so two builds run with the same arguments can be compared output for output."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in zip(('bon', 'cor'), outputs):
        np.save(os.path.join(path, name + '.npy'), t.detach().float().cpu().numpy())


def train_step_aux(dev, batch=8, steps=3):
    """One optimizer step of train.py (:272-281) through the library's autograd boundary: train-mode forward with tape,
    L1 + BCE-with-logits (train.py:53-56), loss.backward() (hn_train_backward + one gradient per parameter),
    Adam (train.py:221-223) and the re-upload of the stepped weights.  Device-timed with CUDA events."""
    import torch
    import torch.nn.functional as F
    from horizonnet_b200.model import HorizonNet
    from horizonnet_b200.weights import synthetic_state_dict, synthetic_panoramas
    net = HorizonNet('resnet50', True)
    net.load_state_dict(synthetic_state_dict(0, 'random'))
    net = net.to(dev).train()
    opt = torch.optim.Adam(net.parameters(), lr=1e-4, betas=(0.9, 0.999))
    x = synthetic_panoramas(batch, seed=5).to(dev)
    g = torch.Generator().manual_seed(6)
    y_bon = (torch.rand(batch, 2, 1024, generator=g) - 0.5).to(dev)
    y_cor = torch.rand(batch, 1, 1024, generator=g).to(dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    fw = bw = op = 0.0
    loss = None
    for it in range(steps + 2):
        torch.cuda.synchronize(dev)
        ev[0].record()
        opt.zero_grad()
        bon, cor = net(x)
        loss = F.l1_loss(bon, y_bon) + F.binary_cross_entropy_with_logits(cor, y_cor)
        ev[1].record()
        loss.backward()
        ev[2].record()
        opt.step()
        ev[3].record()
        torch.cuda.synchronize(dev)
        if it >= 2:
            fw += ev[0].elapsed_time(ev[1]); bw += ev[1].elapsed_time(ev[2]); op += ev[2].elapsed_time(ev[3])
    net.check()
    phases = net.train_profile()
    from horizonnet_b200 import _lib
    wgrad_tc = bool(_lib.lib().hn_wgrad_tc_enabled())
    fw, bw, op = fw / steps, bw / steps, op / steps
    out = {'batch': batch, 'forward_ms': round(fw, 2), 'backward_ms': round(bw, 2), 'optimizer_ms': round(op, 2),
           'step_ms': round(fw + bw + op, 2), 'panoramas_per_s': round(batch / (fw + bw + op) * 1e3, 2),
           'backward_phases_ms': phases, 'final_loss': round(float(loss.detach()), 5),
           'dtype': ('convolutions, their data gradients and the weight gradients of the Cin/Cout % 64 == 0 convolutions + the LSTM weights: tcgen05 '
                     'split-fp16 planes (fp32-equivalent); other weight gradients, BatchNorm, LSTM BPTT: fp32 CUDA cores'
                     if wgrad_tc else
                     'convolutions + their data gradients: tcgen05 split-fp16 planes (fp32-equivalent); weight gradients, '
                     'BatchNorm, LSTM BPTT: fp32 CUDA cores'),
           'wgrad_tc': wgrad_tc,
           'api': 'HorizonNet.train(); net(x); loss.backward(); Adam.step()  (hn_train_forward / hn_train_backward)',
           'note': 'forward_ms includes the re-upload + re-packing of the weights the optimizer just changed'}
    del net, opt
    return out


def cpu_train_step_baseline(batch=2):
    """The same step on the host cores: the CPU oracle (torch CPU fp32, the reference's arithmetic) forward + autograd
    backward in train mode at batch 2 (bounded: a few seconds)."""
    import torch
    import torch.nn.functional as F
    from oracle import horizonnet_ref
    from horizonnet_b200.model import HorizonNet
    from horizonnet_b200.weights import synthetic_state_dict, synthetic_panoramas
    sd = synthetic_state_dict(0, 'random')
    names = [k for k, _ in HorizonNet('resnet50', True).named_parameters()]
    x = synthetic_panoramas(batch, seed=5)
    g = torch.Generator().manual_seed(6)
    y_bon, y_cor = torch.rand(batch, 2, 1024, generator=g) - 0.5, torch.rand(batch, 1, 1024, generator=g)
    times = []
    for _ in range(1):
        psd = {k: (v.clone().requires_grad_() if k in names else v) for k, v in sd.items()}
        t0 = time.perf_counter()
        bon, cor = horizonnet_ref.forward(psd, x, train=horizonnet_ref.TrainMode())
        loss = F.l1_loss(bon, y_bon) + F.binary_cross_entropy_with_logits(cor, y_cor)
        torch.autograd.grad(loss, [psd[k] for k in names])
        times.append(time.perf_counter() - t0)
    return {'panoramas_per_s': round(batch / min(times), 4), 'batch': batch, 'step_s': round(min(times), 3),
            'cores': torch.get_num_threads(), 'kind': 'port', 'sample': 'forward + autograd backward of the CPU oracle in train mode, '
            'one run, no optimizer step'}


_JSON_FD = None


def claim_stdout():
    """stdout must carry exactly ONE JSON line: keep a private duplicate of fd 1 for it and point fd 1 at stderr, so
    that anything else written to stdout at the C level (e.g. NCCL's "NCCL version ..." banner) lands on stderr."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit_json(line):
    data = (json.dumps(line) + '\n').encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--fp32', action='store_true', help='exact fp32 CUDA-core kernels instead of tcgen05')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-comparators', action='store_true', help='skip the PyTorch-eager GPU comparator')
    ap.add_argument('--quick-cpu', action='store_true', help='CPU baseline: bs1 only')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the outputs of the last timed step to DIR/bon.npy and DIR/cor.npy (float32)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs applies to --impl ours')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
