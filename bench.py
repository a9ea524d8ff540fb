# -*- coding: utf-8 -*-
"""bench.py -- images/sec of the LFD hot path (forward + device post-process) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config WIDERFACE_S] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (BASELINE.json configs[1]): WIDERFACE-S, 1280x720, batch 8 per GPU, bf16, synthetic frames and synthetic
weights (tests/synth.py; no network for datasets / checkpoints).  One step = one batch: backbone + neck + head
(CUDA-graph replay of the layer plan) + score / decode / NMS (lfd_postprocess).  Multi-GPU: the batch dimension
shards across ranks, one process per GPU, no collective on the inference path (weak scaling: 8 frames per GPU).

Prints ONE JSON line (rank 0).  `value` = images/s with the uint8 frames already resident in HBM; `e2e` = the same
through StreamingDetector with HOST (pinned) frames in and HOST detections out; `roofline` = the dominant kernel of the
step timed live with CUDA events; `cpu_baseline` = the oracle port (the reference's PyTorch CPU arithmetic) on a bounded
sample.  --impl reference times that CPU path as the reference arm.

`value` is timed over exactly K steps after W warm-up steps (at least 3).  Frames and weights are seeded, so the same
arguments give the same inputs on every run; --dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy
(float32 / float64), to compare two builds output for output.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, 'lfd-a-light-and-fast-detector_b200'), os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs[1]: the workload `metric` is quoted on (default)
    'WIDERFACE_S': dict(cfg='WIDERFACE_S', N=8, H=720, W=1280, dtype='bf16', name='WIDERFACE-S inference 1280x720 batch=8 per GPU'),
    # configs[0] geometry on the GPU (the CPU-runnable plumbing case)
    'WIDERFACE_XS': dict(cfg='WIDERFACE_XS', N=1, H=480, W=640, dtype='bf16', name='WIDERFACE-XS inference 640x480 batch=1'),
    # configs[3]
    'TT100K_L': dict(cfg='TT100K_L', N=16, H=1080, W=1920, dtype='bf16', name='TT100K LFD_L inference 1920x1080 batch=16 per GPU', pass_fraction=0.0002, cap=16384),
    # configs[4]: fp16 4K throughput sweep, batch-sharded (2 frames per GPU per step)
    'WIDERFACE_XS_4K': dict(cfg='WIDERFACE_XS', N=2, H=2160, W=3840, dtype='fp16', name='WIDERFACE-XS inference 3840x2160 batch=2 per GPU', pool=4),
}
POOL = 8          # device-resident input batches rotated through (8 x 22 MB = 177 MB > 126 MB L2)
IOU_THR = 0.3     # WIDERFACE_train/predict.py:22
PASS_FRACTION = 0.005
DUMP_MAX_BYTES = 64 << 20   # --dump-outputs: the largest workload (TT100K_L, 16 x 16384 detection slots) needs < 10 MB


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm_gbs=float(d['hbm_gbs']), bf16_tflops=float(d.get('bf16_tflops_sustained', d['bf16_tflops'])), source='measured (MEASURED_PEAKS.json)')
    return dict(hbm_gbs=6650.0, bf16_tflops=1400.0, source='fallback (B200_PROFILING.md)')


class ClockSampler(object):
    """SM clock / throttle reasons sampled DURING the timed region.  NVML in a thread every 2 ms (the timed region of the
    default run is ~0.1 s, shorter than nvidia-smi's minimum useful polling period); falls back to `nvidia-smi -lms`."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index, self.rows, self.proc, self.nvml, self.handle = index, [], None, None, None
        self.samples, self.bits, self.stop_flag, self.max_mhz = [], 0, False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(index).uuid)
            try:
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(('GPU-' + uuid) if not uuid.startswith('GPU-') else uuid)
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                self.samples.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                self.bits |= int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nvml is not None:
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=1.0)
            n = self.nvml
            names = (('hw_slowdown', n.nvmlClocksEventReasonHwSlowdown), ('hw_thermal_slowdown', n.nvmlClocksEventReasonHwThermalSlowdown),
                     ('sw_thermal_slowdown', n.nvmlClocksEventReasonSwThermalSlowdown), ('sw_power_cap', n.nvmlClocksEventReasonSwPowerCap),
                     ('hw_power_brake', n.nvmlClocksEventReasonHwPowerBrakeSlowdown))
            reasons = sorted(name for name, bit in names if self.bits & int(bit))
            return dict(sm_mhz=float(np.median(self.samples)) if self.samples else None, sm_max_mhz=self.max_mhz, reasons=reasons,
                        samples=len(self.samples), source='nvml')
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                pass
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=sorted(reasons), samples=len(sm),
                    source='nvidia-smi')


def ncu_traffic(cfg, dtype, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, from the committed `ncu --set full` capture:
    profiles/ncu_traffic.json is written by profiles/ncu_parse.py from the .ncu-rep that profiles/ncu_run.sh produces
    (re-run both after a kernel change).  None when that kernel has no capture."""
    path = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if not os.path.exists(path):
        return None
    try:
        table = json.load(open(path))
    except Exception:
        return None
    e = table.get('%s/%s' % (cfg, dtype), {}).get(kernel)
    return None if e is None else int(e['dram_bytes_read'] + e['dram_bytes_write'])


def op_algorithmic(row, N, input_bytes_per_px):
    """(bytes, flops) one launch must move / compute: input once, output once, residual once, weights once."""
    k, cin, cout = row['ksize'], row['Cin'], row['Cout']
    px_in, px_out = N * row['H'] * row['W'], N * row['Ho'] * row['Wo']
    tc = row.get('tail_cout', 0)            # fused 1x1 tail: the cout-channel intermediate never reaches HBM
    cf = tc if tc else cout
    tail_b, tail_f = (cout * tc * 2, 2.0 * px_out * cout * tc) if tc else (0, 0.0)
    if row['kind'] == 'stem0':
        return px_in * input_bytes_per_px + px_out * cf * 2 + 27 * cout * 2 + tail_b, 2.0 * px_out * cout * 27 + tail_f
    if row['kind'] == 'conv':
        dc = row.get('ds_cout', 0)          # fused shortcut conv: second output, reads the same input
        b = px_in * cin * 2 + px_out * cf * 2 * (2 if row['res'] else 1) + k * k * cin * cout * 2 + tail_b + px_out * dc * 2 + cin * dc * 2
        return b, 2.0 * px_out * cout * cin * k * k + tail_f + 2.0 * px_out * dc * cin
    if row['kind'] == 'gn_apply':
        return px_in * cin * 2 * 2, 0.0
    return px_in * cin * 2 + px_out * cout * 4, 2.0 * px_out * cout * cin   # head_final


def op_read_write(row, N, input_bytes_per_px):
    """(read bytes, written bytes) of op_algorithmic's byte count."""
    b, _ = op_algorithmic(row, N, input_bytes_per_px)
    px_out = N * row['Ho'] * row['Wo']
    if row['kind'] in ('stem0', 'conv'):
        w = px_out * ((row.get('tail_cout', 0) or row['Cout']) + row.get('ds_cout', 0)) * 2
    elif row['kind'] == 'gn_apply':
        w = b // 2
    else:
        w = px_out * row['Cout'] * 4
    return b - w, w


def directional_peaks(dev):
    """HBM ceilings for one-directional streams, measured here (best of 5, CUDA events): a layer that mostly writes (the stem: 22 MB in,
    236 MB out) or mostly reads cannot reach the copy figure the roofline divides by, which is half reads and half writes."""
    n = 1 << 27                                 # 512 MB of fp32
    a = torch.empty(n, dtype=torch.float32, device=dev)

    def best(fn):
        fn()
        torch.cuda.synchronize()
        t = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            t.append(e0.elapsed_time(e1))
        return 4.0 * n / (min(t) * 1e-3) / 1e9
    w = best(lambda: a.fill_(1.0))
    r = best(lambda: a.sum())
    del a
    return dict(write_only_gbs=w, read_only_gbs=r, how='torch fill_ / sum over 512 MB fp32, best of 5')


def op_name(row):
    return '%s %dx%d/s%d %d->%d @%dx%d' % (row['kind'], row['ksize'], row['ksize'], row['stride'], row['Cin'], row['Cout'], row['Ho'], row['Wo'])


def init_nccl(dev):
    """NCCL prints its version banner on stdout at communicator creation: keep stdout for the ONE JSON line."""
    import torch.distributed as dist
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        dist.init_process_group('nccl', device_id=dev)
        dist.barrier()
        torch.cuda.synchronize()
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)


TRAIN_WORKLOADS = {
    # BASELINE.json configs[2]: WIDERFACE-L training, bf16, 640x640 synthetic crops, data parallel (16 crops per GPU = the reference's
    # batch_size 64 on 4 GPUs, WIDERFACE_train/WIDERFACE_LFD_L.py:58,168); SGD(0.9, 1e-4) + clip_grad_norm_(10) as :218-226
    'WIDERFACE_L_train': dict(cfg='WIDERFACE_L', N=16, H=640, W=640, dtype='bf16', name='WIDERFACE-L training 640x640 batch=16 per GPU'),
}
_TOP_NAMES = ['pack', 'stem0', 'conv', 'bn_stats', 'bn_apply', 'gn_apply', 'head_final', 'head_final_bwd', 'norm_bwd_reduce', 'norm_bwd_apply',
              'wgrad', 'wgrad_stem', 'unpack', 'zero']


def train_op_algorithmic(op, N):
    """(bytes, flops) one training-plan launch must move / compute (bf16 activations, fp32 weight-gradient staging)."""
    kind = _TOP_NAMES[op['kind']]
    g = lambda k, d=0: op.get(k, d) or d
    px_in, px_out = N * g('H') * g('W'), N * g('Ho', g('H')) * g('Wo', g('W'))
    cin, cout, k = g('Cin'), g('Cout'), g('ksize', 1)
    if kind in ('conv', 'stem0'):
        res = 1 if op['off'].get(2) is not None else 0
        in_b = px_in * 3 if kind == 'stem0' else px_in * cin * 2
        return in_b + px_out * cout * 2 * (1 + res) + k * k * cin * cout * 2, 2.0 * px_out * cout * cin * k * k
    if kind in ('wgrad', 'wgrad_stem'):
        in_b = px_in * 3 if kind == 'wgrad_stem' else px_in * cin * 2
        return in_b + px_out * cout * 2 + k * k * cin * cout * 4, 2.0 * px_out * cout * cin * k * k
    if kind == 'bn_stats':
        return px_in * cout * 2, 0.0
    if kind in ('bn_apply', 'gn_apply'):
        return px_in * cout * 2 * (2 + (1 if op['off'].get(2) is not None else 0)), 0.0
    if kind == 'norm_bwd_reduce':
        return px_in * cout * 2 * (2 + (1 if op['off'].get(1) is not None else 0)), 0.0
    if kind == 'norm_bwd_apply':
        return px_in * cout * 2 * (3 + (1 if op['off'].get(1) is not None else 0) + (1 if op['off'].get(7) is not None else 0)), 0.0
    if kind == 'head_final':
        no = g('n_cls') + g('n_reg')
        return px_in * 128 * 2 + px_in * no * 4, 2.0 * px_in * no * 128
    if kind == 'head_final_bwd':
        no = g('n_cls') + g('n_reg')
        return px_in * 128 * 2 * 2 + px_in * no * 4, 3 * 2.0 * px_in * no * 128
    return 0, 0.0


def train_op_name(op):
    kind = _TOP_NAMES[op['kind']]
    if kind in ('conv', 'stem0', 'wgrad', 'wgrad_stem'):
        return '%s %dx%d/s%d %d->%d @%dx%d' % (kind, op['ksize'], op['ksize'], op['stride'], op['Cin'], op['Cout'], op['Ho'], op['Wo'])
    if 'H' in op:
        return '%s C=%d @%dx%d' % (kind, op.get('Cout', 0), op['H'], op['W'])
    return kind


def train_config(wl, world):
    return dict(workload=wl['name'], model=wl['cfg'], frames_per_step_per_gpu=wl['N'], height=wl['H'], width=wl['W'], dtype=wl['dtype'],
                input='synthetic uint8 BGR crops + synthetic ground truth (0..30 boxes per crop, sides log-uniform in [4, 320], one negative crop '
                      'per batch; tests/synth.py weights; no network for datasets / checkpoints)',
                step='forward (train mode, BatchNorm batch statistics) + label assignment + focal / IoU loss + backward (dgrad, wgrad, norm '
                     'backward) + gradient all-reduce + clip_grad_norm_(10) + SGD(momentum 0.9, weight decay 1e-4) step',
                parallelism='data parallel x%d: per-rank shards, global positive-count normalisation, ONE flat-buffer NCCL all-reduce' % world)


def cpu_train_leg(wl, steps, warmup, frames, budget_s=None):
    """The reference's CPU training step for this workload: the same module graph in fp32 by ATen + autograd (tests/aten_train_reference.py:
    the reference's arithmetic, lfd/model/lfd.py:511-542), the oracle's label assignment + losses (lfd.py:109-395), clip_grad_norm_ + torch SGD
    (optimizer_hook.py:21-36), all host threads.  With a `budget_s`, the timed loop stops early once that many seconds have passed."""
    import synth
    from aten_train_reference import train_forward as aten_forward
    from helpers import build_model as product_model
    from oracle import lfd_oracle as orc
    cfg = orc.CONFIGS[wl['cfg']]
    model = product_model(wl['cfg'])
    model.train()
    x = synth.synth_input(frames, wl['H'], wl['W'])
    ann = synth.synth_annotations(frames, wl['H'], wl['W'], cfg['lfd']['num_classes'], seed=7, max_boxes=30)
    opt = torch.optim.SGD(model.parameters(), lr=0.001, momentum=0.9, weight_decay=1e-4)
    torch.set_num_threads(min(os.cpu_count() or 1, 32))

    def step():
        cls, reg = aten_forward(model, x)
        sizes = [model._head_indexes_to_feature_map_sizes[i] for i in range(len(model._head_indexes_to_feature_map_sizes))]
        out = orc.get_loss(cfg, cls, reg, sizes, ann)
        opt.zero_grad()
        out['loss'].backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm=10, norm_type=2)
        opt.step()
    for _ in range(warmup):
        step()
    t0, done = time.time(), 0
    for _ in range(steps):
        step()
        done += 1
        if budget_s is not None and time.time() - t0 > budget_s:
            break
    dt = time.time() - t0
    return dict(ips=frames * done / dt, ms=dt / done * 1e3, done=done, cores=torch.get_num_threads())


def train_main(args):
    wl = TRAIN_WORKLOADS[args.config]
    rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    warmup = max(args.warmup, 3)
    metric = 'images/sec %s %s' % (wl['name'], wl['dtype'])
    config = train_config(wl, max(world, args.gpus))
    N, H, W = wl['N'], wl['H'], wl['W']
    if args.impl == 'reference':
        if rank != 0:
            return 0
        frames = 2
        r = cpu_train_leg(wl, args.steps, 1, frames)
        line = dict(metric=metric, value=r['ips'], unit='images/s', n_gpus=args.gpus, steps=r['done'], warmup=1, ms_per_step=r['ms'], higher_is_better=True,
                    scaling='weak', vs_baseline=None, dtype='f32', data='synthetic', impl='reference', config=config,
                    impl_detail=dict(note='CPU training step of the reference: ATen fp32 forward + autograd over the same module graph, '
                                          'oracle label assignment + losses, clip_grad_norm_ + torch SGD', frames_per_step=frames),
                    cpu_baseline=dict(value=r['ips'], unit='images/s', cores=r['cores'], kind='port', sample='%d crops per step, %d steps' % (frames, r['done'])),
                    e2e=dict(value=r['ips'], unit='images/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
        print(json.dumps(line))
        return 0

    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (there is no CPU fallback for the product path)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    import torch.distributed as dist
    if world > 1:
        init_nccl(dev)
    import synth
    from helpers import build_model as product_model
    from lfd.execution.hooks import OptimizerHook
    from lfd.execution.optim import FusedSGD
    from lfd.pipeline import bind_host_to_gpu_numa_node
    numa_node = bind_host_to_gpu_numa_node(dev)
    model, _ = build_model(wl['cfg'])
    model.to(dev).train()
    model.use_cuda_graph_training = not args.no_graph
    if world > 1:
        from lfd.execution.parallel import broadcast_module_state
        broadcast_module_state(model)
    opt = FusedSGD.from_torch(torch.optim.SGD(model.parameters(), lr=0.001, momentum=0.9, weight_decay=1e-4), model)
    hook = OptimizerHook(dict(max_norm=10, norm_type=2), 10)

    class _Exec(object):
        config_dict = dict(model=model, optimizer=opt, epoch=0)
    g = torch.Generator().manual_seed(2000 + rank)
    npool = 4        # 4 x 19.7 MB of frames; the ~13 GB activation / gradient workspace is rewritten every step (>> L2)
    pool = [torch.randint(0, 256, (N, H, W, 3), generator=g, dtype=torch.uint8).to(dev) for _ in range(npool)]
    host_pool = [torch.randint(0, 256, (N, H, W, 3), generator=g, dtype=torch.uint8).pin_memory() for _ in range(2)]
    anns = [synth.synth_annotations(N, H, W, 1, seed=100 * rank + i, max_boxes=30) for i in range(npool)]
    times = dict(assign=0.0)

    def step(i, x=None):
        out = model(pool[i % npool] if x is None else x)
        ld = model.get_loss(out, anns[i % npool])
        _Exec.config_dict['loss'] = ld['loss']
        hook.after_train_iter(_Exec)
        return ld['loss_values']

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    if args.ncu_step:      # profiling aid (`ncu --profile-from-start off`): warm up, then ONE eager training step between cudaProfilerStart/Stop
        model.use_cuda_graph_training = False
        for p_ in model._train_plans.values():
            p_.use_graph = False
        for i in range(3):
            step(i)
        for p_ in model._train_plans.values():
            p_.use_graph = False
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step(3)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return 0
    step(0)                                   # set-up: builds the plans
    sync_all()
    tuned = {}
    if not args.no_autotune and not args.no_graph:
        for p_ in model._train_plans.values():
            tuned = p_.autotune()             # set-up: CTA bounds of the side-branch kernels, picked by timing the replayed graphs
    for i in range(max(warmup, 3)):           # W warm-up steps (the first ones also capture the forward / backward CUDA graphs)
        lv = step(i)
    sync_all()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):               # exactly K timed steps
        lv = step(i)
        if i == 0:
            lv_first = lv
    e1.record()
    sync_all()
    clocks = sampler.stop() if rank == 0 else None
    outputs = dict(lv, parameters=model._flat_parameters.data.cpu().numpy()) if args.dump_outputs and rank == 0 else None
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / args.steps
    value = world * N * args.steps / (ms_total / 1e3)

    # ---- end to end: pinned host uint8 crops in (H2D inside the timed region), loss values out (the reference's three .item() reads)
    e2e_steps = args.steps
    copy_stream = torch.cuda.Stream(device=dev)
    stage = [torch.empty((N, H, W, 3), dtype=torch.uint8, device=dev) for _ in range(2)]
    sync_all()
    t0 = time.perf_counter()
    with torch.cuda.stream(copy_stream):
        stage[0].copy_(host_pool[0], non_blocking=True)
    ev = [torch.cuda.Event(), torch.cuda.Event()]
    ev[0].record(copy_stream)
    for i in range(e2e_steps):
        if i + 1 < e2e_steps:                 # prefetch the next batch while this one trains
            with torch.cuda.stream(copy_stream):
                stage[(i + 1) % 2].copy_(host_pool[(i + 1) % 2], non_blocking=True)
            ev[(i + 1) % 2].record(copy_stream)
        torch.cuda.current_stream().wait_event(ev[i % 2])
        step(i, x=stage[i % 2])
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * N * e2e_steps / float(te.item())
    ann_bytes = int(sum(a[0].nbytes + a[1].nbytes for a in anns[0]))

    # ---- all-reduce of the flat gradient buffer alone (what the collective costs inside the step)
    flat = model._flat_parameters
    ar_us = None
    if world > 1:
        sync_all()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(20):
            dist.all_reduce(flat.grad)
        a1.record()
        sync_all()
        ar = torch.tensor([a0.elapsed_time(a1) / 20 * 1e3], dtype=torch.float64, device=dev)
        dist.all_reduce(ar, op=dist.ReduceOp.MAX)
        ar_us = float(ar.item())
    if rank != 0:
        if world > 1:
            dist.barrier()
        return 0

    # ---- label assignment: native kernel vs the reference's CPU annotation_to_target (oracle restatement), one batch
    from oracle import lfd_oracle as orc
    sizes = model._sizes()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(10):
        model._assign(sizes, [a[0] for a in anns[0]], [a[1] for a in anns[0]], dev)
    torch.cuda.synchronize()
    assign_ms = (time.perf_counter() - t0) * 1e3 / 10
    t0 = time.perf_counter()
    for a in anns[0][:4]:                     # one image at a time, like the reference's python loop (lfd.py:121-150)
        orc.assign_targets(orc.CONFIGS[wl['cfg']], sizes, a[0], a[1])
    assign_cpu_ms = (time.perf_counter() - t0) * 1e3 / 4 * N

    # ---- live per-op roofline of the forward and backward plans (eager passes with an event pair around every launch)
    pk = peaks()
    plan = list(model._train_plans.values())[0]
    table = []
    for which, ops in (('fwd', plan.fwd_ops), ('bwd', plan.bwd_ops)):
        acc = np.zeros(len(ops))
        for rep in range(4):
            ms = plan.profile(which)
            if rep:
                acc += np.asarray(ms)
        for op, ms in zip(ops, acc / 3):
            b, f = train_op_algorithmic(op, N)
            table.append(dict(op=op, which=which, ms=float(ms), bytes=b, flops=f, t_bound_ms=max(b / (pk['hbm_gbs'] * 1e9), f / (pk['bf16_tflops'] * 1e12)) * 1e3))
    top = sorted(table, key=lambda r: -r['ms'])[0]
    hbm_bound = top['bytes'] / (pk['hbm_gbs'] * 1e9) >= top['flops'] / (pk['bf16_tflops'] * 1e12)
    if hbm_bound:
        achieved, peak, unit = top['bytes'] / (top['ms'] * 1e-3) / 1e9, pk['hbm_gbs'], 'GB/s'
    else:
        achieved, peak, unit = top['flops'] / (top['ms'] * 1e-3) / 1e12, pk['bf16_tflops'], 'TFLOP/s'
    sum_ms = float(sum(r['ms'] for r in table))
    by_kind = {}
    for r in table:
        kname = ('dgrad' if (r['which'] == 'bwd' and _TOP_NAMES[r['op']['kind']] == 'conv') else _TOP_NAMES[r['op']['kind']])
        e = by_kind.setdefault(kname, dict(ms=0.0, bound_ms=0.0, launches=0))
        e['ms'] += r['ms']; e['bound_ms'] += r['t_bound_ms']; e['launches'] += 1
    net_bound_ms = float(sum(r['t_bound_ms'] for r in table))
    roofline = dict(bound='hbm' if hbm_bound else 'tensor', achieved=achieved, peak=peak, unit=unit, frac=achieved / peak, traffic=None,
                    peak_source=pk['source'], kernel='%s (%s)' % (train_op_name(top['op']), top['which']), kernel_ms=top['ms'],
                    kernel_share_of_step=top['ms'] / sum_ms, algorithmic_bytes=top['bytes'], algorithmic_flops=top['flops'],
                    net=dict(layerwise_bound_ms=net_bound_ms, plan_ms_eager_sum=sum_ms, frac_of_layerwise_bound=net_bound_ms / sum_ms,
                             frac_of_layerwise_bound_in_step=net_bound_ms / ms_step,
                             by_kind={k: dict(ms=round(v['ms'], 4), bound_ms=round(v['bound_ms'], 4), launches=v['launches']) for k, v in sorted(by_kind.items())}))
    if args.profile_ops:
        for r in table:
            sys.stderr.write('%s %-44s %8.3f ms  bound %7.3f ms  %5.1f%%\n' % (r['which'], train_op_name(r['op']), r['ms'], r['t_bound_ms'], 100 * r['t_bound_ms'] / max(r['ms'], 1e-9)))
        sys.stderr.write('sum of plan ops %.3f ms; step %.3f ms\n' % (sum_ms, ms_step))
    launches = len(plan.fwd_ops) + len(plan.bwd_ops) + 5 + 2      # + assign, 2 loss kernels, 2 memsets; + sqnorm, sgd
    line = dict(metric=metric, value=value, unit='images/s', n_gpus=world, steps=args.steps, warmup=warmup, ms_per_step=ms_step, higher_is_better=True,
                scaling='weak', vs_baseline=None, dtype=wl['dtype'], data='synthetic', config=config,
                impl_detail=dict(timed_s=ms_total / 1e3, loss_first_last=[lv_first['loss'], lv['loss']],
                                 cuda_graph=bool(model.use_cuda_graph_training), launches_per_step=launches,
                                 side_branch_ctas={k: {str(b): c for b, c in v['ctas'].items()} for k, v in tuned.items()},
                                 workspace_gb=plan.workspace_bytes / 1e9, parameters=int(flat.numel),
                                 l2='the %.1f GB activation / gradient workspace is rewritten every step; inputs rotate over %d batches' % (plan.workspace_bytes / 1e9, npool),
                                 label_assign_ms=assign_ms, label_assign_reference_cpu_ms=assign_cpu_ms,
                                 label_assign_note='native lfd_assign_targets incl. the H2D copy of the boxes vs the oracle restatement of '
                                                   'annotation_to_target (lfd.py:109-259) on the host, same batch',
                                 allreduce_us=ar_us, allreduce_bytes=int(flat.numel * 4)),
                clocks=clocks, gpu_launches=launches * args.steps,
                e2e=dict(value=e2e_value, unit='images/s', h2d_bytes_per_step=N * H * W * 3 + ann_bytes, d2h_bytes_per_step=12, steps=e2e_steps,
                         host_numa_node=numa_node, note='pinned host uint8 crops -> device (prefetched on a copy stream) -> training step -> loss values on the host'),
                roofline=roofline)
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_train_leg(wl, 3, 1, 2, budget_s=20.0)
        line['cpu_baseline'] = dict(value=r['ips'], unit='images/s', cores=r['cores'], kind='port',
                                    sample='2 crops 640x640 per step, %d steps (ATen fp32 forward + autograd + oracle losses + clip + SGD on the host)' % r['done'])
    print(json.dumps(line))
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.barrier()
    return 0


def build_model(cfg_name):
    from helpers import synth_model
    model, sd = synth_model(cfg_name, cls_bias=-1.0)
    return model, sd


def reference_nms():
    """The REFERENCE's own compiled CPU NMS (lfd/model/utils/build/nms/src/cpu/nms_cpu.cpp, built by oracle/build_ref.py into
    oracle/_ref/nms_ext_ref.so, which travels to the GPU box) as a drop-in for the oracle's numpy NMS; None when absent."""
    try:
        from oracle import build_ref
        mod = build_ref.load_module()
    except Exception:
        mod = None
    if mod is None:
        return None, None
    return (lambda dets, thr: mod.nms(torch.from_numpy(np.ascontiguousarray(dets, np.float32)), float(thr)).numpy()), build_ref.so_path()


def cpu_leg(wl, sd, steps, warmup, frames_per_step, budget_s=None):
    """The reference's CPU path for this workload: fp32 forward (oracle PORT: the same ATen conv / norm calls the reference
    modules make) + decode + class-aware NMS with the REFERENCE's compiled nms_cpu.cpp when oracle/_ref/nms_ext_ref.so is
    present (numpy restatement otherwise).  With a `budget_s`, the thread calibration and the timed loop stop early once
    that many seconds have passed."""
    import synth
    from oracle import lfd_oracle as orc
    cfg = orc.CONFIGS[wl['cfg']]
    x = synth.synth_input(frames_per_step, wl['H'], wl['W'])
    nms_fn, nms_so = reference_nms()
    # "all the host threads it can use": PyTorch's CPU convs stop scaling (and then collapse) well before 128 threads on these
    # feature maps, so the thread count is calibrated on the REAL step batch (second of two forwards) and reported as `cores`.
    ncpu = os.cpu_count() or 1
    best = (None, 1e30)
    t_cal = time.time()
    for nt in sorted(set([min(ncpu, c) for c in (8, 16, 32, 64, ncpu)])):
        torch.set_num_threads(nt)
        orc.forward(cfg, sd, x[:1])
        t0 = time.time()
        orc.forward(cfg, sd, x)
        dt = time.time() - t0
        if dt < best[1]:
            best = (nt, dt)
        if budget_s is not None and time.time() - t_cal > 0.4 * budget_s:
            break
    torch.set_num_threads(best[0])
    meta = [dict(resized_height=wl['H'], resized_width=wl['W'], resize_scale=1.0) for _ in range(frames_per_step)]
    pf = wl.get('pass_fraction', PASS_FRACTION)

    def step():
        cls, reg, sizes = orc.forward(cfg, sd, x)
        if cfg['head']['classification_loss_type'] == 'FocalLoss':
            sc = cls.sigmoid()
        else:
            sc = cls.softmax(-1)[..., :-1]
        thr = float(torch.quantile(sc.flatten()[:200000], 1.0 - pf))
        orc.get_results(cfg, cls, reg, sizes, meta, thr, IOU_THR, nms_fn=nms_fn)
    for _ in range(warmup):
        step()
    t0 = time.time()
    done = 0
    for _ in range(steps):
        step()
        done += 1
        if budget_s is not None and time.time() - t0 > budget_s and done >= 2:
            break
    dt = time.time() - t0
    return dict(ips=frames_per_step * done / dt, ms=dt / done * 1e3, done=done, cores=best[0],
                nms='reference nms_cpu.cpp (oracle/_ref/nms_ext_ref.so)' if nms_fn is not None else 'oracle numpy restatement',
                native_so=nms_so)


def workload_config(wl, dtype, world):
    """The keys both arms (ours and --impl reference) print under `config`: what is computed, not how."""
    return dict(workload=wl['name'], model=wl['cfg'], frames_per_step_per_gpu=wl['N'], height=wl['H'], width=wl['W'], dtype=dtype,
                input='synthetic uint8 BGR frames (tests/synth.py weights; no network for datasets / checkpoints)',
                step='forward (backbone + neck + head) + score / decode / class-aware NMS of one batch',
                score_thr='calibrated so that %.3f%% of the (point, class) scores pass' % (100 * wl.get('pass_fraction', PASS_FRACTION)),
                iou_thr=IOU_THR, parallelism='batch-sharded replicas x%d, no collective on the inference path' % world)


def detections(results, n):
    """The valid rows of one batch's post-process results (dets [N,cap,5], labels [N,cap], src [N,cap], count [N + 1]) on the
    host, image after image; `count` keeps its last entry, the capacity-overflow flag."""
    dets, labels, src, count = (t.cpu().numpy() for t in results)
    valid = [slice(0, int(k)) for k in count[:n]]
    return dict(dets=np.concatenate([dets[i, v] for i, v in enumerate(valid)]),
                labels=np.concatenate([labels[i, v] for i, v in enumerate(valid)]),
                src=np.concatenate([src[i, v] for i, v in enumerate(valid)]), count=count)


def dump_outputs(out_dir, outputs):
    """--dump-outputs: every array as out_dir/<name>.npy; float32 arrays as they are, anything else (integers, python floats) as
    float64, which holds those values exactly."""
    arrays = {k: np.asarray(v) for k, v in outputs.items()}
    arrays = {k: a if a.dtype == np.float32 else a.astype(np.float64) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError('--dump-outputs: %d bytes of outputs, more than the %d allowed' % (total, DUMP_MAX_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='WIDERFACE_S', choices=sorted(WORKLOADS) + sorted(TRAIN_WORKLOADS))
    ap.add_argument('--dtype', default=None, choices=['bf16', 'fp16'], help="16-bit storage type of the plan (default: the workload's)")
    ap.add_argument('--conv-impl', default='umma', choices=['umma', 'simt'])
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-autotune', action='store_true', help='skip InferencePlan.autotune (CTA bounds of the side-branch convs)')
    ap.add_argument('--profile-ops', action='store_true', help='print the per-op timing table to stderr')
    ap.add_argument('--ncu-step', action='store_true',
                    help='for `ncu --profile-from-start off`: warm up, then ONE eager step between cudaProfilerStart/Stop, and exit')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last timed step returned (rank 0) as DIR/<name>.npy: the detections of the '
                         'inference configs, the loss values and the flat parameters of the training config')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'ours' or args.ncu_step):
        ap.error('--dump-outputs writes the outputs of the timed GPU steps: it needs --impl ours and no --ncu-step')
    if args.config in TRAIN_WORKLOADS:
        return train_main(args)
    wl = WORKLOADS[args.config]
    dtype = args.dtype or wl['dtype']
    rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    warmup = max(args.warmup, 3)
    metric = 'images/sec %s %s' % (wl['name'], dtype)
    config = workload_config(wl, dtype, max(world, args.gpus))

    if args.impl == 'reference':
        if rank != 0:
            return 0
        model, sd = build_model(wl['cfg'])
        frames = wl['N']
        r = cpu_leg(wl, sd, args.steps, warmup, frames)
        line = dict(metric=metric, value=r['ips'], unit='images/s', n_gpus=args.gpus, steps=r['done'], warmup=warmup, ms_per_step=r['ms'],
                    higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32', data='synthetic', impl='reference',
                    config=config,
                    impl_detail=dict(note='CPU path of the reference: PyTorch fp32 forward (oracle port of the reference modules) '
                                          '+ decode + class-aware NMS', nms=r['nms'],
                                     threads='calibrated on the %d-frame step batch over {8,16,32,64,all} host threads' % frames),
                    cpu_baseline=dict(value=r['ips'], unit='images/s', cores=r['cores'], kind='port',
                                      sample='%d frames per step, %d steps; NMS: %s' % (frames, r['done'], r['nms'])),
                    e2e=dict(value=r['ips'], unit='images/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
        print(json.dumps(line))
        return 0

    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (there is no CPU fallback for the product path)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        import torch.distributed as dist
        init_nccl(dev)
    from lfd import _native as nat
    from lfd.pipeline import ForwardPostPipeline, StreamingDetector, bind_host_to_gpu_numa_node
    import synth
    numa_node = bind_host_to_gpu_numa_node(dev)     # before any pinned allocation: host pools land on the GPU's NUMA node
    model, sd = build_model(wl['cfg'])
    model.to(dev)
    model.conv_impl = nat.CONV_SIMT if args.conv_impl == 'simt' else nat.CONV_UMMA
    model.act_dtype = dtype
    model.use_cuda_graph = not args.no_graph
    model.max_detections_per_image = wl.get('cap', 8192)
    pass_fraction = wl.get('pass_fraction', PASS_FRACTION)
    N, H, W = wl['N'], wl['H'], wl['W']
    npool = wl.get('pool', POOL)
    g = torch.Generator().manual_seed(1000 + rank)
    host_pool = [torch.randint(0, 256, (N, H, W, 3), generator=g, dtype=torch.uint8).pin_memory() for _ in range(2)]
    pool = [torch.randint(0, 256, (N, H, W, 3), generator=g, dtype=torch.uint8).to(dev) for _ in range(npool)]
    plan = model.inference_plan(N, H, W, dev)
    if not args.no_autotune and not args.no_graph and not args.ncu_step:
        plan.autotune()                     # set-up: CTA bounds of the side-branch convs, picked by timing the replayed graph
    for i, hw in enumerate(plan.level_sizes):
        model._head_indexes_to_feature_map_sizes[i] = hw
    post = model.post_plan(N, plan.level_sizes, dev)
    post.set_meta([W] * N, [H] * N, [1.0] * N)
    with torch.no_grad():
        cls, _ = plan.forward(pool[0], use_graph=False)
        scores = cls.sigmoid() if plan.cls_channels == model._num_classes else cls.softmax(-1)[..., :-1]
        score_thr = float(torch.quantile(scores.flatten()[:2000000].float(), 1.0 - pass_fraction))
    # one step = forward + post-process of one batch; over consecutive batches the (latency-bound) post-process of batch i
    # runs on a second stream next to the forward of batch i+1 (lfd/pipeline.py), as a serving loop would do it
    pipe = ForwardPostPipeline(model, plan, post, score_thr, IOU_THR)

    def step(i):
        return pipe.enqueue(pool[i % npool])

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    if args.ncu_step:      # profiling aid, prints no bench line
        model.use_cuda_graph = False
        with torch.no_grad():
            for i in range(4):
                step(i)
            torch.cuda.synchronize()
            torch.cuda.profiler.start()
            step(4)
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
        return 0
    with torch.no_grad():
        for i in range(npool):                 # set-up, not warm-up: instantiates one CUDA graph per (pool buffer, output slot) pair;
            step(i)                            # the slots alternate per step, so the pool is walked twice with one step in between
        step(0)
        for i in range(npool):
            step(i)
        for i in range(warmup):                # the W warm-up steps
            step(i)
        sync_all()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(pipe.fwd_stream)
        for i in range(args.steps):            # exactly K timed steps
            results = step(i)
        e1.record(pipe.post_stream)
        sync_all()
        clocks = sampler.stop() if rank == 0 else None
        counts = post.count.tolist()
        # the post-process buffers are rewritten by the end-to-end pass below: take the last timed step's detections now
        outputs = detections(results, N) if args.dump_outputs and rank == 0 else None
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)       # the slowest rank
    ms_total = float(t.item())
    ms_step = ms_total / args.steps
    value = world * N * args.steps / (ms_total / 1e3)

    # ---- end to end: pinned host frames in, host detections out, copies inside the timed region
    det = StreamingDetector(model, N, H, W, score_thr, IOU_THR, max_out=1024, device=dev)
    e2e_steps = args.steps
    with torch.no_grad():
        for i in range(3):
            det.infer(host_pool[i % 2])
        sync_all()
        t0 = time.perf_counter()
        pending = []                           # up to depth - 1 batches stay in flight behind the one being submitted
        host_submit_s = 0.0
        for i in range(e2e_steps):
            ts = time.perf_counter()
            pending.append(det.submit(host_pool[i % 2]))
            host_submit_s += time.perf_counter() - ts
            if len(pending) >= det.depth:
                det.collect(pending.pop(0))
        while pending:
            out = det.collect(pending.pop(0))
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * N * e2e_steps / float(te.item())
    # how long the host->device copy of one batch takes on its own (diagnostic: is e2e bound by the PCIe link?)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(10):
        det.stage_input(i % 2, host_pool[i % 2])      # on the detector's copy streams
    torch.cuda.synchronize()
    h2d_ms = (time.perf_counter() - t0) * 1e3 / 10
    h2d_all = torch.tensor([det.h2d_bytes / (h2d_ms * 1e-3) / 1e9], dtype=torch.float64, device=dev)
    if world > 1:
        gathered = [torch.zeros_like(h2d_all) for _ in range(world)]
        dist.all_gather(gathered, h2d_all)
        h2d_per_rank = [round(float(v.item()), 1) for v in gathered]
    else:
        h2d_per_rank = [round(float(h2d_all.item()), 1)]

    if rank != 0:
        if world > 1:
            dist.barrier()
        return 0

    # ---- live per-op roofline (eager pass with an event pair around every launch)
    pk = peaks()
    n_ops = plan.num_launches
    acc = np.zeros(n_ops, np.float64)
    buf = (C.c_float * n_ops)()
    reps = 5
    with torch.no_grad():
        for rep in range(reps + 1):
            nat.check(nat.lib().lfd_plan_profile(plan.handle, nat.ptr(pool[rep % npool]), nat.INPUT_U8_NHWC, nat.ptr(plan.workspace),
                                                 nat.ptr(plan.cls_out), nat.ptr(plan.reg_out), buf, nat.stream_ptr()))
            if rep:
                acc += np.frombuffer(buf, dtype=np.float32)
    per_op_ms = acc / reps
    rows = plan.describe()
    table = []
    for row, ms in zip(rows, per_op_ms):
        b, f = op_algorithmic(row, N, 3)
        t_bound = max(b / (pk['hbm_gbs'] * 1e9), f / (pk['bf16_tflops'] * 1e12))
        table.append(dict(row=row, ms=float(ms), bytes=b, flops=f, t_bound_ms=t_bound * 1e3))
    table_sorted = sorted(table, key=lambda r: -r['ms'])
    top = table_sorted[0]
    hbm_bound = top['bytes'] / (pk['hbm_gbs'] * 1e9) >= top['flops'] / (pk['bf16_tflops'] * 1e12)
    if hbm_bound:
        achieved, peak, unit = top['bytes'] / (top['ms'] * 1e-3) / 1e9, pk['hbm_gbs'], 'GB/s'
    else:
        achieved, peak, unit = top['flops'] / (top['ms'] * 1e-3) / 1e12, pk['bf16_tflops'], 'TFLOP/s'
    sum_ms = float(per_op_ms.sum())
    conv_ms = float(sum(r['ms'] for r in table if r['row']['kind'] == 'conv'))
    net_bound_ms = float(sum(r['t_bound_ms'] for r in table))
    total_bytes, total_flops = sum(r['bytes'] for r in table), sum(r['flops'] for r in table)
    dp = directional_peaks(dev)
    dir_bound_ms = 0.0
    for r in table:
        rd, wr = op_read_write(r['row'], N, 3)
        r['t_dir_ms'] = 1e3 * max(r['flops'] / (pk['bf16_tflops'] * 1e12), (rd + wr) / (pk['hbm_gbs'] * 1e9), rd / (dp['read_only_gbs'] * 1e9),
                                  wr / (dp['write_only_gbs'] * 1e9))
        dir_bound_ms += r['t_dir_ms']
    kname = op_name(top['row'])
    roofline = dict(bound='hbm' if hbm_bound else 'tensor', achieved=achieved, peak=peak, unit=unit, frac=achieved / peak,
                    traffic=ncu_traffic(args.config, dtype, kname),
                    peak_source=pk['source'],
                    kernel=kname,
                    kernel_ms=top['ms'], kernel_share_of_step=top['ms'] / sum_ms, algorithmic_bytes=top['bytes'], algorithmic_flops=top['flops'],
                    net=dict(layerwise_bound_ms=net_bound_ms, forward_ms_eager_sum=sum_ms, frac_of_layerwise_bound=net_bound_ms / sum_ms,
                             frac_of_layerwise_bound_in_graph=net_bound_ms / ms_step,
                             directional_peaks=dp, directional_bound_ms=dir_bound_ms, frac_of_directional_bound_in_graph=dir_bound_ms / ms_step,
                             directional_note='per layer max(flops / peak, (R + W) / copy peak, R / read-only peak, W / write-only peak): the bound '
                                              'a layer with a lopsided read / write mix can actually reach',
                             conv_share=conv_ms / sum_ms, algorithmic_gb=total_bytes / 1e9, algorithmic_gflop=total_flops / 1e9,
                             hbm_view=total_bytes / (ms_step * 1e-3) / 1e9 / pk['hbm_gbs'],
                             tensor_view=total_flops / (ms_step * 1e-3) / 1e12 / pk['bf16_tflops']))
    if args.profile_ops:
        for r in table:
            row = r['row']
            sys.stderr.write('%-10s k%d s%d %3d->%3d%s %4dx%-4d res=%d  %8.3f ms  bound %7.3f ms  %5.1f%%  %7.1f GB/s %7.1f TF/s\n' % (
                row['kind'], row['ksize'], row['stride'], row['Cin'], row['Cout'], ('->%3d' % row['tail_cout']) if row.get('tail_cout') else '     ', row['Ho'], row['Wo'], int(row['res']), r['ms'], r['t_bound_ms'],
                100 * r['t_bound_ms'] / max(r['ms'], 1e-9), r['bytes'] / (r['ms'] * 1e-3) / 1e9, r['flops'] / (r['ms'] * 1e-3) / 1e12))
        sys.stderr.write('sum of ops %.3f ms; graph step (incl. post-process) %.3f ms\n' % (sum_ms, ms_step))

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_leg(wl, sd, 50, 1, 1, budget_s=20.0)
        cpu = dict(value=r['ips'], unit='images/s', cores=r['cores'], kind='port',
                   sample='1 frame %dx%d per step, %d steps (forward fp32 + decode + NMS [%s] on the host)' % (W, H, r['done'], r['nms']))
    line = dict(metric=metric, value=value, unit='images/s', n_gpus=world, steps=args.steps, warmup=warmup, ms_per_step=ms_step,
                higher_is_better=True, scaling='weak', vs_baseline=None, dtype=dtype, data='synthetic',
                config=config,
                impl_detail=dict(score_thr=score_thr, detections_last_step=counts[:N],
                                 timed_s=ms_total / 1e3,
                                 setup_steps=2 * npool + 1,
                                 l2='inputs rotate over a %d-batch pool (%.0f MB > L2); the %.0f MB activation workspace is rewritten every step'
                                    % (npool, npool * N * H * W * 3 / 1e6, plan.workspace_bytes / 1e6),
                                 cuda_graph=model.use_cuda_graph, conv_impl=args.conv_impl, launches_per_step=plan.num_launches + 2,
                                 side_branch_ctas={str(b): c for b, c in plan.side_ctas.items()},
                                 autotune=[(k, round(v, 4)) for k, v in getattr(plan, 'autotune_log', [])],
                                 pipelining='post-process of batch i overlaps the forward of batch i+1 (two streams, two output slots)'),
                clocks=clocks, gpu_launches=(plan.num_launches + 2) * args.steps,
                e2e=dict(value=e2e_value, unit='images/s', h2d_bytes_per_step=det.h2d_bytes, d2h_bytes_per_step=det.d2h_bytes, steps=e2e_steps,
                         h2d_copy_alone_ms=h2d_ms, h2d_gbps=det.h2d_bytes / (h2d_ms * 1e-3) / 1e9, h2d_gbps_per_rank=h2d_per_rank,
                         copy_streams=len(det.copy_streams), host_numa_node=numa_node, host_submit_ms_per_step=host_submit_s / e2e_steps * 1e3,
                         note='pinned host uint8 frames -> device -> detections -> pinned host; copy / forward / post-process pipelined on three streams'),
                roofline=roofline)
    if cpu is not None:
        line['cpu_baseline'] = cpu
    print(json.dumps(line))
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.barrier()
    return 0


if __name__ == '__main__':
    sys.exit(main())
