#!/usr/bin/env python
"""bench.py -- headline benchmark of the Cold-Diffusion hot path on B200 (contract: see the task brief).

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...     # the reference algorithm (oracle port) on the host cores
    python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs DIR     # + what the last timed step computed, as DIR/*.npy

Workload (BASELINE.json config 3, "C3"): CelebA-128 deblurring, Unet(dim 64, mults (1,2,4,8), 3 channels),
T=200, Exponential_reflect k=15 std=0.01, x0_step_down; synthetic U(-1,1) images, random-init weights.
A "step" is ONE optimizer step of Trainer.train (DB:1188-1204): 2 micro-batches x 32 images per GPU of
p_losses forward + backward, one gradient all-reduce (N>1), fused Adam + EMA.  `value` = images/sec over all
GPUs with the batches already resident in HBM; `e2e` = the same through the public Trainer.train_step call with
pinned-host batches copied H2D and the loss read back D2H inside the timed region (two untimed steps of that path first).  At
N > 1 the all-reduce of every finished suffix of the flat gradient buffer overlaps the rest of the backward.  Nothing is skipped
inside a timed region.

Both arms print the SAME `metric` string, unit and workload so that the driver can divide them.  The reference arm
(`--impl reference`) times the reference algorithm (oracle/: the eager-PyTorch restatement of the reference's p_losses, 200-step
Python q_sample loop included; the reference itself is Python under /root/reference and does not exist on the GPU box) on the host
cores at a bounded batch per step.  The same restatement on cuda:0 at the full micro-batch of 32 -- how the reference is deployed,
cuDNN / cuBLAS eager -- is measured once per single-GPU run and reported as `reference_eager_b200` (the comparator SURVEY 8d
calls the real bar).  The sampling half of the metric is one complete `GaussianDiffusion.sample(batch_size=32, img=...)` call of
200 reverse steps through the public API (`sample`).  `op_profile` is the in-situ time per C-ABI entry point of one step.
All kernels run in their default configuration (no start-up tuning).
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

C3 = dict(dim=64, dim_mults=(1, 2, 4, 8), channels=3, image_size=128, timesteps=200, kernel_size=15, kernel_std=0.01,
          blur_routine='Exponential_reflect', sampling_routine='x0_step_down', batch=32, accum=2)
FWD_GFLOP_PER_IMG = 67.41          # BASELINE.md section 2 (torch FlopCounterMode on the reference Unet)
TRAIN_GFLOP_PER_IMG = 3 * FWD_GFLOP_PER_IMG


def read_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d, 'measured'
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0), 'fallback'


class ClockSampler(threading.Thread):
    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag = gpu, [], False

    def run(self):
        q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        while not self.stop_flag:
            try:
                o = subprocess.run(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + q, '--format=csv,noheader,nounits'],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([c.strip() for c in o.split(',')])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        import statistics
        sm = [float(r[0]) for r in self.rows if r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith('active') for r in self.rows if len(r) >= 6)]
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(self.rows))


# ------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference algorithm (oracle port; the reference itself is pure Python
# under /root/reference, absent on the GPU box) on the host cores
# ------------------------------------------------------------------------------------------------------
def cpu_train_sample(batch=2, steps=1, warmup=0, threads=None, device='cpu'):
    """times p_losses forward + backward + Adam of config 3 with the eager-PyTorch restatement of the reference (oracle/) at a
    bounded batch; -> (img/s, info).  device='cpu' is the contract's CPU baseline; device='cuda' (bench.py --impl reference
    --reference-device cuda, informational) runs the same eager PyTorch code on the GPU, which is how the reference is deployed."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import unet_oracle as UO
    import deblur_oracle as DO
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count()
    calibrate = threads is None and device == 'cpu'
    threads = threads or avail
    torch.set_num_threads(threads)
    dev = torch.device(device)
    sd = {k: v.clone().to(dev).requires_grad_(True) for k, v in UO.make_unet_state_dict(C3['dim'], C3['dim_mults'], C3['channels']).items()}
    orc = DO.DeblurOracle(lambda a, b: UO.unet_forward(sd, a, b), image_size=C3['image_size'], channels=3,
                          timesteps=C3['timesteps'], kernel_std=C3['kernel_std'], kernel_size=C3['kernel_size'],
                          blur_routine=C3['blur_routine'], sampling_routine=C3['sampling_routine']).to(dev)
    opt = torch.optim.Adam(list(sd.values()), lr=2e-5)
    g = torch.Generator().manual_seed(1234)
    sync = torch.cuda.synchronize if dev.type == 'cuda' else (lambda: None)
    times = []
    tried = ''
    if calibrate:
        # eager PyTorch on "all cores" of a many-core host can be far slower than on a few (round 1 measured 0.059 images/s with 128
        # threads on the GPU box against ~0.9 with 8 threads elsewhere): one untimed step per candidate thread count, keep the fastest
        best = None
        for n in sorted({c for c in (8, 16, 32, 64, avail) if c <= avail} or {avail}):
            torch.set_num_threads(n)
            x = torch.rand(batch, 3, 128, 128, generator=g) * 2 - 1
            t = torch.randint(0, C3['timesteps'], (batch,), generator=g)
            t0 = time.time()
            orc.p_losses(x, t).backward()
            opt.step(); opt.zero_grad()
            dt = time.time() - t0
            tried += ' %d:%.1fs' % (n, dt)
            if best is None or dt < best[0]:
                best = (dt, n)
            if dt > 60:                  # bounded sample: do not walk further up a slope that is already this slow
                break
        threads = best[1]
        torch.set_num_threads(threads)
        warmup = 0                       # the calibration steps were the warm-up
    for it in range(warmup + steps):
        x = (torch.rand(batch, 3, 128, 128, generator=g) * 2 - 1).to(dev)
        t = torch.randint(0, C3['timesteps'], (batch,), generator=g).to(dev)
        sync()
        t0 = time.time()
        loss = orc.p_losses(x, t)
        loss.backward()
        opt.step(); opt.zero_grad()
        sync()
        if it >= warmup:
            times.append(time.time() - t0)
    sec = sum(times) / len(times)
    return batch / sec, dict(cores=threads, sample='p_losses fwd+bwd+Adam, config-3 network, batch %d x %d step(s), T=200 q_sample%s'
                             % (batch, steps, ('; threads tried (one step each)' + tried + ' of %d available' % avail) if tried else ''),
                             ms_per_step=sec * 1e3)


METRIC = "training-step images/sec (CelebA-128 deblur UNet, config 3)"
WORKLOAD = "C3: CelebA-128 deblur train step = 2 micro-batches x 32 img/GPU (p_losses fwd+bwd) + grad all-reduce + Adam + EMA"
REF_CPU_BATCH = 4          # images per reference step on the host cores (a full 64-image step takes ~20 s of CPU)


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    on_gpu = args.reference_device == 'cuda'
    nb = 32 if on_gpu else REF_CPU_BATCH
    v, info = cpu_train_sample(batch=nb, steps=max(1, args.steps), warmup=max(1, args.warmup) if on_gpu else min(1, args.warmup),
                               device=args.reference_device)
    where = "cuda:0" if on_gpu else "the host cores"
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "images/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": info['ms_per_step'],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "net": "Unet(dim=64, dim_mults=(1,2,4,8), channels=3)", "T": 200,
                       "blur": "Exponential_reflect k=15 std=0.01",
                       "reference_sample": "bounded sample of that workload: %d images per step (p_losses fwd+bwd+Adam, same network, T=200 "
                                           "q_sample loop); eager PyTorch restatement of the reference on %s" % (nb, where),
                       "device": args.reference_device},
            "cpu_baseline": {"value": v, "unit": "images/s", "cores": info['cores'], "kind": "port", "sample": info['sample']},
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


DUMP_SAMPLE = 1 << 21      # weights drawn per network by --dump-outputs: <= 8 MB of float32 out of the 226 MB of config 3


def dump_outputs(out_dir, loss, nets):
    """writes the loss of the last timed step and, for every net, a fixed seeded sample of its weights after that step (all
    tensors of state_dict() flattened in key order: the reference layout, whatever layout the engine keeps internally)"""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'loss.npy'), np.asarray([loss.item()], dtype=np.float32))
    for name, net in nets.items():
        with torch.no_grad():
            flat = torch.cat([v.reshape(-1).float() for v in net.state_dict().values()])
            idx = np.unique(np.random.RandomState(0).randint(0, flat.numel(), DUMP_SAMPLE))
            np.save(os.path.join(out_dir, name + '.npy'), flat[torch.from_numpy(idx).to(flat.device)].cpu().numpy())


def _timed_loop(fn, n, sync):
    import torch
    sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(n):
        fn(s)
    e1.record()
    sync()
    return e0.elapsed_time(e1)


# ------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-sample', action='store_true', help='skip the 200-step sample() measurement (quick runs)')
    ap.add_argument('--no-others', action='store_true', help='skip the other BASELINE configs and the eager comparator (quick runs)')
    ap.add_argument('--no-autotune', action='store_true', help='accepted for compatibility; there is no start-up tuning any more')
    ap.add_argument('--reference-device', default='cpu', choices=['cpu', 'cuda'],
                    help="--impl reference only: 'cpu' (the contract) or 'cuda' = the same eager-PyTorch restatement on the GPU (informational)")
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed training step computed (its loss, seeded samples of the weights and EMA weights '
                         'after it) as DIR/<name>.npy; the inputs are seeded, so two builds can be compared output for output')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        return run_reference(args)

    import io
    import contextlib
    import torch
    import torch.distributed as dist
    import cold_diffusion_models_b200 as cdm
    from cold_diffusion_models_b200 import _lib

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    dev = torch.device('cuda', local)
    W = max(3, args.warmup)
    K = args.steps

    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        unet = cdm.Unet(dim=C3['dim'], dim_mults=C3['dim_mults'], channels=C3['channels']).to(dev)
        diffusion = cdm.GaussianDiffusion(unet, image_size=C3['image_size'], device_of_kernel='cuda', channels=3,
                                          timesteps=C3['timesteps'], loss_type='l1', kernel_std=C3['kernel_std'],
                                          kernel_size=C3['kernel_size'], blur_routine=C3['blur_routine'],
                                          train_routine='Final', sampling_routine=C3['sampling_routine'], discrete=False).to(dev)
        trainer = cdm.Trainer(diffusion, None, image_size=128, train_batch_size=C3['batch'], train_lr=2e-5,
                              train_num_steps=10 ** 9, gradient_accumulate_every=C3['accum'], ema_decay=0.995, fp16=False,
                              results_folder='/tmp/colddiff_bench_results', dataset='synthetic')
    B, A = C3['batch'], C3['accum']
    img_per_step = B * A

    # distinct batches so consecutive steps never re-read the same inputs; activations (>3 GB/step) exceed the 126 MB L2
    g = torch.Generator().manual_seed(1234 + rank)
    nb = 4
    host = [torch.rand(B, 3, 128, 128, generator=g).mul_(2).sub_(1).pin_memory() for _ in range(nb * A)]
    resident = [h.to(dev) for h in host]
    torch.manual_seed(1234 + rank)          # per-rank RNG stream for t (DB:980)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        ms = _timed_loop(fn, steps, sync_all)
        if world > 1:
            tt = torch.tensor([ms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = tt.item()
        return ms

    last_loss = [None]

    def step_resident(s):
        last_loss[0] = trainer.train_step(batches=[resident[(s * A + i) % (nb * A)] for i in range(A)])
        trainer.step += 1

    losses = []
    loss_host = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ev = [torch.cuda.Event() for _ in range(2)]

    def step_e2e(s):
        # every step copies its loss device -> pinned host (4 bytes, asynchronous) and the host reads it one step later, when the
        # copy has long completed: the D2H read of every step's result stays inside the timed region without draining the launch
        # queue at every step boundary (a blocking .item() per step exposes ~1 ms of kernel-launch latency)
        loss = trainer.train_step(batches=[host[(s * A + i) % (nb * A)] for i in range(A)])
        trainer.step += 1
        loss_host[s & 1].copy_(loss.detach(), non_blocking=True)
        loss_ev[s & 1].record()
        if s > 0:
            loss_ev[(s - 1) & 1].synchronize()
            losses.append(float(loss_host[(s - 1) & 1]))
        if s == K - 1:
            loss_ev[s & 1].synchronize()
            losses.append(float(loss_host[s & 1]))

    for s in range(W):
        step_resident(s)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    _lib.reset_launch_count()
    ms = timed(step_resident, K)
    launches = _lib.launch_count()
    if args.dump_outputs and rank == 0:     # before any later step moves the weights on
        dump_outputs(args.dump_outputs, last_loss[0], {'weights': unet, 'ema_weights': trainer.ema_model.denoise_fn})
    for s in range(2):                      # untimed: first use of the pinned batches / loss buffers / events of the end-to-end path
        wl = trainer.train_step(batches=[host[(s * A + i) % (nb * A)] for i in range(A)])
        trainer.step += 1
        loss_host[s & 1].copy_(wl.detach(), non_blocking=True)
        loss_ev[s & 1].record()
    sync_all()
    ms_e2e = timed(step_e2e, K)
    value = img_per_step * world * K / (ms / 1e3)
    e2e = img_per_step * world * K / (ms_e2e / 1e3)

    # ---- sampling half of the metric: ONE complete 200-step x0_step_down sample() through the public API per rank
    # (degradation of the input to x_T + 200 x [UNet forward + Algorithm-2 update]); CUDA-graph replay of the inference forward on
    ema = trainer.ema_model
    sample = None
    if not args.no_sample:
        ema.denoise_fn.engine.enable_cuda_graph(True)
        xs = resident[0]
        with torch.no_grad():
            ema.sample(batch_size=B, img=xs, t=3)                 # warm-up: graph capture, workspaces (3 reverse steps)
            ms_s = timed(lambda s_: ema.sample(batch_size=B, img=resident[1]), 1)
        ema.denoise_fn.engine.enable_cuda_graph(False)
        sample = {"value": B * world / (ms_s / 1e3), "unit": "images/s", "what": "GaussianDiffusion.sample(batch_size=32, img=...) per GPU: "
                  "200-step x0_step_down through the public API, timed whole (max over ranks)", "seconds_per_call": ms_s / 1e3,
                  "ms_per_reverse_step": ms_s / C3['timesteps'], "cuda_graph": True, "batch_per_gpu": B,
                  "tflops": B * world * 200 * FWD_GFLOP_PER_IMG / (ms_s / 1e3) / 1e3}
    if sampler:
        sampler.stop_flag = True

    # ---- context, rank 0 of a single-GPU run only: the other BASELINE configs that fit one GPU and the eager-PyTorch comparator
    others, eager = {}, None
    if rank == 0 and world == 1 and not args.no_others:
        others = other_configs(cdm, trainer, resident, dev, B)
        try:
            v, info = cpu_train_sample(batch=32, steps=2, warmup=1, device='cuda')
            eager = {"value": v, "unit": "images/s", "ms_per_micro_batch": info['ms_per_step'],
                     "what": "the reference algorithm as eager PyTorch (cuDNN / cuBLAS, TF32 convolutions allowed like torch's default) on this GPU: "
                             "p_losses fwd+bwd+Adam at micro-batch 32, 200-step Python q_sample loop included (oracle/ restatement)",
                     "ours_over_eager": value / v}
        except Exception as e:
            eager = {"error": repr(e)[:200]}
        torch.cuda.empty_cache()

    # ---- roofline of the dominant kernel (tcgen05 tap-list convolution), CUDA events around every launch --------
    peaks, peak_kind = read_peaks()
    roof = None
    eng = unet.engine
    if rank == 0:
        eng.profile_convs = []
    step_resident(0)                      # every rank takes part (the step contains the gradient all-reduce)
    torch.cuda.synchronize()
    if rank == 0:
        tot_ms = sum(a.elapsed_time(b) for (a, b, f) in eng.profile_convs)
        tot_fl = sum(f for (a, b, f) in eng.profile_convs)
        n_launch = len(eng.profile_convs)
        eng.profile_convs = None
        tf32_peak = peaks['bf16_tflops_sustained'] / 2.0     # kind::tf32 runs at half the bf16 rate
        ach = tot_fl / (tot_ms / 1e3) / 1e12
        traffic, traffic_src = None, None
        for name in ('conv_tc_traffic_r02.json', 'conv_tc_traffic_r01.json'):
            try:
                with open(os.path.join(ROOT, 'profiles', name)) as f:
                    traffic, traffic_src = json.load(f)['dram_bytes_per_launch'], name
                break
            except Exception:
                pass
        roof = {"bound": "tensor", "kernel": "conv_tc_kernel / conv_tc2_kernel / conv_tc4_kernel (tcgen05 kind::tf32 implicit GEMM; fwd + dgrad launches)",
                "achieved": ach, "peak": tf32_peak, "unit": "TFLOP/s", "frac": ach / tf32_peak, "traffic": traffic,
                "traffic_unit": "DRAM bytes per launch (ncu capture of one step, profiles/%s)" % traffic_src,
                "peak_source": "%s bf16_tflops_sustained / 2 (TF32 rate)" % peak_kind, "launches_timed": n_launch,
                "share_of_step_ms": tot_ms / (ms / K)}

    # ---- where one optimizer step goes, in situ (CUDA events around every C-ABI call, tools/op_profile.py's mechanism) ----
    op_profile = None
    try:
        if rank == 0:
            _lib.profile_start()
        step_resident(1)                  # every rank takes part (all-reduce)
        if rank == 0:
            prof = _lib.profile_stop()
            agg = {}
            for name, (calls, tms) in prof.items():
                base = name.split('(')[0]
                c0, t0_ = agg.get(base, (0, 0.0))
                agg[base] = (c0 + calls, t0_ + tms)
            top = sorted(agg.items(), key=lambda kv: -kv[1][1])[:14]
            op_profile = {"total_ms_with_events": round(sum(v[1] for v in agg.values()), 3),
                          "entry_points": {k: {"calls": v[0], "ms": round(v[1], 3)} for k, v in top}}
    except Exception as e:
        op_profile = {"error": repr(e)[:200]}
        try:
            _lib._prof = None
        except Exception:
            pass

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline:
            v, info = cpu_train_sample(batch=REF_CPU_BATCH, steps=2, warmup=0)
            cpu = {"value": v, "unit": "images/s", "cores": info['cores'], "kind": "port", "sample": info['sample']}
        line = {
            "metric": METRIC,
            "value": value, "unit": "images/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "tf32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "net": "Unet(dim=64, dim_mults=(1,2,4,8), channels=3)", "T": 200, "blur": "Exponential_reflect k=15 std=0.01",
                       "global_batch": img_per_step * world, "parallelism": "dp%d" % world,
                       "micro_batches": "%d x %d, gradients accumulated" % (A, B),
                       "l2": "inputs rotate over 4 distinct batch sets; per-step activations (>3 GB) exceed the 126 MB L2"},
            "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": img_per_step * 3 * 128 * 128 * 4,
                    "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / K, "last_loss": losses[-1] if losses else None,
                    "losses_read": len(losses),
                    "how": "Trainer.train_step on pinned-host batches (H2D inside the step); the step's loss is copied D2H every step and read by the host one step later"},
            "sample": sample,
            "gpu_launches": launches,
            "roofline": roof,
            "cpu_baseline": cpu,
            "reference_eager_b200": eager,
            "clocks": sampler.summary() if sampler else None,
            "train_tflops": value * TRAIN_GFLOP_PER_IMG / 1e3,
            "other_configs": others,
            "op_profile": op_profile,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def other_configs(cdm, trainer, resident, dev, B):
    """the other BASELINE configs that fit one GPU, as context (not the headline, bounded to a few steps; default kernels)"""
    import io
    import contextlib
    import torch
    others = {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def per_step(fn, warm, n):
        for s_ in range(warm):
            fn(s_)
        torch.cuda.synchronize()
        e0.record()
        for s_ in range(n):
            fn(s_)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    try:
        with contextlib.redirect_stdout(io.StringIO()):
            # config 2: CIFAR-10 32x32 deblur, DDPM `Model`, T=50 Special_6_routine, batch 128: train step (dropout 0.1 on) and sampling
            m2 = cdm.Model(resolution=32, in_channels=3, out_ch=3, ch=128, ch_mult=(1, 2, 2, 2), num_res_blocks=2,
                           attn_resolutions=(16,), dropout=0.1).to(dev)
            g2 = cdm.GaussianDiffusion(m2, image_size=32, device_of_kernel='cuda', channels=3, timesteps=50, loss_type='l1',
                                       kernel_std=0.1, kernel_size=3, blur_routine='Special_6_routine', train_routine='Final',
                                       sampling_routine='x0_step_down').to(dev)
            tr2 = cdm.Trainer(g2, None, image_size=32, train_batch_size=128, train_lr=2e-5, train_num_steps=10 ** 9,
                              gradient_accumulate_every=2, results_folder='/tmp/colddiff_bench_results_c2', dataset='synthetic')
        xb = [torch.rand(128, 3, 32, 32, device=dev) * 2 - 1 for _ in range(2)]

        def st2(s_):
            tr2.train_step(batches=xb)
            tr2.step += 1
        ms2t = per_step(st2, 2, 5)
        others['C2_cifar10_Model_train'] = {"ms_per_step": ms2t, "images_per_sec": 256 / (ms2t / 1e3), "batch": "2 x 128",
                                            "tflops": 256 * 3 * 12.44 / ms2t}
        with torch.no_grad():
            m2.eval()
            img2 = g2.opt(xb[0])
            t2 = [50]

            def rev2(s_):
                nonlocal img2
                st = torch.full((128,), t2[0] - 1, dtype=torch.long, device=dev)
                img2 = g2._reverse_step(img2, m2(img2, st), t2[0])
                t2[0] -= 1
            ms2 = per_step(rev2, 3, 5)
        others['C2_cifar10_Model_sample'] = {"ms_per_reverse_step": ms2, "images_per_sec_50_step_sample": 128 / (ms2 * 50 / 1e3), "batch": 128}
        del m2, g2, tr2
    except Exception as e:  # context only: never let it break the headline line
        others['error_C2'] = repr(e)[:200]
    try:
        with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
            # config 5: AFHQ-128 denoising baseline, cosine T=200, ddim sampling, batch 32 (same Unet, reverse step = 1 fused kernel)
            from cold_diffusion_models_b200.denoising_diffusion_pytorch import GaussianDiffusion as DNGD
            g5 = DNGD(trainer.ema_model.denoise_fn, image_size=128, channels=3, timesteps=200, loss_type='l1', sampling_routine='ddim').to(dev)
            im5 = torch.randn(B, 3, 128, 128, device=dev)
            t5 = [200]

            def rev5(s_):
                nonlocal im5
                st = torch.full((B,), t5[0] - 1, dtype=torch.long, device=dev)
                im5 = g5._step(im5, g5.denoise_fn(im5, st), None, 0, t5[0])
                t5[0] -= 1
            ms5 = per_step(rev5, 2, 5)
            others['C5_afhq_denoise_ddim_sample'] = {"ms_per_reverse_step": ms5, "images_per_sec_200_step_sample": B / (ms5 * 200 / 1e3), "batch": B}
    except Exception as e:
        others['error_C5'] = repr(e)[:200]
    try:
        with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
            # config 4: CelebA-128 resolution diffusion (avg-pool pixelate D), x0_step_down, batch 32, same Unet.  BASELINE's
            # time_steps=200 is not constructible (RS:389-414: `Incremental*` shrinks by one pixel per step, <= 127 steps at
            # 128x128; SURVEY section 0.3), so T = 100 here
            from cold_diffusion_models_b200.resolution_diffusion_pytorch import GaussianDiffusion as RSGD
            T4 = 100
            g4 = RSGD(trainer.ema_model.denoise_fn, image_size=128, device_of_kernel='cuda', channels=3, timesteps=T4, loss_type='l1',
                      resolution_routine='Incremental_area', train_routine='Final', sampling_routine='x0_step_down').to(dev)
            im4 = g4.opt(resident[0])
            t4 = [T4]

            def rev4(s_):
                nonlocal im4
                st = torch.full((B,), t4[0] - 1, dtype=torch.long, device=dev)
                im4 = g4._reverse_step(im4, g4.denoise_fn(im4, st), t4[0])
                t4[0] -= 1
            ms4 = per_step(rev4, 2, 5)
            others['C4_celeba_resolution_sample'] = {"ms_per_reverse_step": ms4, "images_per_sec_100_step_sample": B / (ms4 * T4 / 1e3), "batch": B,
                                                     "routine": "Incremental_area, T=100 (200 steps are not constructible at 128x128)"}
    except Exception as e:
        others['error_C4'] = repr(e)[:200]
    return others


if __name__ == '__main__':
    main()
