"""Benchmark of the NeRO stage-I training hot path on B200 (BASELINE.json metric: train rays/sec at 128 samples/ray).

    python bench.py --gpus 1 --steps 20 --warmup 5                 # this repo's CUDA path
    torchrun ... bench.py --gpus N ...                             # ray-sharded data parallel, one rank per GPU
    python bench.py --impl reference ...                           # the reference algorithm (oracle port) on the host CPU

A "step" = one training step on the workload of BASELINE.json configs[1] ("bell shape stage, 1024 rays x 128 samples"):
sample_ray (64 coarse + 4x16 up-sampled + 32 background samples) + render_core forward + the YAML loss set
(charbonnier rgb + 0.1*eikonal + occlusion loss, step 30000 so the occlusion march is active) + backward + Adam step.
Three legs, all on THE SAME 1024 synthetic rays per GPU (nero_b200.synthetic.synthetic_rays, seed 6033):
  value   rays already resident in HBM, sample_ray/render_core called directly;
  e2e     through the public API `net({'step': s})`: the ray batch is fetched from the renderer's pinned host ray table
          (H2D inside the timed region), the scalar loss is read back every step (train/trainer.py:168).  The headline leg
          runs with cfg['cuda_graph'] (the step replayed from two captured graphs, nero_b200/graph.py); the eager leg and
          both variants at the reference's default train_ray_num = 512 are reported under `e2e.eager` /
          `e2e.train_ray_num_512`;
  bear    the same resident loop on BASELINE.json configs[2] (human light, 2048 rays on one GPU; 1024 per GPU under
          torchrun = configs[4] at 8 GPUs), reported under the key "bear" of the same JSON line.
--steps sets the number of timed steps of every leg above and of the reference arm.  Fixed-size samples that --steps does
not set: the cpu_baseline records (2 timed steps each on the host CPU: 256 rays of this workload, and BASELINE.json
configs[0] at steps 10000 and 30000), and the one extra step the chain roofline is profiled on.  Prints ONE JSON line on
stdout.

    python bench.py --dump-outputs DIR ...                         # also write resident-step outputs to DIR

--dump-outputs writes, after the resident leg's timed steps, what its last step computed as DIR/<name>.npy (float32, rank
0's shard): z_vals, the render_core outputs, the loss, and the gradients and updated parameters (flattened in parameter
order).  The same arrays of the first warm-up step, which starts from the seeded initial parameters, go to
DIR/first_step_<name>.npy.  The inputs are seeded, so two builds run with the same arguments can be compared output for
output.  Parameter gradients are summed with fp32 atomics, and every step before the last one feeds them to Adam, so two
runs of one build differ in the last step's parameters and outputs by that rounding compounded over warmup + steps
updates; the first step carries only one step's rounding and is the tighter comparison.
"""
import argparse
import json
import os
import resource
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, 'oracle')):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np
import torch

A_SDF, A_SHADE, A_SHADE_H, A_NERF = 524544, 1211648, 1349888, 604160   # MAC / sample (SURVEY.md section 8d)
STEP = 30000
RAYS_PER_GPU = 1024
METRIC = 'train rays/sec (128 samples/ray)'
DUMP_BYTES = 64 << 20       # --dump-outputs budget (about 38 MB are written at the default workload)


def workload_config(bear, R, world):
    """The static description of the workload: identical for the CUDA arm and the reference arm of the same launch."""
    name = (f'bear_human_light_shape_stage_{R}rays_x_(64+64)samples_+32bg_step30000_occ_on' if bear else
            f'bell_shape_stage_{R}rays_x_(64+64)samples_+32bg_step30000_occ_on')
    return {'workload': name, 'rays_per_gpu': R, 'global_rays': R * world,
            'parallelism': f'ray-sharded dp{world}, one NCCL all-reduce of the flat grad buffer' if world > 1 else 'single gpu',
            'l2': 'per-step working set ~6 GB of activations >> 126 MB L2 (inputs larger than L2)',
            'optimizer': 'Adam inside the timed region'}


def rays_per_gpu(bear, world):
    # weak scaling: fixed rays per GPU.  bear: 2048 rays on one GPU (configs[2]); under torchrun 1024 per GPU, i.e. 8192 rays
    # on 8 GPUs (configs[4])
    return (2048 if world == 1 else 1024) if bear else RAYS_PER_GPU


def algorithmic_flops(R, n_in, n_out, p_occ, human=False):
    """F = 2*[R*112*A_sdf + N_in*(6*A_sdf + 3*A_shade) + N_out*3*A_nerf + P_occ*80*A_sdf]   (SURVEY.md 8d)"""
    a_sh = A_SHADE_H if human else A_SHADE
    return 2.0 * (R * 112 * A_SDF + n_in * (6 * A_SDF + 3 * a_sh) + n_out * 3 * A_NERF + p_occ * 80 * A_SDF)


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        d = json.load(open(path))
        return d.get('bf16_tflops_sustained', 1386.8), d.get('hbm_gbs', 6569.6), 'measured'
    return 1400.0, 6650.0, 'fallback'


class ClockSampler(threading.Thread):
    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons = index, False, [], set()
        self.max_mhz = None

    def run(self):
        q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        while not self.stop_flag:
            try:
                o = subprocess.run(['nvidia-smi', f'--id={self.index}', f'--query-gpu={q}', '--format=csv,noheader,nounits'],
                                   capture_output=True, text=True, timeout=5).stdout.strip().split(',')
                self.samples.append(float(o[0]))
                self.max_mhz = float(o[1])
                for n, v in zip(names, o[2:]):
                    if 'Active' in v and 'Not' not in v:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.1)

    def result(self):
        return {'sm_mhz': float(np.median(self.samples)) if self.samples else None, 'sm_max_mhz': self.max_mhz,
                'reasons': sorted(self.reasons)}


def build_net(cfg, device):
    from nero_b200 import params as P, synthetic
    from nero_b200.renderer import NeROShapeRenderer
    sd = synthetic.perturb_params(P.build_shape_state_dict(cfg, seed=6033))
    net = NeROShapeRenderer(cfg, training=False)
    net.load_state_dict(sd)
    return net.to(device), sd


def synthetic_dataset(net, rays, n_batches):
    """Fills the renderer's pinned host ray table (what _init_dataset builds from a database) with `n_batches` copies of
    the benchmark's ray set, one "image" (pose) per ray.  Poses are orthonormal look-at frames at the ray origins and the
    camera-space directions are R d, so the world-space ray that train_step reconstructs (network/renderer.py:258-272:
    origin -R^T t, direction normalize(R^T dirs)) is the synthetic ray (to fp32 rounding): the e2e leg renders the rays of
    the resident leg while going through the table fetch + H2D copy every step."""
    o, d = rays['rays_o'].double(), rays['rays_d'].double()
    zc = torch.nn.functional.normalize(-o, dim=-1)
    up = torch.tensor([0.0, 0.0, 1.0], dtype=torch.float64).expand_as(zc)
    xc = torch.nn.functional.normalize(torch.cross(up, zc, dim=-1), dim=-1)
    yc = torch.cross(zc, xc, dim=-1)
    Rm = torch.stack([xc, yc, zc], 1)                                         # [R,3,3], rows = camera axes
    poses = torch.cat([Rm, -(Rm @ o[:, :, None])], -1).float()
    dirs_cam = (Rm @ d[:, :, None])[:, :, 0].float()
    R = dirs_cam.shape[0]
    rep = lambda x: x.repeat(n_batches, *([1] * (x.dim() - 1)))
    net.train_batch = {'dirs': rep(dirs_cam).pin_memory(), 'rgbs': rep(rays['rgb']).pin_memory(),
                       'idxs': rep(torch.arange(R, dtype=torch.int64)[:, None]).pin_memory()}
    net.train_poses = poses.pin_memory()
    net.tbn = R * n_batches
    net.train_batch_i = 0
    net._shuffle_train_batch = lambda: setattr(net, 'train_batch_i', 0)     # keep the table as laid out (no host reshuffle)
    return R * (12 + 12 + 8 + 48)                                 # H2D bytes per step: dirs + rgbs + idxs rows + the pose table


def training_loss(net, out, rgb_gt, eik_weight=1.0):
    loss = torch.mean(net.compute_rgb_loss(out['ray_rgb'], rgb_gt)) + eik_weight * torch.mean(out['gradient_error'] * 0.1)
    if 'loss_occ' in out:
        loss = loss + torch.mean(out['loss_occ'])
    return loss


class Workload:
    """One renderer + optimizer + resident ray shard; `step()` = a full training step."""

    def __init__(self, bear, rank, world, dev):
        from nero_b200 import synthetic, dp
        from nero_b200.optim import FlatAdam
        self.bear, self.rank, self.world, self.dev, self.dp = bear, rank, world, dev, dp
        cfg = {'shader_config': {'human_light': True}} if bear else {}
        self.net, _ = build_net(cfg, dev)
        self.R = R = rays_per_gpu(bear, world)
        rays = synthetic.synthetic_rays(R * world, seed=6033)
        self.host_rays = {k: v[rank * R:(rank + 1) * R].contiguous() for k, v in rays.items()}
        self.r = {k: v.to(dev).contiguous() for k, v in self.host_rays.items()}
        self.opt = FlatAdam(self.net, lr=5e-4 * 0.05)      # one nero_adam_flat launch over the flat parameter / gradient buffers
        self.car = self.net.get_anneal_val(STEP)
        self.gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        self.params = list(self.net.parameters())

    def sync_grads(self):
        if self.world > 1:          # ONE NCCL all-reduce over the flat fp32 gradient buffer per step
            self.dp.sync_gradients(self.net.engine.grads.flat, self.world, params=self.params)

    def eik_weight(self):
        # gradient_error is a mean over the data-dependent number of inner samples: W*N_in/sum(N_in) makes the average of
        # the per-rank means equal the mean over all samples of the global batch (one scalar all-reduce, no host sync)
        if self.world == 1:
            return 1.0
        e = self.net.engine
        n = e.state['N_in'] if e.state['N_in'] is not None else e.w['n_in']      # graph mode keeps the count on the device
        return self.dp.global_mean_weight(n, self.world)

    def resident_step(self, keep=False):
        net, r, R = self.net, self.r, self.R
        self.opt.zero_grad(set_to_none=True)
        ri = torch.rand([R, 1], device=self.dev, generator=self.gen)
        rb = torch.rand([R, 32], device=self.dev, generator=self.gen)
        z = net.sample_ray(r['rays_o'], r['rays_d'], r['near'], r['far'], 1.0, ri, rb)
        out = net.render_core(r['rays_o'], r['rays_d'], z, r['human_poses'], self.car, STEP)
        loss = training_loss(net, out, r['rgb'], self.eik_weight())
        loss.backward()
        self.sync_grads()
        self.opt.step()
        if keep:        # for step_arrays (--dump-outputs)
            self.last = {'z_vals': z, **out, 'loss': loss}
        return loss

    def e2e_step(self, step):
        self.opt.zero_grad(set_to_none=True)
        out = self.net({'step': step})
        loss = out['loss_rgb'].mean() + self.eik_weight() * torch.mean(out['gradient_error'] * 0.1) + torch.mean(out['loss_occ'])
        loss.backward()
        self.sync_grads()
        self.opt.step()
        return float(loss.detach().cpu())          # the trainer's per-step host read (train/trainer.py:168)

    def counts(self):
        st = self.net.engine.state
        return st['N_in'], int(self.net.engine.w['n_out'].item()), st['P']


def step_arrays(wl):
    """Host float32 copies of what `wl.resident_step(keep=True)` computed: its outputs, gradients and updated parameters."""
    arrays = {k: v.detach() for k, v in wl.last.items()}
    arrays['grads'] = torch.cat([p.grad.reshape(-1) for p in wl.params])
    arrays['params'] = torch.cat([p.detach().reshape(-1) for p in wl.params])
    return {k: v.float().cpu().numpy() for k, v in arrays.items()}


def dump_outputs(out_dir, last, first):
    """Writes step_arrays of the last timed step as <name>.npy and of the first warm-up step as first_step_<name>.npy."""
    arrays = {**last, **{'first_step_' + k: v for k, v in first.items()}}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_BYTES, f'--dump-outputs: {total} bytes exceed the {DUMP_BYTES}-byte budget'
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


def timed(fn, steps, barrier):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(steps):
        fn(i)
    ev1.record()
    barrier()
    return ev0.elapsed_time(ev1) / steps


def run_ours(args):
    import torch.distributed as dist
    from nero_b200 import ops
    rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
    assert args.gpus == world, f'--gpus {args.gpus} but WORLD_SIZE={world}: launch N ranks with torch.distributed.run (one per GPU)'
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        # NCCL prints its version banner to stdout when the communicator is created: keep stdout for the ONE JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group('nccl', device_id=dev)
            dist.all_reduce(torch.zeros(1, device=dev))
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(vals):
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    bear = args.workload == 'bear'
    wl = Workload(bear, rank, world, dev)
    R = wl.R
    dump = bool(args.dump_outputs) and rank == 0
    for i in range(args.warmup):
        wl.resident_step(keep=dump and i == 0)
        if dump and i == 0:
            first = step_arrays(wl)
    barrier()
    sampler = ClockSampler(local)      # clocks / throttle reasons of rank 0's GPU only (one nvidia-smi poller per job, not per rank)
    if rank == 0:
        sampler.start()
    l0 = ops.launch_count
    ms = timed(lambda i: wl.resident_step(keep=dump and i == args.steps - 1), args.steps, barrier)
    launches = (ops.launch_count - l0) // args.steps
    n_in, n_out, p_occ = wl.counts()
    if dump:
        dump_outputs(args.dump_outputs, step_arrays(wl), first)

    # ---- end to end through the public API with host buffers (H2D of the ray batch + D2H of the loss every step):
    # the headline leg replays the step from CUDA graphs (cfg['cuda_graph']); the eager leg and the reference's default
    # train_ray_num = 512 (where the step is launch-bound without graphs) are reported beside it
    n_e2e_warm = max(3, args.warmup // 2)

    def e2e_leg(rays_n, graphed):
        wl.net.cfg['train_ray_num'] = rays_n
        wl.net.cfg['cuda_graph'] = graphed
        h2d = synthetic_dataset(wl.net, {k: v[:rays_n].contiguous() for k, v in wl.host_rays.items()}, n_batches=args.steps + n_e2e_warm + 2)
        for _ in range(n_e2e_warm):
            wl.e2e_step(STEP)
        ms_leg = timed(lambda i: wl.e2e_step(STEP), args.steps, barrier)
        return ms_leg, h2d, int(wl.net.engine.w['n_in'].item())
    ms_e2e_eager, h2d, _ = e2e_leg(R, False)
    ms_e2e, h2d, n_in_e2e = e2e_leg(R, True)
    r_small = min(512, R)
    ms_small_eager, h2d_small, _ = e2e_leg(r_small, False)
    ms_small, _, n_in_small = e2e_leg(r_small, True)
    sampler.stop_flag = True
    if rank == 0:
        sampler.join(timeout=2)
    spread = wl.dp.param_checksum_spread(wl.params, world)
    assert spread == 0.0, f'parameter replicas diverged across ranks (checksum spread {spread})'

    # ---- roofline of the dominant kernel: per-launch CUDA events on the launch stream
    prof = profile_chains(wl) if rank == 0 else None

    # ---- the second workload (configs[2] / configs[4]) under the key "bear"
    other = None
    if not bear and not args.no_bear:
        wb = Workload(True, rank, world, dev)
        for _ in range(3):
            wb.resident_step()
        ms_b = timed(lambda i: wb.resident_step(), args.steps, barrier)
        nb_in, nb_out, pb = wb.counts()
        ms_b, = reduce_max([ms_b])
        other = {'metric': METRIC, 'value': wb.R * world / (ms_b * 1e-3), 'unit': 'rays/s', 'ms_per_step': ms_b, 'steps': args.steps, 'warmup': 3,
                 'config': workload_config(True, wb.R, world), 'counts': {'n_in': nb_in, 'n_out': nb_out, 'p_occ': pb},
                 'step_tensor_tflops': algorithmic_flops(wb.R, nb_in, nb_out, pb, True) / (ms_b * 1e-3) / 1e12}
        del wb
    ms, ms_e2e, ms_e2e_eager, ms_small, ms_small_eager = reduce_max([ms, ms_e2e, ms_e2e_eager, ms_small, ms_small_eager])
    if rank == 0:
        peak_tf, peak_bw, which = measured_peaks()
        F = algorithmic_flops(R, n_in, n_out, p_occ, human=bear)
        line = {
            'metric': METRIC, 'value': R * world / (ms * 1e-3), 'unit': 'rays/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32 (split-bf16 x3 tensor-core MMAs, fp32 accumulate)', 'data': 'synthetic',
            'config': workload_config(bear, R, world),
            'counts': {'n_in': n_in, 'n_out': n_out, 'p_occ': p_occ},
            'e2e': {'value': R * world / (ms_e2e * 1e-3), 'unit': 'rays/s', 'ms_per_step': ms_e2e, 'h2d_bytes_per_step': h2d,
                    'd2h_bytes_per_step': 4, 'n_in': n_in_e2e, 'cuda_graph': True,
                    'eager': {'value': R * world / (ms_e2e_eager * 1e-3), 'ms_per_step': ms_e2e_eager},
                    'train_ray_num_512': {'rays_per_gpu': r_small, 'value': r_small * world / (ms_small * 1e-3), 'ms_per_step': ms_small,
                                          'h2d_bytes_per_step': h2d_small, 'n_in': n_in_small,
                                          'eager': {'value': r_small * world / (ms_small_eager * 1e-3), 'ms_per_step': ms_small_eager}},
                    'note': 'same rays as `value`, fetched from the pinned host ray table through net({"step"}) + loss read-back; '
                            'cfg cuda_graph replays the step from two captured graphs (no host sync inside the step)'},
            'gpu_launches': int(launches),
            'clocks': sampler.result(),
            'step_tensor_tflops': F / (ms * 1e-3) / 1e12,
            'step_tensor_frac_of_bf16_peak': F / (ms * 1e-3) / 1e12 / peak_tf,
            'roofline': None, 'cpu_baseline': None,
        }
        if prof is not None and prof['reverse_sweep'] is not None:
            one = prof['reverse_sweep']
            ach_tf = one['flops'] / one['seconds'] / 1e12
            # algorithmic HBM bytes of the launch: the first operand in + 8 layers x (saved activation in + product out), 1 KB per
            # row and tensor (DESIGN.md section 4); the decoupling experiments of profiles/r02j show the kernel nearer to this roof
            # (epilogue + operand traffic alone: 82 % of the coupled time) than to the tensor roof (MMAs alone: 49 %)
            alg_bytes = one['rows'] * 17408.0
            ach_bw = alg_bytes / one['seconds'] / 1e9
            traffic, tsrc = None, None
            tp = os.path.join(ROOT, 'profiles', 'chain_traffic.json')
            if os.path.exists(tp):      # ncu dram__bytes_read+write of this launch, recorded per row; scaled to this run's rows
                tj = json.load(open(tp))
                traffic, tsrc = tj['dram_bytes_per_row'] * one['rows'], tj.get('source')
            line['roofline'] = {'bound': 'hbm', 'kernel': 'umma_chain_kernel: SDF reverse-sweep chain (8 fused 256-wide layers, one launch)',
                                'achieved': ach_bw, 'peak': peak_bw, 'unit': 'GB/s', 'frac': ach_bw / peak_bw,
                                'peak_source': which + ' HBM copy bandwidth', 'algorithmic_bytes': alg_bytes,
                                'launch_us': one['seconds'] * 1e6, 'rows': one['rows'], 'traffic': traffic, 'traffic_source': tsrc,
                                'traffic_frac_of_peak': None if traffic is None else traffic / one['seconds'] / 1e9 / peak_bw,
                                'tensor': {'achieved': ach_tf, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': ach_tf / peak_tf,
                                           'frac_of_split3_ceiling': ach_tf / (peak_tf / 3.0), 'peak_source': which + ' bf16 sustained',
                                           'note': 'ALGORITHMIC fp32 GEMM flops (2*M*K*N of the un-padded layers); the split-bf16 scheme '
                                                   'issues 3 bf16 MMAs per product, so 1/3 of peak is its ceiling'},
                                'all_chain_launches': {'launches': prof['launches'], 'total_ms': prof['seconds'] * 1e3,
                                                       'tensor_achieved': prof['flops'] / prof['seconds'] / 1e12,
                                                       'tensor_frac': prof['flops'] / prof['seconds'] / 1e12 / peak_tf}}
        if other is not None:
            line['bear'] = other
        if not args.no_cpu and world == 1:      # the CPU leg runs on rank 0 at N=1 only
            line['cpu_baseline'] = cpu_baseline_default()
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def profile_chains(wl):
    """One extra training step with a CUDA-event pair (on the launch stream) around every fused MLP-chain launch
    (ops.PROFILE hook).  Returns the aggregate over all chain launches and the SDF reverse-sweep chain alone (the
    launch whose ncu capture is committed under profiles/)."""
    from nero_b200 import ops
    net, r = wl.net, wl.r
    ops.PROFILE = []
    try:
        net.zero_grad()
        z = net.sample_ray(r['rays_o'], r['rays_d'], r['near'], r['far'], 0)
        out = net.render_core(r['rays_o'], r['rays_d'], z, r['human_poses'], wl.car, STEP)
        training_loss(net, out, r['rgb']).backward()
        torch.cuda.synchronize()
        recs = ops.PROFILE
    finally:
        ops.PROFILE = None
    w = net.engine.w
    counts = {w['n_in'].data_ptr(): net.engine.state['N_in'], w['n_out'].data_ptr(): int(w['n_out'].item())}
    tot_f = tot_s = 0.0
    one = None
    for tag, e0, e1, fl_row, mp, m_cap in recs:
        M = m_cap if mp is None else counts.get(mp, m_cap)
        sec = e0.elapsed_time(e1) * 1e-3
        tot_f += fl_row * M
        tot_s += sec
        if tag == 'sdf_reverse_sweep':
            one = {'flops': fl_row * M, 'seconds': sec, 'rows': M}
    return {'flops': tot_f, 'seconds': tot_s, 'launches': len(recs), 'reverse_sweep': one}


def cpu_baseline(rays_n=128, steps=1, threads=None, cfg=None, step=STEP):
    """The reference algorithm (oracle port, bit-exact to the reference on CPU) timed on the host cores: one training
    step (sample_ray + render_core + loss + backward) on a bounded sample of the same workload."""
    import nero_oracle as O
    from nero_b200 import params as P
    cfg = dict(cfg or {})
    sd = O.perturb_params(P.build_shape_state_dict(cfg, seed=6033))
    rays = O.synthetic_rays(rays_n, seed=6033)
    c = O.merged_cfg(cfg)
    lut = sd['color_network.FG_LUT'][0]
    car = O.get_anneal_val(c, step)

    def one(rr, n):
        p = {k: v.clone().requires_grad_(torch.is_floating_point(v) and not k.endswith('FG_LUT')) for k, v in sd.items()}
        g = torch.Generator().manual_seed(0)
        ri, rb = torch.rand([n, 1], generator=g), torch.rand([n, c['n_bg_samples']], generator=g)
        out = O.render(p, cfg, lut, rr['rays_o'], rr['rays_d'], rr['near'], rr['far'], rr['human_poses'], car, step,
                       rand_inner=ri, rand_bg=rb)
        O.training_loss(out, rr['rgb'], c, step).backward()
    # "all the host threads it can use": torch's intra-op pool is slower when oversubscribed on these small ops, so
    # pick the best of a few pool sizes on a short calibration slice and report the count actually used
    ncpu = os.cpu_count() or 1
    cands = [threads] if threads else sorted({c_ for c_ in (8, 16, 32, 64, ncpu) if c_ <= ncpu})
    if len(cands) > 1:
        n_cal = max(16, min(64, rays_n // 8))
        cal = {k: v[:n_cal] for k, v in rays.items()}
        best = None
        for c_ in cands:
            torch.set_num_threads(c_)
            one(cal, n_cal)
            t0 = time.time()
            one(cal, n_cal)
            dt_c = time.time() - t0
            if best is None or dt_c < best[0]:
                best = (dt_c, c_)
        cores = best[1]
    else:
        cores = cands[0]
    torch.set_num_threads(cores)
    one(rays, rays_n)   # warm-up
    t0 = time.time()
    for _ in range(steps):
        one(rays, rays_n)
    dt = (time.time() - t0) / steps
    model = ''
    try:
        model = [l.split(':')[1].strip() for l in open('/proc/cpuinfo') if l.startswith('model name')][0]
    except Exception:
        pass
    n, ni, nb = c['n_samples'], c['n_importance'], c['n_bg_samples']
    return {'value': rays_n / dt, 'unit': 'rays/s', 'cores': cores, 'host_cores': ncpu, 'kind': 'port', 'seconds_per_step': dt, 'cpu': model,
            'peak_rss_gb': resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1e6,
            'sample': f'{rays_n} rays x ({n}+{ni})+{nb}bg samples, step {step}' + (' (occlusion march on)' if step >= c['occ_loss_step'] else '') +
                      f', fwd+bwd, {steps} timed step(s) after 1 warm-up'}


def cpu_baseline_default():
    """The CPU leg of the default run (~20-30 s of CPU work): a 256-ray sample of the headline workload (same sampling
    depth: (64+64)+32, step 30000), plus BASELINE.json configs[0] as the reference's own CPU-runnable case: 256 rays x
    (32+32)+32 at steps 10000 and 30000 (BASELINE.md section 3)."""
    cb = cpu_baseline(rays_n=256, steps=2)
    threads = cb['cores']
    c0 = {'n_samples': 32, 'n_importance': 32}
    cb['config0_256rays_x_(32+32)+32'] = {f'step{s}': {k: v for k, v in cpu_baseline(256, 2, threads, c0, s).items()
                                                        if k in ('value', 'seconds_per_step', 'sample')} for s in (10000, 30000)}
    return cb


def run_reference(args):
    """The reference arm: the reference's algorithm (bit-exact CPU port) on all host cores, on the headline configuration
    itself -- every step is the full 1024-ray x (64+64)+32 batch of configs[1] (about 10 s per step on 8 cores); --steps
    sets the number of timed steps (--steps 2 for a short run)."""
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if rank != 0:
        return
    bear = args.workload == 'bear'
    R = rays_per_gpu(bear, world)
    cfg = {'shader_config': {'human_light': True}} if bear else {}
    t0 = time.time()
    steps = args.steps
    cb = cpu_baseline(rays_n=R, steps=steps, cfg=cfg)
    c0 = {'n_samples': 32, 'n_importance': 32}
    extra = {f'step{s}': {k: v for k, v in cpu_baseline(256, 2, cb['cores'], c0, s).items() if k in ('value', 'seconds_per_step', 'sample')}
             for s in (10000, 30000)}
    line = {'metric': METRIC, 'value': cb['value'], 'unit': 'rays/s', 'n_gpus': args.gpus,
            'steps': steps, 'warmup': 1, 'ms_per_step': cb['seconds_per_step'] * 1e3, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'impl': 'reference',
            'config': workload_config(bear, R, world),
            'note': 'the reference is a pure-PyTorch script repository that cannot be installed or shipped to the GPU box; this is its '
                    'bit-exact CPU port (oracle/nero_oracle.py, pinned by tests/golden) on the host cores, one rank, timing the '
                    f'full per-GPU batch of the workload ({R} rays) per step; {steps} timed steps (about 10 s each)',
            'config0_256rays_x_(32+32)+32': extra, 'wall_s': time.time() - t0,
            'cpu_baseline': cb,
            'e2e': {'value': cb['value'], 'unit': 'rays/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours')
    ap.add_argument('--workload', default='bell', choices=['bell', 'bear'],
                    help="bell = BASELINE.json configs[1] (the headline, default); bear = configs[2]: human light, 2048 rays")
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg (profiling runs)')
    ap.add_argument('--no-bear', action='store_true', help='skip the second workload (configs[2]) record')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the outputs of the last timed resident step to DIR/<name>.npy and of the first warm-up step to '
                         'DIR/first_step_<name>.npy (float32)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(args.warmup, 3)
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
