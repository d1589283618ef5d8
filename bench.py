"""bench.py -- LatentAugment hot path throughput: augmented images / second.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config c2|c3|c5|c1] [--precision bf16]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path over one batch: ``num_steps`` Adam iterations on w through the
generator (forward + backward-to-w) plus the final synthesis -- one ``LatentAugment.forward()``.

Workloads (BASELINE.json configs):
  c2 (default; the configuration the metric is quoted on): SG2 256x256 3-ch, batch 32 per GPU, 10 steps, 4096-code
     bank; N GPUs = N batches (weak scaling, no data-path collective: samples are independent, SURVEY.md §8e).
  c3: SG2 512x512 3-ch, batch 128 SPLIT over the N ranks (strong scaling), 10 steps, CUDA-graph-captured loop.
  c5: nearest-code sweep, 2^20 real codes sharded over the N ranks x 1024 queries, fused GEMM + top-k, exact
     re-rank, NCCL all-gather + merge inside the timed region (the one collective of the design).
  c1: SG2 128x128 1-ch, batch 4, 5 steps (the reference's CPU-runnable case; a parity-test case, not a bench line).
One JSON line on stdout (rank 0).  The default run (c2, bf16) also carries the other two GPU configurations as sub-objects,
measured after the headline legs in the same launch at the same N: ``c5_sharded_search`` (2^17 codes per GPU -- at N = 8
the 2^20-code sweep of BASELINE.json -- with the all-gather + merge in the timed region and the merged result checked against
the gathered per-rank lists), ``c3_strong_split`` (batch 128 split over the N ranks) and, at N = 1, ``four_terms_author_weights``
(all four criteria at the author's weights).  ``--no-extras`` skips them; a
watchdog (``--extras-timeout``) prints the line without them if a leg wedges, and ``destroy_process_group`` runs under its
own (tests/test_bench_flow.py exercises all of this on CPU with stand-ins for the CUDA-facing pieces).

``--dump-outputs DIR`` writes what the last timed step of the headline leg returned (``img``, ``w_aug``) as
``DIR/<name>.npy`` in float32, so that two builds can be compared output for output: every input, and the random noise of
the final synthesis, comes from fixed seeds, so the same arguments give the same inputs in every run.
"""
import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {          # BASELINE.json configs; oracle/synthetic.py holds the same table for the parity tests
    'c1': dict(img_resolution=128, img_channels=1, batch=4, steps=5, bank=256, img_bank=64),
    'c2': dict(img_resolution=256, img_channels=3, batch=32, steps=10, bank=4096, img_bank=64),
    'c3': dict(img_resolution=512, img_channels=3, batch=128, steps=10, bank=4096, img_bank=64, strong=True),
    'tiny': dict(img_resolution=32, img_channels=2, batch=4, steps=3, bank=64, img_bank=8, channel_base=2048, channel_max=64),
}
C5 = dict(codes=1 << 20, queries=1024, dim=512, k=4)
DUMP_LIMIT = 64 << 20        # bytes that --dump-outputs writes at most


def layer_table(res, img_c, channel_base=32768, channel_max=512):
    """(name, res_out, cin, cout, up) of every conv layer + algorithmic / executed MACs per image."""
    from latentaugment_b200.utils.synthetic import channels_for
    ch = channels_for(res, channel_base, channel_max)
    rows = []
    for r, c in ch.items():
        if r > 4:
            rows.append((f'b{r}.conv0', r, ch[r // 2], c, 2))
        rows.append((f'b{r}.conv1', r, c, c, 1))
    out = []
    for name, r, cin, cout, up in rows:
        if up == 2:      # algorithmic: transposed conv on the input grid + 4x4 FIR; the GEMM executes the 9 taps, the FIR is a SIMT pass
            alg = 9 * (r // 2) ** 2 * cin * cout + 16 * r * r * cout
            exe = 9 * (r // 2) ** 2 * cin * cout
        else:
            alg = exe = 9 * r * r * cin * cout
        out.append(dict(name=name, res=r, cin=cin, cout=cout, up=up, alg_macs=alg, exe_macs=exe))
    rgb = sum(r * r * c * img_c for r, c in ch.items())
    return out, rgb


def f_syn(res, img_c, **kw):
    """Forward FLOPs of one synthesis pass per image (SURVEY.md §8d definition)."""
    rows, rgb = layer_table(res, img_c, **kw)
    return 2.0 * (sum(r['alg_macs'] for r in rows) + rgb)


class ClockSampler:
    """nvidia-smi SM clock + throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.proc = None
        q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={index}', f'--query-gpu={q}', '--format=csv,noheader,nounits',
                                          '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(',')]
            try:
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for n, v in zip(names, f[2:6]):
                    if v.lower().startswith('active'):
                        self.reasons.add(n)
            except (ValueError, IndexError):
                pass

    def mark(self):
        return len(self.samples)

    def stop(self, start=0):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        s = sorted(self.samples[start:]) or sorted(self.samples)
        med = s[len(s) // 2] if s else None
        return {'sm_mhz': med, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons)}


class LineEmitter:
    """Rank 0 prints exactly ONE JSON line.  A watchdog may print it early -- with what is known by then -- and end the
    process: a leg that hangs (a wedged collective, a teardown that never returns) must not lose the measured numbers."""

    def __init__(self, rank, stream):
        self.rank, self.stream, self.lock, self.done, self.line = rank, stream, threading.Lock(), False, None

    def set(self, line):
        with self.lock:
            self.line = line

    def update(self, extra):
        with self.lock:
            if self.line is not None and not self.done:
                self.line.update(extra)

    def emit(self):
        with self.lock:
            if self.done:
                return
            self.done = True
            if self.rank == 0 and self.line is not None:
                print(json.dumps(self.line), file=self.stream, flush=True)


def start_watchdog(seconds, emitter, what):
    """After ``seconds``: print the line as it stands (plus a note) and leave with exit code 0."""
    def fire():
        emitter.update({'watchdog': f'{what} did not finish within {seconds:.0f} s; the line was printed without it and the process ended'})
        emitter.emit()
        sys.stderr.write(f'bench.py: watchdog: {what} exceeded {seconds:.0f} s\n')
        sys.stderr.flush()
        os._exit(0)
    t = threading.Timer(seconds, fire)
    t.daemon = True
    t.start()
    return t


def cuda_device(index):
    import torch
    return torch.device(f'cuda:{index}')


def teardown_group(world, limit=30.0):
    """destroy_process_group under a watchdog (one 8-GPU run of this round hung right here, DESIGN.md §8)."""
    if world <= 1:
        return
    import torch.distributed as dist
    t = threading.Timer(limit, lambda: os._exit(0))
    t.daemon = True
    t.start()
    try:
        dist.destroy_process_group()
    finally:
        t.cancel()


def make_plugin(c, B, local_rank, precision, weights, micro_batches=1):
    """The reference-facing plugin in synthetic mode (random-init generator, synthetic banks)."""
    from latentaugment_b200.augments import create_augment
    from latentaugment_b200.options.aug_options import AugOptions
    w_lat, w_pix, w_lpips, w_disc = weights
    argv = ['--aug', 'latent', '--synthetic', '--batch_size', str(B), '--gpu_ids', str(local_rank), '--gpu_ids_aug', str(local_rank),
            '--img_resolution', str(c['img_resolution']), '--synthetic_channels', str(c['img_channels']), '--synthetic_bank', str(c['bank']),
            '--synthetic_img_bank', str(c['img_bank']), '--synthetic_codes', str(max(4 * B, 256)), '--precision', precision,
            '--opt_num_epochs', str(c['steps']), '--no_log',
            '--synthetic_channel_base', str(c['channel_base']), '--synthetic_channel_max', str(c['channel_max']),
            '--micro_batches', str(micro_batches)]
    opt = AugOptions().parse(args={'p_thres': 0.0, 'w_lpips': w_lpips, 'w_disc': w_disc, 'w_pix': w_pix, 'w_latent': w_lat,
                                   'init_w': 'inv', 'n_imgs': 0}, argv=argv)
    return create_augment(opt)


class PluginTimer:
    """The two timed legs of a plugin workload: device-resident (``core.forward`` on codes already in HBM, CUDA events,
    max over ranks) and end to end (``set_input / forward / get_output`` with host dicts, wall clock around a final
    synchronize, max over ranks)."""

    def __init__(self, aug, B, res, rank, world, dev):
        self.aug, self.B, self.res, self.rank, self.world, self.dev = aug, B, res, rank, world, dev
        self.core = aug.latent_aug.module
        self.names = list(aug.stats_dataset_w.index.keys())

    def batch_data(self, i):
        import torch
        B, res, names = self.B, self.res, self.names
        fn = [names[((self.rank * 131 + i) * B + j) % len(names)] for j in range(B)]
        img = torch.zeros([B, 1, res, res])
        return {'A': img, 'B': img, 'A_paths': fn, 'B_paths': fn}

    def barrier(self):
        import torch
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, x):
        import torch
        if self.world == 1:
            return x
        import torch.distributed as dist
        t = torch.tensor([x], device=self.dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def resident(self, warmup, steps, clocks=None):
        """-> (ms per step as the max over ranks, launches of this rank, the device-resident code batches); ``self.mark`` =
        the clock sampler's position when the timed region starts, ``self.last`` = what the last timed step returned"""
        import torch
        aug, core = self.aug, self.core
        w_dev = [aug.sample_from_inversion(self.batch_data(i)['A_paths']).to(self.dev) for i in range(warmup + steps)]
        for i in range(warmup):
            core.forward(w_dev[i])
        self.barrier()
        self.mark = clocks.mark() if clocks is not None else 0
        l0 = sum(e.launch_count for e in core.engines)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(steps):
            self.last = core.forward(w_dev[warmup + i])
        ev1.record()
        self.barrier()
        launches = sum(e.launch_count for e in core.engines) - l0
        ms = self.max_over_ranks(ev0.elapsed_time(ev1)) / steps
        return ms, launches, w_dev

    def end_to_end(self, steps):
        """-> (seconds per step as the max over ranks, the last output dict)"""
        import torch
        aug = self.aug
        for i in range(3):
            aug.set_input(self.batch_data(i)); aug.forward(); aug.get_output()
        self.barrier()
        t0 = time.perf_counter()
        out = None
        for i in range(steps):
            aug.set_input(self.batch_data(i))
            aug.forward()
            out = aug.get_output()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        return self.max_over_ranks(t1 - t0) / steps, out


def dump_outputs(path, arrays, limit=DUMP_LIMIT):
    """Writes each tensor of ``arrays`` as ``path/<name>.npy`` in float32.  When they exceed ``limit`` bytes in all, each
    keeps the same fixed, seeded subset of its leading-dimension rows (in ascending order), sized to fit."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    total = sum(4 * t.numel() for t in arrays.values())
    for name, t in arrays.items():
        t = t.detach().float()
        if total > limit:
            n = t.shape[0]
            rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:max(1, n * limit // total)].sort().values
            t = t[rows.to(t.device)]
        np.save(os.path.join(path, f'{name}.npy'), t.cpu().numpy())


def _full_cfg(cfg_name):
    c = dict(CONFIGS[cfg_name])
    c.setdefault('channel_base', 32768)
    c.setdefault('channel_max', 512)
    return c


def cpu_baseline(cfg_name, sample_batch=4):
    """The reference's CPU path on the box's host cores, on a BOUNDED sample of the workload.

    kind "reference": the reference's own ``LatentAug.forward`` (augments/utils/util_latent_aug.py:207-310) from the
    shipped copy ``baseline/_ref``, over the reference's ``torch_utils.ops`` ref implementations (oracle/ref_driver.py);
    kind "port": the oracle restatement, when no reference copy is present.  Sample: ``sample_batch`` images, once
    with 1 and once with 3 Adam steps; per-step and fixed (final synthesis) costs follow from the two timings and are
    extrapolated to the config's step count and reported per image."""
    import random

    import torch
    c = _full_cfg(cfg_name)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    bs = min(sample_batch, c['batch'])
    times = {}
    kind = 'reference'
    try:
        from oracle import ref_driver
        ref = ref_driver.import_reference()
        runs = {s: ref_driver.reference_loop(c, batch=bs, steps=s, device='cpu', ref=ref)[0] for s in (1, 3)}
        what = "reference LatentAug.forward from baseline/_ref over the reference's torch_utils.ops (CPU ref paths)"
    except FileNotFoundError:
        from oracle import latent_aug as ola
        from oracle import synthetic
        kind = 'port'
        wl = synthetic.make_workload(c, noise_strength=0.0, batch=bs)
        orcs = {s: ola.LatentAugOracle(wl['G'], wl['W'], wl['X'], num_epochs=s, fused=True) for s in (1, 3)}
        runs = {s: (lambda o=o: o.forward(wl['w0'].clone())) for s, o in orcs.items()}
        what = 'oracle port (torch CPU, fused modconv); no reference copy under baseline/_ref'
    random.seed(0)
    runs[1]()                             # untimed warm-up (thread pool, primitive caches)
    for s in (1, 3):
        random.seed(0)
        t0 = time.perf_counter()
        runs[s]()
        times[s] = time.perf_counter() - t0
    per_step = (times[3] - times[1]) / 2.0
    fixed = max(times[1] - per_step, 0.0)
    t_full = fixed + per_step * c['steps']
    ips = bs / t_full
    return {'value': ips, 'unit': 'img/s', 'cores': torch.get_num_threads(), 'kind': kind,
            'sample': f'{what}; batch {bs}: 1 Adam step + final synthesis {times[1]:.2f} s, 3 steps {times[3]:.2f} s '
                      f'-> {per_step:.2f} s/step + {fixed:.2f} s, extrapolated to {c["steps"]} steps = {t_full:.1f} s per {bs} images'}


def run_reference(args):
    """``--impl reference``: the reference's CPU implementation of the path on the host cores (rank 0 only)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    name = args.config if args.config in CONFIGS else 'c2'
    c = _full_cfg(name)
    world = int(os.environ.get('WORLD_SIZE', '1'))
    per_gpu = args.batch or (c['batch'] // world if c.get('strong') else c['batch'])
    vals = []
    for _ in range(max(args.warmup - 2, 0)):      # each call already does its own untimed warm-up pass
        cpu_baseline(name)
    t_all = time.perf_counter()
    cb = None
    for _ in range(args.steps):
        cb = cpu_baseline(name)
        vals.append(cb['value'])
    wall = time.perf_counter() - t_all
    v = sum(vals) / len(vals)
    cb['value'] = v
    line = {'impl': 'reference', 'metric': 'augmented images/sec', 'value': v, 'unit': 'img/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * wall / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': config_object(name, c, per_gpu, world, args.precision), 'cpu_baseline': cb,
            'e2e': {'value': v, 'unit': 'img/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}
    print(json.dumps(line))


def config_object(name, c, per_gpu, world, precision, weights=(1.0, 1.0, 0.0, 0.0), micro_batches=1):
    """The ``config`` object of the line: the same for the product arm and for ``--impl reference`` given the same flags
    (the reference arm runs "on your arm's config")."""
    w_lat, w_pix, w_lpips, w_disc = weights
    terms = f'w_latent={w_lat:g}, w_pix={w_pix:g}' + (f', w_lpips={w_lpips:g} (VGG16 perceptual term)' if w_lpips > 0 else '') + \
        (f', w_disc={w_disc:g} (StyleGAN2 discriminator term)' if w_disc > 0 else '')
    strong = bool(c.get('strong'))
    return {'workload': workload_name(name, c, per_gpu).replace('w_latent=w_pix=1', terms),
            'precision': precision,
            'l2': 'working set >> L2: ~2 GB of activations written and re-read per Adam step',
            'parallelism': (f'batch {c["batch"]} split over {world} rank(s)' if strong else f'batch-sharded x{world}')
            + ', no data-path collective' + (f'; {micro_batches} concurrent micro-batches per GPU' if micro_batches > 1 else '')}


def workload_name(name, c, per_gpu):
    return (f'{name}: StyleGAN2 {c["img_resolution"]}x{c["img_resolution"]} {c["img_channels"]}-ch, batch {per_gpu}/GPU, '
            f'{c["steps"]} w-opt steps + final synthesis, {c["bank"]}-code bank, {c["img_bank"]}-image bank, w_latent=w_pix=1')


def gpu_reference(cfg_name, core, w0, dev, ours, reps=2):
    """The reference's own fp32 torch GPU path (BASELINE.md §4 B2, the "vs reference fp32 torch path" comparator of C2):
    reference ``LatentAug.forward`` + ``torch_utils.ops`` with its JIT CUDA plugins + cuDNN on this GPU, on the SAME
    generator parameters, banks and initial codes as the product arm.  TF32 off = the parity oracle; TF32 on = the
    speed comparator.  ``ours`` = (img, w_aug) of the product for the same codes -> live parity of this very run."""
    import torch
    try:
        from oracle import ref_driver
        ref = ref_driver.import_reference()
    except FileNotFoundError as exc:
        return {'unavailable': str(exc)}
    c = _full_cfg(cfg_name)
    B = w0.shape[0]
    out = {'impl': "reference LatentAug.forward + torch_utils.ops on cuda (baseline/_ref, unmodified); generator class restated (not in the reference tree)"}
    try:
        out['plugins'] = ref_driver.init_cuda_plugins(ref)
        state = {k: v for k, v in core.generator_state.items()}
        for tf32 in (False, True):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            run, _ = ref_driver.reference_loop(c, batch=B, steps=c['steps'], device=dev, ref=ref, state=state, W=core.W, X=core.X,
                                               w0=w0.reshape(B, 1, -1))
            img, w_aug = run()              # warm-up (cuDNN heuristics, allocator)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                img, w_aug = run()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / reps
            key = 'tf32' if tf32 else 'fp32'
            out[key] = {'value': B / (ms * 1e-3), 'unit': 'img/s', 'ms_per_step': ms}
            if not tf32 and ours is not None:
                def rel(a, b):
                    return float((a.double() - b.double()).norm() / b.double().norm())
                wr = w_aug.detach()[:, 0]
                d = (ours[1].double() - wr.double()).abs()
                out['parity_vs_fp32'] = {'rel_l2_img': rel(ours[0], img.detach()), 'rel_l2_w': rel(ours[1], wr),
                                         'adam_sign_flips': int((d > 0.01).sum()), 'components': int(d.numel())}
            del run, img, w_aug
            torch.cuda.empty_cache()
    except Exception as exc:       # noqa: BLE001 -- a comparator failure must not lose the bench line
        out['error'] = f'{type(exc).__name__}: {str(exc)[:300]}'
    finally:
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = True
    return out


def c5_leg(rank, world, dev, per, warmup, reps, scaling):
    """Config C5 on an initialised process group (or a single process): queries x a row-sharded real-code bank; the local
    search (query split -> GEMM + fused top-k -> exact re-rank) replayed as one CUDA graph, then -- with more than one
    rank -- ONE NCCL all-gather of the per-rank (dist, idx) record + the merge kernel, all inside the timed region.
    Returns the JSON object of the leg (the same on every rank)."""
    import torch
    import torch.distributed as dist

    from latentaugment_b200 import parallel
    from latentaugment_b200.engine import LatentBank, pairwise_sqdist
    K, nq, k = C5['dim'], C5['queries'], C5['k']
    shard = torch.randn([per, K], generator=torch.Generator().manual_seed(1 + rank)).to(dev)
    X = torch.randn([nq, K], generator=torch.Generator().manual_seed(7)).to(dev)
    bank = LatentBank(shard, index_offset=rank * per)
    searcher = parallel.ShardedNearest(bank, nq, k)          # local search captured once; exchange + merge follow it per call
    try:
        for _ in range(warmup):
            d, i = searcher(X)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        clocks = ClockSampler(dev.index)
        mark = clocks.mark()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            d, i = searcher(X)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1) / reps
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        clk = clocks.stop(mark)
        # exact check of this rank's shard on 64 queries against the pairwise kernel (reference association order)
        ds, is_ = bank.nearest(X[:64], k)
        D = pairwise_sqdist(X[:64], shard)
        ref_d, ref_i = torch.topk(D.t(), k, dim=1, largest=False, sorted=True)
        exact = bool((ref_i + rank * per == is_).all()) or bool((ref_d == ds).all())
        merged_ok = None
        if world > 1:
            # ... and of the merged result: every rank's local lists gathered the plain way and merged by a stable sort
            # (rank order = index order, so ties go to the lowest index like the merge kernel's)
            d_loc, i_loc = bank.nearest(X, k)
            dl = [torch.empty_like(d_loc) for _ in range(world)]
            il = [torch.empty_like(i_loc) for _ in range(world)]
            dist.all_gather(dl, d_loc.contiguous())
            dist.all_gather(il, i_loc.contiguous())
            dc, ic = torch.cat(dl, dim=1), torch.cat(il, dim=1)
            order = torch.sort(dc, dim=1, stable=True).indices[:, :k]
            d, i = searcher(X)
            ok = torch.tensor([int(bool((torch.gather(ic, 1, order) == i).all()) and bool((torch.gather(dc, 1, order) == d).all())), int(exact)],
                              device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            merged_ok, exact = bool(ok[0].item()), bool(ok[1].item())
        # host-buffer leg: queries from pinned host memory, (dist, idx) back to the host
        Xh = X.cpu().pin_memory()
        t0 = time.perf_counter()
        for _ in range(20):
            Xd = Xh.to(dev, non_blocking=True)
            dd, ii = searcher(Xd)
            dd.cpu(), ii.cpu()
        torch.cuda.synchronize()
        e2e_ms = (time.perf_counter() - t0) / 20 * 1e3
        if world > 1:
            t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_ms = float(t.item())
        graph = searcher.graph is not None
    finally:
        searcher.close()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except OSError:
        pass
    codes = world * per
    flops = 2.0 * nq * codes * K
    peak_tf = peaks.get('bf16_tflops', 1590.0)
    peak_bw = peaks.get('hbm_gbs', 6650.0)
    ach = flops / world / (ms * 1e-3) / 1e12
    return {'metric': 'nearest-code queries/sec', 'value': nq / (ms * 1e-3), 'unit': 'queries/s', 'n_gpus': world, 'steps': reps,
            'warmup': warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': scaling,
            'vs_baseline': None, 'dtype': 'bf16 candidates (tensor core), f32/f64 exact re-rank', 'data': 'synthetic',
            'config': {'workload': f'c5: {codes} codes x {K} sharded over {world} GPU(s) ({per}/GPU), {nq} queries, k={k}, '
                                   'GEMM with fused top-k + exact re-rank (one CUDA graph)' + (' + NCCL all-gather + merge' if world > 1 else ''),
                       'l2': f'bank shard {per * K * 2 / 2**20:.0f} MiB bf16 + {per * K * 4 / 2**20:.0f} MiB f32 per GPU vs 126 MB L2'},
            'clocks': clk, 'indices_bit_exact_vs_pairwise': exact, 'merged_equals_gathered_lists': merged_ok,
            'e2e': {'value': nq / (e2e_ms * 1e-3), 'unit': 'queries/s', 'h2d_bytes_per_step': nq * K * 4, 'd2h_bytes_per_step': nq * k * 12},
            'gpu_launches': int(reps * (4 if world > 1 else 3)), 'graph_captured': graph,
            'roofline': {'bound': 'tensor', 'kernel': 'tapgemm_kernel<EPI=TopK> (query x bank GEMM + fused per-chunk top-2)',
                         'achieved': ach, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': ach / peak_tf, 'traffic': None,
                         'peak_source': 'MEASURED_PEAKS.json bf16_tflops (burst)' if peaks else 'fallback 1.59 PFLOP/s',
                         'note': 'achieved = 2 * queries * codes * K per GPU / the WHOLE search time (GEMM + re-rank + exchange), so it '
                                 'understates the GEMM kernel alone',
                         'hbm_floor_ms': (per * K * 2) / (peak_bw * 1e9) * 1e3},
            'cpu_baseline': None}


def run_c5(args):
    """``--config c5``: the nearest-code sweep as its own bench line."""
    import torch
    import torch.distributed as dist
    rank, world, lr = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1)), int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(lr)
    dev = cuda_device(lr)
    sys.stdout.flush()
    json_fd = os.dup(1)               # the NCCL banner goes to fd 1: keep stdout for the one JSON line
    os.dup2(2, 1)
    emitter = LineEmitter(rank, os.fdopen(json_fd, 'w'))
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    per = C5['codes'] // max(world, 1) if args.c5_total else C5['codes'] // 8
    wd = start_watchdog(300.0, emitter, 'the c5 sweep')
    line = c5_leg(rank, world, dev, per, max(args.warmup, 3), max(args.steps, 1) * 20, 'strong' if args.c5_total else 'weak')
    wd.cancel()
    emitter.set(line)
    emitter.emit()
    teardown_group(world, args.teardown_timeout)


def four_term_leg(rank, local_rank, world, dev):
    """The headline workload with ALL FOUR criteria at the author's weights (backbone_latentaug.py:46-56: w_lpips 10, w_pix 0.1,
    w_latent 0.001, w_disc 0.01): the discriminator and VGG16 forward / backward run inside every Adam step."""
    import torch
    c = _full_cfg('c2')
    B, res, C, steps = c['batch'], c['img_resolution'], c['img_channels'], c['steps']
    aug = make_plugin(c, B, local_rank, 'bf16', (0.001, 0.1, 10.0, 0.01))
    pt = PluginTimer(aug, B, res, rank, world, dev)
    ms, launches, _ = pt.resident(3, 3)
    e2e_s, out = pt.end_to_end(3)
    ok = out['A'].shape == (B, 1, res, res) and bool(torch.isfinite(out['A']).all())
    del pt, aug
    torch.cuda.empty_cache()
    return {'metric': 'augmented images/sec', 'value': world * B / (ms * 1e-3), 'unit': 'img/s', 'n_gpus': world, 'steps': 3, 'warmup': 3,
            'ms_per_step': ms, 'config': {'workload': workload_name('c2', c, B).replace(
                'w_latent=w_pix=1', 'w_lpips=10 (VGG16 perceptual term), w_pix=0.1, w_latent=0.001, w_disc=0.01 (StyleGAN2 discriminator term)')},
            'e2e': {'value': world * B / e2e_s, 'unit': 'img/s', 'h2d_bytes_per_step': B * 512 * 4, 'd2h_bytes_per_step': B * C * res * res * 4},
            'gpu_launches': int(launches), 'output_finite': ok}


def c3_leg(args, rank, local_rank, world, dev):
    """Config C3 on an initialised process group: SG2 512x512, batch 128 SPLIT over the ranks (strong scaling), through the
    plugin like the headline workload: device-resident and end-to-end numbers."""
    import torch
    c = _full_cfg('c3')
    B = c['batch'] // world
    res, C, steps = c['img_resolution'], c['img_channels'], c['steps']
    aug = make_plugin(c, B, local_rank, 'bf16', (1.0, 1.0, 0.0, 0.0))
    pt = PluginTimer(aug, B, res, rank, world, dev)
    clocks = ClockSampler(local_rank)
    ms, launches, _ = pt.resident(3, 3, clocks)
    e2e_s, out = pt.end_to_end(3)
    clk = clocks.stop(pt.mark)
    ok = out['A'].shape == (B, 1, res, res) and bool(torch.isfinite(out['A']).all())
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except OSError:
        pass
    peak_sust = peaks.get('bf16_tflops_sustained', 1400.0)
    fsyn = f_syn(res, C, channel_base=c['channel_base'], channel_max=c['channel_max'])
    value = world * B / (ms * 1e-3)
    del pt, aug
    torch.cuda.empty_cache()
    return {'metric': 'augmented images/sec', 'value': value, 'unit': 'img/s', 'n_gpus': world, 'steps': 3, 'warmup': 3, 'ms_per_step': ms,
            'scaling': 'strong', 'config': {'workload': workload_name('c3', c, B), 'parallelism': f'batch {c["batch"]} split over {world} rank(s), no data-path collective'},
            'e2e': {'value': world * B / e2e_s, 'unit': 'img/s', 'h2d_bytes_per_step': B * 512 * 4, 'd2h_bytes_per_step': B * C * res * res * 4},
            'gpu_launches': int(launches), 'clocks': clk, 'output_finite': ok,
            'whole_path_frac': (value / world) * (2 * steps + 1) * fsyn / (peak_sust * 1e12)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', default='c2', choices=sorted(CONFIGS) + ['c5'])
    ap.add_argument('--precision', default='bf16', choices=['bf16', 'fp32_parity'])
    ap.add_argument('--w-disc', type=float, default=0.0, help='weight of the discriminator realism term (0 = the headline workload)')
    ap.add_argument('--w-lpips', type=float, default=0.0, help='weight of the perceptual term (0 = the headline workload)')
    ap.add_argument('--author-weights', action='store_true',
                    help="the author's run configuration (backbone_latentaug.py:46-56): w_lpips 10, w_pix 0.1, w_latent 0.001, w_disc 0.01")
    ap.add_argument('--batch', type=int, default=0, help='override the per-GPU batch')
    ap.add_argument('--micro-batches', type=int, default=1, help='concurrent parts per GPU batch (own stream + graph each)')
    ap.add_argument('--c5-total', action='store_true', help='c5: keep 2^20 codes in total (strong scaling) instead of 2^17 per GPU')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-gpu-reference', action='store_true')
    ap.add_argument('--no-fp32-parity', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='default c2 run only: skip the C5 (sharded search) and C3 (512x512 split) legs')
    ap.add_argument('--extras-timeout', type=float, default=240.0, help='watchdog of those legs, seconds')
    ap.add_argument('--teardown-timeout', type=float, default=30.0, help='watchdog of destroy_process_group, seconds')
    ap.add_argument('--profile', action='store_true', help='short run for ncu: skips the e2e leg, the baselines and the per-GEMM timing')
    ap.add_argument('--layers-out', default='', help='write the per-layer tap-GEMM timing table (JSON) here')
    ap.add_argument('--dump-outputs', default='', metavar='DIR',
                    help="write rank 0's outputs of the last timed step (img, w_aug) as DIR/<name>.npy, float32, at most 64 MB "
                         'in all (beyond that, a fixed seeded subset of the batch)')
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == 'reference' or args.config == 'c5'):
        ap.error('--dump-outputs writes the outputs of the synthesis path: not with --impl reference or --config c5')
    sys.dont_write_bytecode = True          # the tree may be read-only: no bytecode caches are written into it
    if args.impl == 'reference':
        return run_reference(args)
    if args.config == 'c5':
        return run_c5(args)

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.warmup < 3:
        args.warmup = 3
    random.seed(0)            # crop windows of the perceptual term
    torch.manual_seed(0)      # noise of the final synthesis
    torch.cuda.set_device(local_rank)
    dev = cuda_device(local_rank)
    # stdout carries exactly ONE JSON line: everything else (plugin banners, the NCCL version line that
    # the C library writes to fd 1) goes to stderr -- at the file-descriptor level.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    real_stdout = os.fdopen(json_fd, 'w')
    sys.stdout = sys.stderr
    emitter = LineEmitter(rank, real_stdout)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    c = _full_cfg(args.config)
    strong = bool(c.get('strong'))
    B = args.batch or (c['batch'] // world if strong else c['batch'])
    steps, res, C = c['steps'], c['img_resolution'], c['img_channels']
    w_lat, w_pix, w_lpips, w_disc = 1.0, 1.0, args.w_lpips, args.w_disc
    if args.author_weights:
        w_lpips, w_pix, w_lat, w_disc = 10.0, 0.1, 0.001, 0.01

    # ---- the reference-facing plugin, synthetic mode (random-init generator, synthetic banks)
    aug = make_plugin(c, B, local_rank, args.precision, (w_lat, w_pix, w_lpips, w_disc), args.micro_batches)
    core = aug.latent_aug.module
    eng = core.engines[0]
    pt = PluginTimer(aug, B, res, rank, world, dev)

    # ---- kernel-resident metric: inputs already in HBM, no host copies in the timed region
    clocks = ClockSampler(local_rank)
    ms, launches, w_dev = pt.resident(args.warmup, args.steps, clocks)
    mark = pt.mark
    value = world * B / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(('img', 'w_aug'), pt.last)))

    if args.profile:
        clocks.stop(mark)
        emitter.set({'metric': 'augmented images/sec', 'value': value, 'unit': 'img/s', 'ms_per_step': ms,
                     'gpu_launches': int(launches), 'note': 'profile mode (no e2e / roofline / baseline legs)'})
        emitter.emit()
        return

    # ---- end to end through the plugin API: host dict in, host dict out (the output of batch t is fetched while
    # batch t+1 runs: double-buffered pinned outputs, latent_aug.py get_output)
    time.sleep(3.0)      # both legs start from a comparable power / thermal state (the kernels are power-capped)
    e2e_s, out = pt.end_to_end(args.steps)
    clk = clocks.stop(mark)
    e2e = {'value': world * B / e2e_s, 'unit': 'img/s', 'h2d_bytes_per_step': B * eng.w_dim * 4,
           'd2h_bytes_per_step': B * C * res * res * 4}
    assert out['A'].shape == (B, 1, res, res) and bool(torch.isfinite(out['A']).all())

    line = None
    if rank == 0:
        # ---- roofline of the dominant kernel (tap-GEMM): every launch of one Adam step timed ALONE (burst peak)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except OSError:
            pass
        peak_burst = peaks.get('bf16_tflops', 1590.0)
        peak_sust = peaks.get('bf16_tflops_sustained', 1400.0)
        src = 'MEASURED_PEAKS.json' if peaks else 'fallback (B200_PROFILING.md)'
        rows, rgb_macs = layer_table(res, C, c['channel_base'], c['channel_max'])
        t = eng.debug_time_gemms(reps=10)
        tot_ms = sum(t['forward']) + sum(t['dgrad'])
        Bm = eng.batch                                                    # (a micro-batch part when --micro-batches > 1)
        alg = 2.0 * 2.0 * Bm * sum(r['alg_macs'] for r in rows)         # fwd + dgrad launches of one step
        exe = 2.0 * 2.0 * Bm * sum(r['exe_macs'] for r in rows) * (3 if args.precision == 'fp32_parity' else 1)
        ach = alg / (tot_ms * 1e-3) / 1e12
        fsyn = f_syn(res, C, channel_base=c['channel_base'], channel_max=c['channel_max'])
        traffic, traffic_src = None, None   # DRAM bytes (read + write) of the same launches: one ncu --set full capture of this workload
        if args.config == 'c2' and args.precision == 'bf16' and B == 32:
            for fn in ('r2_tapgemm_traffic.json', 'r1c_tapgemm_traffic.json'):       # newest capture first
                try:
                    traffic = json.load(open(os.path.join(ROOT, 'profiles', fn)))['dram_bytes_read_plus_write']
                    traffic_src = f'profiles/{fn} (ncu dram__bytes_read.sum + dram__bytes_write.sum, not measured in this run)'
                    break
                except (OSError, KeyError, ValueError):
                    pass
        roof = {'bound': 'tensor', 'kernel': f'tapgemm_kernel ({2 * len(rows)} launches of one Adam step: forward + data-gradient)',
                'achieved': ach, 'peak': peak_burst, 'unit': 'TFLOP/s', 'frac': ach / peak_burst, 'traffic': traffic,
                'traffic_source': traffic_src,
                'peak_source': f'{src} bf16_tflops (burst: the launches are timed alone)', 'executed_tflops': exe / (tot_ms * 1e-3) / 1e12,
                'launch_ms_sum': tot_ms, 'seed_ms': t['seed'], 'fir_pass_ms_sum': sum(t['fir_forward']) + sum(t['fir_backward']),
                'whole_path_frac': (value / world) * (2 * steps + 1) * fsyn / (peak_sust * 1e12),
                'whole_path_peak': peak_sust, 'whole_path_peak_source': f'{src} bf16_tflops_sustained (kernels timed inside the seconds-long step)'}
        if args.layers_out:
            tab = [dict(r, fwd_ms=t['forward'][i], dgrad_ms=t['dgrad'][i], fir_fwd_ms=t['fir_forward'][i], fir_bwd_ms=t['fir_backward'][i],
                        fwd_alg_tflops=2.0 * Bm * r['alg_macs'] / (t['forward'][i] * 1e-3) / 1e12,
                        dgrad_alg_tflops=2.0 * Bm * r['alg_macs'] / (t['dgrad'][i] * 1e-3) / 1e12) for i, r in enumerate(rows)]
            json.dump({'config': args.config, 'precision': args.precision, 'batch': B, 'layers': tab, 'seed_ms': t['seed']},
                      open(args.layers_out, 'w'), indent=1)
        # ---- the tolerance-matched mode (<= 1e-3) measured in the same run
        extra = {}
        if world == 1 and args.precision == 'bf16' and not args.no_fp32_parity and w_lpips == 0 and w_disc == 0:
            from latentaugment_b200.engine import SynthesisEngine
            e32 = SynthesisEngine(core.generator_state, img_resolution=res, img_channels=C, w_dim=eng.w_dim, z_dim=eng.z_dim,
                                  batch=B, precision='fp32_parity', device=dev)
            e32.set_latent_bank(core.W)
            e32.set_image_bank(core.X)
            for i in range(2):
                e32.augment(w_dev[i], num_steps=steps)
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for i in range(3):
                e32.augment(w_dev[i], num_steps=steps)
            a1.record()
            torch.cuda.synchronize()
            v32 = B / (a0.elapsed_time(a1) / 3 * 1e-3)
            extra['fp32_parity'] = {'value': v32, 'unit': 'img/s', 'whole_path_frac': v32 * (2 * steps + 1) * fsyn / (peak_sust * 1e12),
                                    'note': 'split-bf16 (hi+lo) operands, 3 MMA passes: the <= 1e-3 tolerance mode'}
            del e32
            torch.cuda.empty_cache()
        if world == 1 and not args.no_gpu_reference and w_lpips == 0 and w_disc == 0:
            w0 = w_dev[0]
            ours = core.forward(w0)
            torch.cuda.synchronize()
            extra['gpu_reference'] = gpu_reference(args.config, core, w0.reshape(B, -1), dev, (ours[0].detach(), ours[1].detach()[:, 0]))
        cb = None
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_baseline(args.config)
        line = {'metric': 'augmented images/sec', 'value': value, 'unit': 'img/s', 'n_gpus': world, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'strong' if strong else 'weak',
                'vs_baseline': None,
                'dtype': 'bf16 operands, f32 accumulate' if args.precision == 'bf16' else 'split-bf16 (hi+lo) operands, f32 accumulate',
                'data': 'synthetic',
                'config': config_object(args.config, c, B, world, args.precision, (w_lat, w_pix, w_lpips, w_disc), args.micro_batches),
                'clocks': clk, 'e2e': e2e, 'gpu_launches': int(launches), 'roofline': roof, 'cpu_baseline': cb}
        line.update(extra)
    emitter.set(line)
    # ---- the other two GPU configurations of BASELINE.json in the same (driver-launched) run: C5 = the sharded nearest-code
    # sweep with the design's ONE collective, C3 = 512x512 with batch 128 split over the ranks.  All collectives of the
    # headline measurement are complete by now; a watchdog prints the line without these legs if one of them wedges.
    headline = (args.config == 'c2' and args.precision == 'bf16' and w_lpips == 0 and w_disc == 0 and not args.author_weights
                and not args.batch and args.micro_batches == 1)
    if headline and not args.no_extras:
        wd = start_watchdog(args.extras_timeout, emitter, 'the C5 / C3 legs')
        extras = {}
        legs = [('c5_sharded_search', lambda: c5_leg(rank, world, dev, C5['codes'] // 8, 3, 40, 'weak')),
                ('c3_strong_split', lambda: c3_leg(args, rank, local_rank, world, dev))]
        if world == 1:
            legs.append(('four_terms_author_weights', lambda: four_term_leg(rank, local_rank, world, dev)))
        for key, leg in legs:
            try:
                extras[key] = leg()
            except Exception as exc:      # noqa: BLE001 -- a failing extra leg must not lose the headline line
                extras[key] = {'error': f'{type(exc).__name__}: {str(exc)[:300]}'}
                break                     # the ranks may be out of step now: no further collective
        wd.cancel()
        emitter.update(extras)
        if any('error' in v for v in extras.values()):
            emitter.emit()                # the ranks may be out of step (or the context poisoned): no graceful teardown
            sys.stderr.write(f'bench.py: extra leg failed: {extras}\n')
            sys.stderr.flush()
            real_stdout.flush()
            os._exit(0)
    emitter.emit()
    teardown_group(world, args.teardown_timeout)


if __name__ == '__main__':
    main()
