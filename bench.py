#!/usr/bin/env python
"""bench.py -- pair scores / second of the all-pairs ViT-ED scoring path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload puzzle|hisfrag --items F]

A "step" is one pass of the hot path over one batch of synthetic input:
  * N=1 : BASELINE.json configs[1] -- one synthetic 540-piece puzzle (18x30 grid of 64 px pieces, erosion 7 %,
          4-bin puzzle model patch8/64): 291,060 ordered pairs per step;
  * N>1 : BASELINE.json configs[2] -- 1000-piece puzzles (25x40, erosion 14 %), the (puzzle, row) units of the pair
          grid sharded over the ranks with no data-path collective, 2,500 units per GPU (= exactly configs[2] at
          N=8), one NCCL all-gather of the score blocks at the end of the step ("weak" scaling), through the
          package's own entry point grid.score_puzzles.
  * --workload hisfrag: BASELINE.json configs[3]'s model (patch16 / 512 px) on `--items` synthetic fragments, all
          pairs a <= b, rows sharded over the ranks by the reference sampler's boundaries, through
          grid.score_fragments (NCCL all-gather inside); fixed total work -> "strong" scaling.
`--dump-outputs DIR` writes what the timed path returned in its last timed step to DIR/<name>.npy (see dump_outputs);
the inputs are seeded, so two builds run with the same arguments can be compared output for output.
`value` is timed on the device with the piece images already resident in HBM; `e2e` goes through the public API with
HOST buffers (pinned), H2D and D2H inside the timed region. `roofline` is measured live: one extra step with a CUDA
event before every launch (engine option PROFILE) gives every kernel family's summed duration; the family with the
largest share of the step is the roofline object (algorithmic bytes or FLOPs of its launches / that time), the others
are listed under `other_kernels`. `cpu_baseline` / `--impl reference` time the reference's algorithm for this
path (evaluation.py:101-107: one-shot fp32 model(images) on stacked pairs, nothing cached) as restated by the oracle,
on the box's host cores, on a bounded sample.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from as it found it (it may be read-only)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = 'pair scores/sec (all-pairs ViT-ED)'
UNIT = 'pairs/s'
UNITS_PER_GPU = int(os.environ.get('VITED_BENCH_UNITS', '2500'))

# algorithmic FLOPs (SURVEY 8d), puzzle model: D=384, N_e=64, N_d=65, L=8, C=4
F_DEC_PAIR = 8 * (28 * 384 * 384 * 65 + 4 * 65 * 65 * 384 + 4 * 65 * 64 * 384) + 2 * 384 * 4
F_ENC_ITEM = 8 * (24 * 384 * 384 * 64 + 4 * 64 * 64 * 384) + 2 * 64 * 192 * 384
F_KV_ITEM = 8 * 4 * 384 * 384 * 64
F_PREP_ITEM = 2 * 64 * 192 * 384
DUMP_LIMIT = 64_000_000   # bytes that --dump-outputs writes at most, .npy headers included


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d['hbm_gbs'], tf_burst=d['bf16_tflops'], tf_sustained=d.get('bf16_tflops_sustained', d['bf16_tflops']),
                    source='measured (MEASURED_PEAKS.json)')
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source='fallback (B200_PROFILING.md)')


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each tensor of `arrays` (name -> tensor) as out_dir/<name>.npy, float64 kept as float64 and
    everything else as float32. Smallest first, each array gets an equal share of what DUMP_LIMIT has left; one that
    does not fit its share is written as a fixed sample of its flattened elements instead (1-D, indices drawn with
    replacement by a generator seeded with 0 and sorted), so every run with the same arguments samples the same
    elements. Outputs that fit DUMP_LIMIT together are written whole."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: (v.detach().double() if v.dtype == torch.float64 else v.detach().float()).cpu() for k, v in arrays.items()}
    header = 4096   # bytes reserved per file for the .npy header
    left = DUMP_LIMIT
    for i, (name, v) in enumerate(sorted(arrays.items(), key=lambda kv: kv[1].numel() * kv[1].element_size())):
        share = left // (len(arrays) - i) - header
        if v.numel() * v.element_size() > share:
            idx = torch.randint(v.numel(), (share // v.element_size(),), generator=torch.Generator().manual_seed(0))
            v = v.reshape(-1)[idx.sort().values]
        np.save(os.path.join(out_dir, f'{name}.npy'), v.numpy())
        left -= v.numel() * v.element_size() + header


# ----------------------------------------------------------------------------------------------- workloads
def _pure(name):
    """vit-ed_b200/<name>.py loaded by path, WITHOUT importing the package (whose __init__ dlopens the CUDA library):
    synthetic.py and pieces.py are plain numpy / torch host code. The reference arm uses only these, so that none of
    this repo's native code is mapped into its process."""
    import importlib.util
    spec = importlib.util.spec_from_file_location(f'_vited_pure_{name}', os.path.join(ROOT, 'vit-ed_b200', f'{name}.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


PUZZLE_KW = dict(img_size=64, patch_size=8, num_classes=4, embed_dim=384, depth=8, c_depth=8, num_heads=12)
HISFRAG_KW = dict(img_size=512, patch_size=16, num_classes=1, embed_dim=384, depth=12, c_depth=12, num_heads=6)


def puzzle_pieces(rows, cols, erosion, seed):
    """Synthetic puzzle -> [rows*cols, 3, 64, 64] fp32 through the reference's a1-a3 steps (pieces.py)."""
    pieces, synthetic = _pure('pieces'), _pure('synthetic')
    img = synthetic.synthetic_puzzle_image(rows, cols, piece=64, seed=seed)
    lab, grid_size = pieces.make_pieces_lab(img, 64, erosion)
    assert grid_size == (rows, cols)
    return pieces.pieces_to_batch(lab, 64)


def build_model():
    import vited_b200
    from vited_b200 import synthetic
    model = vited_b200.build_model(vited_b200.get_config('puzzle'))
    model.load_state_dict(synthetic.synthetic_state_dict(model, seed=0), strict=True)
    return model


class ClockSampler:
    """Samples SM clock and throttle reasons during the timed region (NVML; falls back to nvidia-smi)."""
    REASONS = {0x4: 'sw_power_cap', 0x8: 'hw_slowdown', 0x20: 'sw_thermal_slowdown', 0x40: 'hw_thermal_slowdown',
               0x80: 'hw_power_brake_slowdown'}

    def __init__(self, device_index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        self._h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            try:
                uuid = torch.cuda.get_device_properties(device_index).uuid
                self._h = pynvml.nvmlDeviceGetHandleByUUID(('GPU-' + str(uuid)).encode())
            except Exception:
                self._h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._h = None

    def _loop(self):
        while not self._stop.is_set():
            try:
                if self._h is not None:
                    nv = self._nv
                    self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                    try:
                        bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                    except Exception:
                        bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                    for bit, name in self.REASONS.items():
                        if bits & bit:
                            self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        self._stop.clear()
        self._thread = threading.Thread(target=self._loop, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=2)
        return dict(sm_mhz=float(np.median(self.samples)) if self.samples else None, sm_max_mhz=self.max_mhz,
                    reasons=sorted(self.reasons), samples=len(self.samples))


def dist_setup(n_gpus):
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        torch.cuda.set_device(local)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    else:
        torch.cuda.set_device(0)
    if world != n_gpus:
        raise SystemExit(f'--gpus {n_gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {n_gpus}')
    return rank, world, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(ms, world):
    if world == 1:
        return ms
    import torch.distributed as dist
    t = torch.tensor([ms], dtype=torch.float64, device='cuda')
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


# ----------------------------------------------------------------------------------------------- CPU reference arm
def cpu_reference_rate(budget_s, steps=1, warmup=0, batch=128):
    """The reference's puzzle evaluation forward (evaluation.py:101-107): fp32 one-shot model(images) on stacked
    pairs in batches of 128 (README.md:40), nothing cached -- restated by the oracle, all host threads.
    Returns (pairs/s, cores, sample description, per-step seconds)."""
    from oracle import vited_oracle as orc
    synthetic = _pure('synthetic')
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = synthetic.synthetic_state_dict(synthetic.state_dict_shapes(**PUZZLE_KW), seed=0)
    imgs = puzzle_pieces(4, 8, 0.07, seed=0)  # 32 pieces of the same kind as configs[1]
    pairs = orc.ordered_pairs(imgs.shape[0])

    def run(n_batches):
        done = 0
        for b in range(n_batches):
            sub = pairs[(b * batch) % (len(pairs) - batch):][:batch]
            x = torch.stack([imgs[sub[:, 0]], imgs[sub[:, 1]]], dim=1)
            orc.forward(sd, 12, x)
            done += len(sub)
        return done

    t0 = time.perf_counter()
    run(1)
    probe = time.perf_counter() - t0  # includes first-touch; calibrates the sample size
    per_step_budget = max(budget_s / max(steps + warmup, 1), probe)
    n_batches = max(1, min(8, int(per_step_budget / max(probe, 1e-3))))
    for _ in range(warmup):
        run(n_batches)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        n = run(n_batches)
        times.append(time.perf_counter() - t0)
    sec = float(np.mean(times))
    sample = f'{n_batches} batch(es) of {batch} stacked pairs of 64px pieces per step, one-shot fp32 forward (4.43 GFLOP/pair)'
    return n / sec, cores, sample, sec


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    rate, cores, sample, sec = cpu_reference_rate(budget_s=150.0, steps=args.steps, warmup=args.warmup)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': rate, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': sec * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args.gpus),
        'cpu_baseline': {'value': rate, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': rate, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
        'note': 'reference model file needs timm (absent); the oracle port of its forward is timed on host cores',
    }
    print(json.dumps(line))


def workload_config(n_gpus):
    if n_gpus == 1:
        return {'workload': 'configs[1]: puzzle all-pairs scoring, one synthetic 540-piece puzzle (18x30) at 64px, '
                            'erosion 7%, 4-bin patch8 model, 291060 ordered pairs per step',
                'pairs_per_step': 540 * 539, 'l2': 'per-step working set (~5 GB of activations per 8065-pair chunk) >> 126 MB L2'}
    n_puzzles = max(1, round(n_gpus * UNITS_PER_GPU / 1000))
    return {'workload': f'configs[2]: batch of {n_puzzles} synthetic 1000-piece puzzles (25x40) at 64px, erosion 14%, the '
                        f'{n_puzzles * 1000} (puzzle,row) units sharded over {n_gpus} GPUs by grid.score_puzzles '
                        f'({n_puzzles * 1000 // n_gpus} per GPU), one NCCL all-gather of the score blocks per step',
            'pairs_per_step': n_puzzles * 1000 * 999, 'parallelism': f'grid rows sharded x{n_gpus}',
            'l2': 'per-step working set >> 126 MB L2'}


def torch_gpu_rate(dev, host_pieces, rows=48, batch=4096):
    """pairs/s of the reference's algorithm run by stock PyTorch on this GPU: the oracle's functional restatement of the
    model (oracle/vited_oracle.py; the reference's model file itself needs timm) under fp16 autocast -- the reference's
    own GPU setting, config.py:216 -- with F.scaled_dot_product_attention, two-phase and cached as hisfrag.py:214,229
    does (encode every piece once, decode pairs against cached tokens), on the first `rows` grid rows of the bench
    puzzle. cuBLAS / SDPA kernels only; none of this repo's kernels. Reported as context, like cpu_baseline."""
    from oracle import vited_oracle as orc
    sd = {k: v.to(dev) for k, v in _pure('synthetic').synthetic_state_dict(
        _pure('synthetic').state_dict_shapes(**PUZZLE_KW), seed=0).items()}
    imgs = host_pieces.to(dev)
    n = imgs.shape[0]
    rows = min(rows, n)
    ii, jj = torch.meshgrid(torch.arange(rows, device=dev), torch.arange(n, device=dev), indexing='ij')
    keep = ii != jj
    ii, jj = ii[keep], jj[keep]
    orc.USE_SDPA = True
    try:
        def run():
            with torch.no_grad(), torch.autocast('cuda', dtype=torch.float16):
                tokens = torch.cat([orc.forward_first_part(imgs[i:i + 512], sd, 12) for i in range(0, n, 512)])
                outs = [orc.forward_head(orc.forward_second_part(tokens[ii[p:p + batch]], imgs[jj[p:p + batch]], sd, 12), sd)
                        for p in range(0, ii.numel(), batch)]
            return torch.cat(outs)
        run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run()
        e1.record()
        torch.cuda.synchronize()
    finally:
        orc.USE_SDPA = False
    ms = e0.elapsed_time(e1)
    return {'value': ii.numel() / (ms / 1e3), 'unit': UNIT, 'kind': 'oracle functional model on cuda, fp16 autocast, SDPA, '
            'two-phase cached (all pieces encoded, then pairs decoded in batches of %d)' % batch,
            'sample': f'{rows} grid rows x {n - 1} columns = {ii.numel()} pairs of the bench puzzle, 1 timed pass after 1 warm-up',
            'ms': ms}


# ----------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import vited_b200
    from vited_b200 import grid
    # stdout carries exactly ONE JSON line: anything libraries print meanwhile (NCCL's version banner) goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    rank, world, local = dist_setup(args.gpus)
    dev = torch.device('cuda', local if world > 1 else 0)
    peaks = load_peaks()
    model = build_model().to(dev).eval()

    if world == 1:
        host_images = {0: puzzle_pieces(18, 30, 0.07, seed=0).pin_memory()}
        n_pieces = [540]
        mine = [(0, 0, 540)]
    else:
        # configs[2]: 1000-piece puzzles, (puzzle, row) units sharded by the package (grid.puzzle_unit_ranges)
        n_puzzles = max(1, round(world * UNITS_PER_GPU / 1000))
        n_pieces = [1000] * n_puzzles
        mine = grid.puzzle_unit_ranges(n_pieces, world, rank)
        host_images = {pz: puzzle_pieces(25, 40, 0.14, seed=pz).pin_memory() for pz, _, _ in mine}
    n_pairs_rank = sum((hi - lo) * (n_pieces[pz] - 1) for pz, lo, hi in mine)
    n_pairs_job = sum(n * (n - 1) for n in n_pieces)
    dev_images = {pz: h.to(dev) for pz, h in host_images.items()}
    host_out = [torch.empty((n, n, 4), dtype=torch.float32).pin_memory() for n in n_pieces]

    def step(images):
        """One pass of the hot path through the package's public entry points: a whole puzzle (N = 1) or this rank's
        share of the batch of puzzles plus the all-gather of the score blocks (N > 1). Returns the full score
        matrices, resident on this GPU."""
        if world == 1:
            return [grid.score_puzzle(model, images[0])]
        return grid.score_puzzles(model, [images.get(pz) for pz in range(len(n_pieces))], n_pieces=n_pieces)

    def step_e2e():
        imgs = {pz: h.to(dev, non_blocking=True) for pz, h in host_images.items()}
        for dst, res in zip(host_out, step(imgs)):
            dst.copy_(res, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    # ---- device-resident timing
    for _ in range(args.warmup):
        step(dev_images)
    barrier(world)
    clocks = ClockSampler(dev.index or 0)
    launches0 = model.launch_count()
    clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        scores = step(dev_images)
    e1.record()
    torch.cuda.synchronize()
    clock_info = clocks.stop()
    barrier(world)
    launches = model.launch_count() - launches0
    ms_step = max_over_ranks(e0.elapsed_time(e1) / args.steps, world)
    value = n_pairs_job / (ms_step / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {f'logits_puzzle{pz}': s for pz, s in enumerate(scores)})
    del scores

    # ---- end to end through the public API with host buffers
    for _ in range(2):
        step_e2e()
    barrier(world)
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        step_e2e()
    t1.record()
    torch.cuda.synchronize()
    ms_e2e = max_over_ranks(t0.elapsed_time(t1) / args.steps, world)
    e2e_value = n_pairs_job / (ms_e2e / 1e3)
    h2d = int(sum(h.numel() * 4 for h in host_images.values()))
    d2h = int(sum(h.numel() * 4 for h in host_out))

    # ---- per-kernel timing of one more step (roofline of the dominant kernel)
    model.set_option(vited_b200.OPT_PROFILE, 1)
    step(dev_images)
    prof = model.profile_read()
    model.set_option(vited_b200.OPT_PROFILE, 0)
    total_ms = sum(v['ms'] for v in prof.values()) or 1.0
    # kernel families of the step; the roofline object describes the one with the largest share of the step
    #   gemm_ln : gemm_ln_pair_kernel (Linear + residual + LayerNorm fused, N = 384): bound by HBM (fp32 residual in/out)
    #   gemm    : gemm_tc_pair_kernel / gemm_tc_kernel (tcgen05 GEMMs with bias / GELU epilogue): tensor bound
    #   attn    : attn_p64_kernel (tcgen05 attention, 65-token sequences): HBM bound
    # `traffic` (dram__bytes_read.sum + dram__bytes_write.sum per launch) cannot be measured inside this process; it
    # is filled from the committed ncu --set full capture of the SAME kernels at the SAME per-launch shape
    # (profiles/ncu_traffic.json, written by tools/ncu_traffic.py from the raw page) when this run's algorithmic bytes
    # per launch match the capture's to 2 %, and is null otherwise.
    #   mlp_ln  : mlp_ln_pair_kernel (fc1 + GELU + fc2 + residual + LayerNorm, hidden activations in TMEM): tensor bound
    fams = {
        'mlp_ln': dict(match=lambda k: k.startswith('mlp_ln'), bound='tensor',
                       kernel='mlp_ln_pair_kernel (tcgen05 fc1 -> GELU -> fc2 with the hidden chunk handed over in TMEM, + residual + LayerNorm full-row epilogue)'),
        'gemm_ln': dict(match=lambda k: k.startswith('gemm_ln_'), bound='hbm',
                        kernel='gemm_ln_pair_kernel (tcgen05 Linear + residual + LayerNorm, full-row epilogue out of TMEM)'),
        'gemm': dict(match=lambda k: k.startswith('gemm_n'), bound='tensor',
                     kernel='gemm_tc_pair_kernel (tcgen05/TMEM/TMA cta_group::2 GEMM, bias / GELU epilogue)'),
        'attn': dict(match=lambda k: k in ('attn_self', 'attn_cross'), bound='hbm',
                     kernel='attn_p64_kernel (tcgen05 attention, S/P/O in TMEM)'),
    }
    traffic_db = {}
    tpath = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if os.path.exists(tpath):
        traffic_db = json.load(open(tpath))

    def measured_traffic(sel):
        """launch-weighted DRAM bytes per launch of a family from the ncu capture, or (None, why)."""
        tot, n = 0.0, 0
        for k, v in sel.items():
            rec = traffic_db.get('kernels', {}).get(k)
            if rec is None:
                return None, f'no ncu capture of {k} in profiles/ncu_traffic.json'
            alg = v['bytes'] / max(v['launches'], 1)
            if abs(alg - rec['algorithmic_bytes']) > 0.02 * rec['algorithmic_bytes']:
                return None, f'{k}: this run moves {alg:.4g} algorithmic B/launch, the capture {rec["algorithmic_bytes"]:.4g}'
            tot += rec['dram_bytes'] * v['launches']
            n += v['launches']
        return (tot / n if n else None), traffic_db.get('source', 'profiles/ncu_traffic.json')

    def family_roofline(name):
        f = fams[name]
        sel = {k: v for k, v in prof.items() if f['match'](k)}
        ms = sum(v['ms'] for v in sel.values())
        n = sum(v['launches'] for v in sel.values())
        if ms <= 0:
            return None
        traffic = measured_traffic(sel)
        if f['bound'] == 'tensor':
            ach = sum(v['flops'] for v in sel.values()) / (ms / 1e3) / 1e12
            peak, unit = peaks['tf_sustained'], 'TFLOP/s'
        else:
            ach = sum(v['bytes'] for v in sel.values()) / (ms / 1e3) / 1e9
            peak, unit = peaks['hbm_gbs'], 'GB/s'
        return {'bound': f['bound'], 'kernel': f['kernel'], 'achieved': ach, 'peak': peak, 'unit': unit, 'frac': ach / peak,
                'peak_source': peaks['source'] + (', sustained dense 16-bit figure (measured by the driver with bf16; fp16 operands run at the same rate; kernel timed inside a long step)' if f['bound'] == 'tensor' else ''),
                'traffic': traffic[0], 'traffic_source': traffic[1],
                'launches_per_step': n, 'avg_launch_ms': ms / max(n, 1),
                'algorithmic_per_launch': (sum(v['flops'] for v in sel.values()) if f['bound'] == 'tensor'
                                           else sum(v['bytes'] for v in sel.values())) / max(n, 1),
                'share_of_step': ms / total_ms}

    fam_lines = {k: family_roofline(k) for k in fams}
    fam_lines = {k: v for k, v in fam_lines.items() if v}
    top = max(fam_lines, key=lambda k: fam_lines[k]['share_of_step'])
    roofline = dict(fam_lines[top])
    roofline['other_kernels'] = {k: v for k, v in fam_lines.items() if k != top}
    roofline['classes'] = {k: {'ms': round(v['ms'], 3), 'share': round(v['ms'] / total_ms, 4),
                               'tflops': round(v['flops'] / max(v['ms'], 1e-9) / 1e9, 1),
                               'gbs': round(v['bytes'] / max(v['ms'], 1e-9) / 1e6, 1), 'launches': v['launches']}
                           for k, v in sorted(prof.items(), key=lambda kv: -kv[1]['ms'])}
    # whole-step algorithmic work against the tensor roofline
    n_items_total = sum(img.shape[0] for img in dev_images.values())
    n_ctx = sum(hi - lo for _, lo, hi in mine)
    f_step = n_pairs_rank * F_DEC_PAIR + n_items_total * F_PREP_ITEM + n_ctx * (F_ENC_ITEM + F_KV_ITEM)
    step_frac = f_step / (ms_step / 1e3) / 1e12 / peaks['tf_sustained']
    # FLOPs actually launched (layer-0 self-attention runs once per item, the last layer runs on class-token rows
    # only): sum of the per-launch algorithmic flops the engine attached to the profiled step
    f_exec = sum(v['flops'] for v in prof.values())
    step_frac_exec = f_exec / (ms_step / 1e3) / 1e12 / peaks['tf_sustained']

    # ---- the multi-GPU workload on ONE GPU (so that the 1 -> N curve can be read on the same workload): rank 0's share
    #      of configs[2] at 8 GPUs -- 2,500 (puzzle, row) units of 1000-piece puzzles -- scored here, no collective
    same_workload = None
    if world == 1 and not args.no_extras:
        share = grid.puzzle_unit_ranges([1000] * max(1, round(8 * UNITS_PER_GPU / 1000)), 8, 0)
        imgs2 = {pz: puzzle_pieces(25, 40, 0.14, seed=pz).to(dev) for pz, _, _ in share}

        def step2():
            for pz, lo, hi in share:
                model.score_grid(imgs2[pz], vited_b200.GRID_ORDERED_OFFDIAG, lo, hi)

        step2()
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        step2()
        s1.record()
        torch.cuda.synchronize()
        units = sum(hi - lo for _, lo, hi in share)
        same_workload = {'value': units * 999 / (s0.elapsed_time(s1) / 1e3), 'unit': UNIT, 'units': units,
                         'workload': 'configs[2] share of one of 8 GPUs (1000-piece puzzles, erosion 14%), 1 timed step after 1 warm-up'}
        del imgs2

    # ---- the reference's own torch path on this GPU (SURVEY 2: "the same PyTorch model running through the stock torch
    #      libraries"): context for the speed-up, timed OUTSIDE the timed regions above
    torch_gpu = None
    if world == 1 and not args.no_extras:
        torch_gpu = torch_gpu_rate(dev, host_images[0])

    if rank == 0:
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': vited_b200.ACT_NAME,
            'data': 'synthetic', 'config': workload_config(world),
            'clocks': clock_info,
            'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                    'ms_per_step': ms_e2e},
            'gpu_launches': int(launches),
            'roofline': roofline,
            'step_tensor_frac': step_frac,
            'step_tensor_frac_executed': step_frac_exec,
            'flops_note': 'step_tensor_frac uses SURVEY 8d nominal work (2.250 GFLOP/pair, all 8 decoder layers on all 65 '
                          'rows); _executed counts only launched flops (layer-0 self-attention cached per item, last '
                          'layer pruned to the class-token row)',
        }
        if same_workload is not None:
            line['config']['same_workload_n1_rate'] = same_workload
        if torch_gpu is not None:
            line['torch_gpu_baseline'] = torch_gpu
        if world == 1 and not args.no_cpu:
            rate, cores, sample, _ = cpu_reference_rate(budget_s=20.0, steps=1, warmup=0)
            line['cpu_baseline'] = {'value': rate, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample}
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def run_hisfrag(args):
    """BASELINE.json configs[3]'s model (Hisfrag20 patch16 / 512 px, 12 + 12 layers) on an all-pairs grid of `--items`
    synthetic fragments at `--gpus` N, THROUGH grid.score_fragments: rows sharded by the reference sampler's boundaries
    (data/samplers.py:108-137), every rank encodes and scores its rows, one NCCL all-gather of the row blocks, the
    upper triangle mirrored. Total work is fixed -> "strong" scaling. Reports whole-job pairs/s (max over ranks), the
    tensor-roofline fraction with the Hisfrag FLOP model of SURVEY 8d (89.50 GFLOP / pair, 63.42 + 7.25 + 0.60 GFLOP
    per item), each rank's rows / pairs / local time (no collective), and rank 0's per-kernel shares."""
    import vited_b200
    from vited_b200 import grid, synthetic
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    rank, world, local = dist_setup(args.gpus)
    dev = torch.device('cuda', local if world > 1 else 0)
    peaks = load_peaks()
    model = vited_b200.build_model(vited_b200.get_config('hisfrag'))
    model.load_state_dict(synthetic.synthetic_state_dict(model, seed=0), strict=True)
    model = model.to(dev).eval()
    n = args.items
    if n <= 512:
        images = synthetic.synthetic_images(n, 512, seed=1000, smooth=False).to(dev)
    else:   # built in blocks of 128 so that eight ranks do not hold 8 x 40 GB of host temporaries (4096 fragments)
        images = torch.empty(n, 3, 512, 512, device=dev)
        for c0 in range(0, n, 128):
            images[c0:c0 + 128] = synthetic.synthetic_images(min(128, n - c0), 512, seed=1000 + c0, smooth=False).to(dev)
    n_pairs = n * (n + 1) // 2
    if world == 1:
        lo, hi = 0, n
    else:
        sizes = grid.indicates_row_ranges(grid.upper_tri_pairs(n)[:, 0], world)
        lo, hi = (sizes[rank], sizes[rank + 1]) if rank + 1 < len(sizes) else (n, n)
    my_pairs = (hi - lo) * n - (hi * (hi - 1) - lo * (lo - 1)) // 2
    if args.lean:
        # full-size runs (4096 fragments = 8.4 M pairs: minutes per pass): warm up on the first 96 fragments, one timed
        # pass, no extra local / profile passes
        for _ in range(max(args.warmup, 1)):
            grid.score_fragments(model, images[:96])
    else:
        for _ in range(max(args.warmup, 1)):
            grid.score_fragments(model, images)
    barrier(world)
    clocks = ClockSampler(dev.index or 0)
    clocks.start()
    launches0 = model.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        sim = grid.score_fragments(model, images)
    e1.record()
    torch.cuda.synchronize()
    clock_info = clocks.stop()
    barrier(world)
    launches = model.launch_count() - launches0
    ms = max_over_ranks(e0.elapsed_time(e1) / args.steps, world)
    assert sim.shape == (n, n)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'similarity': sim})
    # each rank's own share without the collective (what limits the curve: the sampler's boundaries balance PAIRS, the
    # per-rank encoder work follows the ROWS)
    l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0.record()
    if not args.lean:
        grid.score_fragments(model, images, gather=False)
    l1.record()
    torch.cuda.synchronize()
    mine = {'rank': rank, 'rows': [int(lo), int(hi)], 'pairs': int(my_pairs),
            'ms_local': l0.elapsed_time(l1) if not args.lean else e0.elapsed_time(e1) / args.steps}
    per_rank = [mine]
    if world > 1:
        import torch.distributed as dist
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
    model.set_option(vited_b200.OPT_PROFILE, 1)
    grid.score_fragments(model, images[:96] if args.lean else images, gather=False)
    prof = model.profile_read()
    model.set_option(vited_b200.OPT_PROFILE, 0)
    total = sum(v['ms'] for v in prof.values()) or 1.0
    flops = n_pairs * 89.50e9 + n * (63.42e9 + 7.248e9 + 0.604e9)
    if rank == 0:
        line = {
            'metric': METRIC, 'value': n_pairs / (ms / 1e3), 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
            'dtype': vited_b200.ACT_NAME, 'data': 'synthetic',
            'config': {'workload': f'configs[3] model (Hisfrag20 patch16 512px, 12+12 layers), {n} synthetic fragments, '
                                   f'{n_pairs} pairs (a<=b), rows sharded x{world} as DistributedIndicatesSampler, '
                                   'through grid.score_fragments (one NCCL all-gather)',
                       'pairs_per_step': n_pairs, 'l2': 'K/V cache of a row block (18.9 MB per fragment) >> 126 MB L2',
                       'lean': bool(args.lean)},
            'clocks': clock_info, 'gpu_launches': int(launches),
            'step_tensor_frac': flops / (ms / 1e3) / 1e12 / (peaks['tf_sustained'] * world),
            'per_rank': per_rank,
            'imbalance': max(r['ms_local'] for r in per_rank) / (sum(r['ms_local'] for r in per_rank) / world),
            'classes_rank0': {k: {'ms': round(v['ms'], 3), 'share': round(v['ms'] / total, 4),
                                  'tflops': round(v['flops'] / max(v['ms'], 1e-9) / 1e9, 1), 'launches': v['launches']}
                              for k, v in sorted(prof.items(), key=lambda kv: -kv[1]['ms'])},
        }
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def run_train(args):
    """Side measurement of BASELINE.json configs[4]: one Hisfrag20 training step (forward with saved activations,
    BCE-with-logits, backward to every parameter, gradient all-reduce) per rank on 24 synthetic 512 px images of 8
    writers (3 per writer as MPerClassSampler(m=3), hisfrag.py:107 -> 24 positive + 48 negative pairs), through
    vited_b200.train.train_step. Reports steps/s and pairs/s over all ranks. The attention forward / backward of this
    path are plain fp32 kernels so far (DESIGN.md), so this is a functional number, not a tuned one."""
    import vited_b200
    from vited_b200 import synthetic, train
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    rank, world, local = dist_setup(args.gpus)
    dev = torch.device('cuda', local if world > 1 else 0)
    model = vited_b200.build_model(vited_b200.get_config('hisfrag'))
    model.load_state_dict(synthetic.synthetic_state_dict(model, seed=0), strict=True)
    model = model.to(dev)
    n_img = args.items if args.items != 512 else 24
    samples, labels = synthetic.synthetic_fragments(n_img // 3, 3, 512, seed=100 + rank)
    samples = samples.to(dev)
    gen = torch.Generator().manual_seed(rank)
    for _ in range(max(args.warmup, 1)):
        loss, logits, groups, _ = train.train_step(model, samples, labels, generator=gen)
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss, logits, groups, pair_labels = train.train_step(model, samples, labels, generator=gen)
    e1.record()
    torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1) / args.steps, world)
    if args.dump_outputs and rank == 0:
        # rank 0's own pairs and logits; the gradients are averaged over the ranks (flattened, named_parameters order)
        dump_outputs(args.dump_outputs, {
            'loss': loss.reshape(1), 'logits': logits, 'groups': groups.double(), 'labels': pair_labels,
            'grads': torch.cat([p.grad.reshape(-1) for p in model.parameters()])})
    gnorm = float(torch.sqrt(sum(p.grad.double().pow(2).sum() for p in model.parameters())))
    train.train_step(model, samples, labels, generator=gen, profile=True)
    prof = model.train_profile
    if rank == 0:
        line = {'metric': 'training steps/sec (Hisfrag20 ViT-ED, fwd + bwd + gradient all-reduce)', 'value': 1e3 / ms,
                'unit': 'steps/s', 'pairs_per_s': world * groups.shape[0] * 1e3 / ms, 'n_gpus': world, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': vited_b200.ACT_NAME, 'data': 'synthetic',
                'config': {'workload': f'configs[4]: Hisfrag20 patch16 512px training step, {n_img} images / GPU -> '
                                       f'{groups.shape[0]} pairs / GPU, DDP-style gradient averaging over {world} GPU(s)'},
                'loss': float(loss), 'grad_norm': gnorm, 'gpu_launches': int(model.train_launches) * args.steps,
                'classes_rank0': prof}
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg (profiling runs)')
    ap.add_argument('--no-extras', action='store_true',
                    help='skip the same-workload N=1 rate and the torch GPU baseline (profiling runs)')
    ap.add_argument('--workload', default='puzzle', choices=['puzzle', 'hisfrag', 'train'],
                    help="'hisfrag' = the Hisfrag20 model (configs[3]) on an all-pairs grid of --items fragments; "
                         "'train' = one Hisfrag20 training step per rank (configs[4])")
    ap.add_argument('--items', type=int, default=512, help='fragments for --workload hisfrag')
    ap.add_argument('--lean', action='store_true',
                    help='--workload hisfrag at full size: warm up on 96 fragments, one timed pass, no local / profile passes '
                         '(ms_local = the rank\'s own timed pass incl. the all-gather, kernel shares from a 96-fragment pass)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the timed path returned in its last timed step as DIR/<name>.npy (float32 / '
                         'float64, %d bytes at most: larger outputs as a fixed seeded sample)' % DUMP_LIMIT)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.warmup < 0:
        ap.error('--warmup must not be negative')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs: the reference arm sizes its sample by the host\'s speed, so its outputs differ from run to run')
    if args.impl == 'reference':
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit('bench.py: no CUDA device; the scoring path has no CPU fallback (use --impl reference)')
        if args.workload == 'hisfrag':
            run_hisfrag(args)
        elif args.workload == 'train':
            run_train(args)
        else:
            run_ours(args)


if __name__ == '__main__':
    main()
