#!/usr/bin/env python
"""bench.py — mesh-tokens/sec of the auto-regressive decode hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--max-new T] [--workload decode|tf|dit|train] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...      (one rank per GPU, replicas)

A "step" is one complete pass of the hot path over one synthetic request of BASELINE.json configs[1]:
ArAE preset, seeded synthetic fp16 weights, one 8192-point cloud, test_num_face=4000, greedy,
max_new_tokens=16000 (seq_len ~ 18k): point encoder -> 2050-row prefill -> 16000-token decode (one persistent
kernel) [-> detokenize in the e2e leg].  Decode shards as independent replicas (generate asserts B == 1,
core/models.py:215): N GPUs = N requests, no collective on the data path; "scaling": "weak".

Output: ONE JSON line on rank 0 (see the task contract): value = whole-job tokens/s with inputs resident in HBM,
e2e = the same through LMM.generate with host buffers (H2D of the cloud and D2H of the ids inside the timed region),
roofline = algorithmic HBM bytes of the decode kernel / its CUDA-event duration vs MEASURED_PEAKS.json,
cpu_baseline = the REFERENCE's own modules (oracle/_ref/py, copied by `make -C oracle refpy`; kind "reference") on this box's host
cores on a bounded sample (cached decode steps at three context lengths, extrapolated to the 16k request with t(L) = a + bL); if
that copy is absent, the CPU oracle port (kind "port").  reference_gpu = the same modules on the GPU exactly as infer.py runs them
(model.half() + autocast(fp16) + flash-attn), the ">= 10x" denominator.  `--impl reference` prints the CPU reference arm alone.
"""

import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

METRIC = 'mesh-tokens/sec at 4k-face greedy decode'
UNIT = 'tokens/s'


def workload(args):
    from dataclasses import replace
    from core.options import config_defaults
    from edgerunner_b200 import synth
    if args.tiny:
        opt = synth.tiny_options()
        return opt, 'tiny-debug', min(args.max_new, 400), 1000
    opt = replace(config_defaults['ArAE'], generate_mode='greedy')
    return opt, 'ArAE greedy decode test_num_face=4000 max_new_tokens=%d batch=1 (BASELINE configs[1])' % args.max_new, args.max_new, 4000


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q, '--format=csv,noheader,nounits', '-lms', '200'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)                     # no sampler left running if the benchmark fails before stop()
            self.thread = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for l in self.lines:
            f = [x.strip() for x in l.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """--dump-outputs: what the timed path returned in its last step, one <path>/<name>.npy per array in float64.  An array larger than its
    share of DUMP_BYTES is replaced by a fixed, seeded sample of its flattened elements, and <name>_index.npy holds their flat indices.
    The inputs are seeded, so two builds run with the same arguments can be compared file by file."""
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // (2 * len(arrays))
    for name, a in arrays.items():
        a = torch.as_tensor(a).detach()
        if a.numel() * 8 > share:                           # sampled where the array lives: no float64 copy of it on the host
            idx = np.sort(np.random.default_rng(0).choice(a.numel(), share // 8, replace=False))
            np.save(os.path.join(path, name + '_index.npy'), idx.astype(np.float64))
            a = a.reshape(-1)[torch.from_numpy(idx).to(a.device)]
        np.save(os.path.join(path, name + '.npy'), a.cpu().numpy().astype(np.float64))


def algorithmic_decode_bytes(eng, L0, T):
    """SURVEY.md §8(d): per generated token bytes(L) = W + kv_row * L (KV read) + kv_row (KV write); the kernel runs T-1
    forward passes for T sampled tokens (the last token needs none), at cache lengths L0 .. L0+T-2."""
    W, kv = eng.weight_bytes_per_token(), eng.kv_bytes_per_row()
    n = T - 1
    return n * (W + kv) + kv * (n * L0 + n * (n - 1) // 2)


def pick_threads(step_fn, candidates):
    """The CPU port is a chain of small GEMVs: more threads is not faster.  Time a few steps per candidate, keep the best."""
    best, best_t = candidates[0], float('inf')
    for n in candidates:
        torch.set_num_threads(n)
        step_fn()
        t0 = time.perf_counter()
        step_fn(); step_fn()
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def thread_candidates():
    n = os.cpu_count() or 1
    return sorted({c for c in (4, 8, 16, 32, 64, n) if c <= n})


def ref_leg(kind, steps, warmup, tokens, tiny=False, timeout=900):
    """Run oracle/ref_leg.py (the reference's own modules) in its own process -> dict | None.  Its package is called `core` like this
    repository's drop-in mirror, so it cannot share a process with the product path."""
    script = os.path.join(REPO, 'oracle', 'ref_leg.py')
    if not os.path.isdir(os.path.join(REPO, 'oracle', '_ref', 'py', 'core')):
        return None
    cmd = [sys.executable, script, kind, '--steps', str(steps), '--warmup', str(warmup), '--tokens', str(tokens)] + (['--tiny'] if tiny else [])
    env = dict(os.environ)
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK', 'MASTER_ADDR', 'MASTER_PORT', 'TORCHELASTIC_RUN_ID'):
        env.pop(k, None)
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
    except subprocess.TimeoutExpired:
        return {'error': f'reference {kind} leg timed out after {timeout}s'}
    for line in out.stdout.splitlines():
        if line.startswith('REF_LEG '):
            return json.loads(line[8:])
    return {'error': (out.stderr or out.stdout)[-400:]}


def cpu_port_tokens_per_s(opt, seconds_budget, threads):
    """Fallback when oracle/_ref/py is absent: the CPU oracle (fp32 port of the reference's CPU path) on a bounded sample."""
    from edgerunner_b200 import synth
    from oracle.er_oracle import Oracle     # bench.py's cpu_baseline leg is allowed to execute the oracle
    torch.set_num_threads(min(threads, 32))
    sd = synth.synth_state_dict(opt, seed=0, eos_logit=-30.0)
    orc = Oracle(opt, sd, mode='fp32')
    del sd
    cond = synth.synth_point_cloud(0, opt.point_num)
    ce = orc.encode_cond(cond, 4000)[0]
    n_max = 256 + 32
    orc.reset_cache(ce.shape[0] + 1 + n_max + 1)
    orc.prefill(ce, [opt.bos_token_id])
    state = {'tok': 5}

    def one():
        pre = orc.step(state['tok'])
        state['tok'] = 6 + int(torch.argmax(pre[0, 6:]))
    threads = pick_threads(one, thread_candidates())
    L0 = orc.L
    tok, n, t0 = state['tok'], 0, time.perf_counter()
    while n < n_max and (time.perf_counter() - t0 < seconds_budget or n < 8):
        pre = orc.step(tok)
        tok = 6 + int(torch.argmax(pre[0, 6:]))
        n += 1
    dt = time.perf_counter() - t0
    return n / dt, threads, f'{n} greedy decode steps from a prefilled cache at L={L0}..{L0 + n} (fp32, torch CPU ops, {threads} threads); ' \
                   f'prefill/encoder excluded; short-L sample flatters the CPU'


def cpu_baseline_leg(args, opt, steps=1, warmup=1):
    """-> the `cpu_baseline` object: the reference's own CPU path when its copy travelled to this box, else the oracle port."""
    r = ref_leg('cpu', steps, warmup, tokens=2 if not args.tiny else 4, tiny=args.tiny)
    if r is not None and 'error' not in r:
        return {'value': r['tok_s'], 'unit': UNIT, 'cores': r['threads'], 'kind': 'reference', 'sample': r['sample'] + f"; {r['path']}; "
                f"{r['threads']} of {r['host_threads']} host threads; per-window tokens/s {r['windows_tok_s']}; {r['model']}",
                'extrapolated_request_s': r['extrapolated_request_s'], 'sample_s_per_step': r['sample_s_per_step'], 'windows_tok_s': r['windows_tok_s']}
    threads = os.cpu_count() or 1
    v, used, sample = cpu_port_tokens_per_s(opt, 15.0, threads)
    why = 'oracle/_ref/py absent' if r is None else 'reference leg failed: ' + r['error']
    return {'value': v, 'unit': UNIT, 'cores': used, 'kind': 'port', 'sample': sample + f' ({why}; thread count picked from {thread_candidates()} of {threads} host threads)'}


def run_reference_arm(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the host cores (oracle/_ref/py when it travelled with
    the snapshot, else the oracle port), same metric / unit / config as our arm.  Each step = one bounded sample of the 16k request
    (see oracle/ref_leg.py); value = 16000 tokens / the extrapolated request time.  Rank 0 alone runs it (the host cores are shared by
    all replicas: CPU throughput does not grow with --gpus)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    opt, wl, T, nf = workload(args)
    cb = cpu_baseline_leg(args, opt, steps=args.steps, warmup=args.warmup)
    v = cb['value']
    ms = cb.get('sample_s_per_step', 0.0) * 1e3
    emit(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic', 'config': {'workload': wl, 'tokens_per_step_per_gpu': T, 'prefix_rows': opt.num_cond_tokens + 1,
                                        'sample': cb['sample'], 'note': 'ms_per_step is the measured bounded sample; value extrapolates it to the full request; '
                                        'the host cores are shared by all replicas, so the CPU arm does not scale with --gpus'},
        'cpu_baseline': cb,
        'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }), flush=True)


def run_teacher_forced(args):
    """BASELINE configs[3]: ArAE teacher-forced forward, seq_len 8192 (+ 2049 condition rows + BOS/EOS = 10 243 rows), batch 4 per GPU, data
    parallel: every rank runs the forward on its own batch through LMM.forward, ONE NCCL all-reduce of the fp64 {ce_sum, n_tokens, kl}.  Forward
    only (the full training step is `--workload train`).  value = supervised tokens/s over all ranks; roofline: tensor-bound, algorithmic FLOPs (SURVEY §8d)
    against MEASURED_PEAKS bf16_tflops_sustained."""
    rank = int(os.environ.get('RANK', '0')); world = int(os.environ.get('WORLD_SIZE', '1')); local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    from dataclasses import replace
    from core.models import LMM
    from core.options import config_defaults
    from edgerunner_b200 import synth
    opt = replace(config_defaults['ArAE'], generate_mode='greedy') if not args.tiny else synth.tiny_options()
    B, T = 4, (8194 if not args.tiny else 48)
    P, C, NL = opt.num_cond_tokens, opt.hidden_dim, opt.num_layers
    N = P + T
    sd = synth.synth_state_dict(opt, seed=0, eos_logit=-30.0, dtype=torch.float16)
    with torch.device('meta'):
        model = LMM(opt)
    model.load_state_dict(sd, strict=True, assign=True)
    del sd
    model = model.half().eval().to(dev)
    g = torch.Generator().manual_seed(100 + rank)
    tokens = torch.randint(6, model.vocab_size, (B, T), generator=g)
    tokens[:, 0] = opt.bos_token_id
    data = {'conds': torch.cat([synth.synth_point_cloud(rank * B + b, opt.point_num) for b in range(B)]).to(dev), 'tokens': tokens,
            'labels': torch.cat([torch.full((B, P), -100, dtype=torch.long), tokens.long()], dim=1), 'masks': torch.ones((B, N), dtype=torch.bool),
            'num_faces': torch.tensor([4000] * B), 'num_tokens': torch.full((B,), T)}

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()
    # SURVEY §8e / BASELINE configs[3] "grad all-reduce": the flattened fp32 gradient buffer of the model's parameter count, all-reduced over
    # NCCL in 4 reverse-order slices per step, launched before the forward so that it overlaps it.  SYNTHETIC gradients: this workload is forward only
    # (`--workload train` all-reduces the real ones).
    fg = None
    comm_ms = None
    if args.grad_allreduce and world > 1:
        from edgerunner_b200.dist import FlatGradAllReduce
        n_params = sum(p.numel() for p in model.parameters())
        fg = FlatGradAllReduce(n_params, dev, n_slices=4)
        for _ in range(2):
            fg.launch().wait()
        barrier()
        ce = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ce[0].record()
        for _ in range(3):
            fg.launch().wait()
        ce[1].record()
        barrier()
        comm_ms = ce[0].elapsed_time(ce[1]) / 3
    for _ in range(max(args.warmup, 1)):
        if fg:
            fg.launch()
        out = model(data)
        if fg:
            fg.wait()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    l0 = model._engine.kernel_launches()
    ev[0].record()
    for _ in range(args.steps):
        if fg:
            fg.launch()
        out = model(data)
        loss = float(out['loss'])                          # D2H of the step's result
        if fg:
            fg.wait()
    ev[1].record()
    barrier()
    ms = ev[0].elapsed_time(ev[1])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms, comm_ms or 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0].item())
        comm_ms = float(t[1].item()) if fg else None
        dist.destroy_process_group()
    clocks = sampler.stop() if rank == 0 else None
    if rank != 0:
        return
    ms_step = ms / args.steps
    flops = (2 * 680_752_128 * B * N + 2 * N * N * C * NL * B + 0.16e12 * B) if not args.tiny else float('nan')
    peaks_path = os.path.join(REPO, 'MEASURED_PEAKS.json')
    peak = float(json.load(open(peaks_path)).get('bf16_tflops_sustained', 1400.0)) if os.path.exists(peaks_path) else 1400.0
    tf = flops / (ms_step * 1e-3) / 1e12
    emit(json.dumps({
        'metric': 'teacher-forced tokens/sec, ArAE forward seq_len 8192 batch 4/GPU (BASELINE configs[3], forward only)', 'value': world * B * T / (ms_step * 1e-3),
        'unit': 'tokens/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f16', 'data': 'synthetic', 'loss': loss,
        'config': {'workload': f'ArAE teacher-forced forward B={B}/GPU N={N} (P={P} + T={T}), data parallel x{world}, one NCCL all-reduce of 3 fp64 numbers per step',
                   'backward': 'none (forward only)', 'l2': f'activations of {B * N} rows x 1536 exceed L2'},
        'clocks': clocks, 'gpu_launches': int(model._engine.kernel_launches() - l0),
        'roofline': {'bound': 'tensor', 'achieved': tf, 'peak': peak, 'unit': 'TFLOP/s', 'frac': tf / peak, 'traffic': None,
                     'kernel': 'er::tc::gemm_tcgen05_kernel + er::fa::attention_tcgen05_kernel', 'algorithmic_flops_per_step_per_gpu': flops,
                     'peak_source': 'MEASURED_PEAKS.json bf16_tflops_sustained (of measured)'},
        'e2e': {'value': world * B * T / (ms_step * 1e-3), 'unit': 'tokens/s', 'h2d_bytes_per_step': int(tokens.numel() * 4 + data['labels'].numel() * 8),
                'd2h_bytes_per_step': 4, 'note': 'LMM.forward(data): tokens / labels uploaded and the loss read back every step inside the timed region'},
        'comm': None if not fg else {
            'grad_allreduce': 'flattened fp32 buffer of %d elements (%.2f GB), NCCL all-reduce in 4 reverse-order slices per step, overlapped with the forward; '
                              'SYNTHETIC gradients (forward-only workload; --workload train all-reduces real ones)' % (fg.buf.numel(), fg.buf.numel() * 4 / 1e9),
            'standalone_ms': comm_ms, 'busbw_GBps': (fg.buf.numel() * 4 * 2 * (world - 1) / world) / (comm_ms * 1e-3) / 1e9 if comm_ms else None,
            'ms_per_step_includes_it': True},
    }), flush=True)


def run_train(args):
    """BASELINE configs[3] as a FULL training step (SURVEY §8 f2): ArAE, seq_len 8192 (+ 2049 condition rows + BOS/EOS = 10 243 rows), batch 4 per GPU,
    data parallel.  A step = edgerunner_b200.train.FlatTrainer.step: training-mode forward (dropout 0.1) + backward with per-layer recomputation
    (opt.checkpointing) + flat fp32 gradient all-reduce over NCCL + global-norm clipping + fused AdamW + fp16 weight refresh; tokens / labels are
    uploaded and the loss is read back every step.  All 766.8 M parameters are trained as in the ArAE preset (--freeze-encoder: the point encoder and the
    KL term are constants).  value = supervised tokens/s over all ranks;
    roofline: tensor-bound, MODEL FLOPs (forward + 2 x GEMM + 2.5 x attention; the recomputation is not counted) against bf16_tflops_sustained."""
    rank = int(os.environ.get('RANK', '0')); world = int(os.environ.get('WORLD_SIZE', '1')); local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    from dataclasses import replace
    from core.models import LMM
    from core.options import config_defaults
    from edgerunner_b200 import synth
    from edgerunner_b200.train import FlatTrainer
    # the ArAE preset trains the point encoder too (options.py:167 freeze_encoder=False); --freeze-encoder = the Options default instead
    fz = bool(args.freeze_encoder)
    opt = replace(config_defaults['ArAE'], generate_mode='greedy', freeze_encoder=fz) if not args.tiny else synth.tiny_options(freeze_encoder=fz)
    B, T = (4, 8194) if not args.tiny else (2, 48)
    P, C, NL = opt.num_cond_tokens, opt.hidden_dim, opt.num_layers
    N = P + T
    sd = synth.synth_state_dict(opt, seed=0, eos_logit=-30.0, dtype=torch.float16)
    with torch.device('meta'):
        model = LMM(opt)
    model.load_state_dict(sd, strict=True, assign=True)
    del sd
    model = model.half().train().to(dev)
    g = torch.Generator().manual_seed(100 + rank)
    tokens = torch.randint(6, model.vocab_size, (B, T), generator=g)
    tokens[:, 0] = opt.bos_token_id
    data = {'conds': torch.cat([synth.synth_point_cloud(rank * B + b, opt.point_num) for b in range(B)]).to(dev), 'tokens': tokens.pin_memory(),
            'labels': torch.cat([torch.full((B, P), -100, dtype=torch.long), tokens.long()], dim=1).pin_memory(), 'masks': None,
            'num_faces': torch.tensor([4000] * B)}
    tr = FlatTrainer(model, total_steps=1000, max_batch=B, max_tokens=T)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()
    hist = []
    for _ in range(max(args.warmup, 1)):
        hist.append(float(tr.step(data)['loss']))
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    l0 = tr.engine.kernel_launches()
    ev[0].record()
    for _ in range(args.steps):
        out = tr.step(data)
        hist.append(float(out['loss']))                       # D2H of the step's result
    ev[1].record()
    barrier()
    ms = ev[0].elapsed_time(ev[1])
    if args.dump_outputs and rank == 0:
        # the step's losses and gradient norm, and the updated fp32 parameters it leaves in the trainer
        dump_outputs(args.dump_outputs, {**{k: out[k] for k in ('loss', 'loss_ce', 'loss_kl', 'grad_norm')}, 'parameters': tr.param})
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0].item())
        dist.destroy_process_group()
    clocks = sampler.stop() if rank == 0 else None
    if rank != 0:
        return
    ms_step = ms / args.steps
    gemm_f, attn_f = 2 * 680_752_128 * B * N, 2 * N * N * C * NL * B
    flops = (3 * gemm_f + 3.5 * attn_f + (1 if fz else 3) * 0.16e12 * B) if not args.tiny else float('nan')
    peaks_path = os.path.join(REPO, 'MEASURED_PEAKS.json')
    peak = float(json.load(open(peaks_path)).get('bf16_tflops_sustained', 1400.0)) if os.path.exists(peaks_path) else 1400.0
    tf = flops / (ms_step * 1e-3) / 1e12
    line = {
        'metric': 'training tokens/sec, ArAE full step seq_len 8192 batch 4/GPU (BASELINE configs[3]; ' + ('decoder trained, point encoder frozen)' if fz else 'all parameters trained)'),
        'value': world * B * T / (ms_step * 1e-3), 'unit': 'tokens/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_step,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f16', 'data': 'synthetic', 'loss_history': hist,
        'config': {'workload': f'ArAE training step B={B}/GPU N={N} (P={P} + T={T}): training forward (dropout {tr.dropout_p}) + backward (activations kept in HBM unless '
                               f'--debug train_recompute=1) + flat gradient all-reduce x{world} + clip + fused AdamW + fp16 weight refresh',
                   'trainable_parameters': int(tr.numel), 'debug': args.debug, 'l2': f'activations of {B * N} rows x 1536 exceed L2'},
        'clocks': clocks, 'gpu_launches': int(tr.engine.kernel_launches() - l0),
        'roofline': {'bound': 'tensor', 'achieved': tf, 'peak': peak, 'unit': 'TFLOP/s', 'frac': tf / peak, 'traffic': None,
                     'kernel': 'er::tc::gemm_tcgen05_kernel (forward, dgrad, wgrad) + er::fa::attention_tcgen05_kernel + er::bwm::dq_kernel / dkv_kernel (mma.sync)',
                     'algorithmic_flops_per_step_per_gpu': flops, 'note': 'model FLOPs: 3 x GEMM + 3.5 x causal attention of the forward; the 1.4 x redundant score products of the two-kernel attention '
                     'backward (and the recomputed forward in --debug train_recompute=1 mode) are not counted',
                     'peak_source': 'MEASURED_PEAKS.json bf16_tflops_sustained (of measured)'},
        'e2e': {'value': world * B * T / (ms_step * 1e-3), 'unit': 'tokens/s', 'h2d_bytes_per_step': int(tokens.numel() * 4 + data['labels'].numel() * 8),
                'd2h_bytes_per_step': 4, 'note': 'FlatTrainer.step(data): tokens / labels uploaded from pinned host memory, loss read back, every step'},
    }
    value = line['value']
    if world == 1 and not args.tiny:
        del tr, model
        torch.cuda.empty_cache()
        if not args.no_reference_gpu:
            rg = ref_train_leg('gpu', 2, 1, timeout=900)
            line['reference_gpu'] = ({'value': rg['tok_s'], 'unit': 'tokens/s', 'kind': 'reference', 'path': rg['path'], 'sample': rg['sample'], 's_per_step': rg['s_per_step_sample'],
                                      'ours_over_reference_gpu': value / rg['tok_s']} if rg and 'tok_s' in rg else
                                     {'unavailable': 'oracle/_ref/py absent' if rg is None else rg.get('error', 'failed')})
        if not args.no_cpu_baseline:
            rc = ref_train_leg('cpu', 1, 0, timeout=1500)
            line['cpu_baseline'] = ({'value': rc['tok_s'], 'unit': 'tokens/s', 'cores': rc['threads'], 'kind': 'reference', 'sample': rc['sample'] + '; ' + rc['path'],
                                     'sample_s_per_step': rc['s_per_step_sample'], 'extrapolated_step_s': rc['extrapolated_c4_step_s']} if rc and 'tok_s' in rc else
                                    {'unavailable': 'oracle/_ref/py absent' if rc is None else rc.get('error', 'failed')})
    emit(json.dumps(line), flush=True)


def ref_train_leg(kind, steps, warmup, tiny=False, timeout=900):
    """oracle/ref_train_leg.py in its own process -> dict | None: the reference's OWN training step (torch autograd over its modules, clip, AdamW) on the
    host cores (bounded sample, extrapolated by model FLOPs) or on the GPU (bf16 autocast + flash-attn at the configs[3] shape)."""
    if not os.path.isdir(os.path.join(REPO, 'oracle', '_ref', 'py', 'core')):
        return None
    cmd = [sys.executable, os.path.join(REPO, 'oracle', 'ref_train_leg.py'), kind, '--steps', str(steps), '--warmup', str(warmup)] + (['--tiny'] if tiny else [])
    env = dict(os.environ)
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK', 'MASTER_ADDR', 'MASTER_PORT', 'TORCHELASTIC_RUN_ID'):
        env.pop(k, None)
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
    except subprocess.TimeoutExpired:
        return {'error': f'reference training {kind} leg timed out after {timeout}s'}
    for line in out.stdout.splitlines():
        if line.startswith('REF_TRAIN_LEG '):
            return json.loads(line[14:])
    return {'error': (out.stderr or out.stdout)[-400:]}


def ref_dit_leg(kind, images, steps, warmup, layers=24, timeout=900):
    """oracle/ref_dit_leg.py in its own process -> dict (reference DiT module when oracle/_ref/py travelled, else the oracle port)."""
    cmd = [sys.executable, os.path.join(REPO, 'oracle', 'ref_dit_leg.py'), kind, '--images', str(images), '--steps', str(steps), '--warmup', str(warmup),
           '--layers', str(layers)]
    env = dict(os.environ)
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK', 'MASTER_ADDR', 'MASTER_PORT', 'TORCHELASTIC_RUN_ID'):
        env.pop(k, None)
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
    except subprocess.TimeoutExpired:
        return {'error': f'reference DiT {kind} leg timed out after {timeout}s'}
    for line in out.stdout.splitlines():
        if line.startswith('REF_DIT_LEG '):
            return json.loads(line[12:])
    return {'error': (out.stderr or out.stdout)[-400:]}


DIT_METRIC = 'DiT denoiser steps/sec, guided DDIM sampling of 4 images (denoiser batch 8 x 2048 latents, 24 layers; BASELINE configs[4] denoise stage)'


def run_dit(args):
    """BASELINE configs[4], the stage this repository adds to the image-conditioned path: MDiT.run — 100 guided DDIM steps for a batch of 4
    images (denoiser batch 8) at the DiT preset size.  A bench step = one whole sampling run.  value = denoiser steps/s over all ranks
    (replicas: every rank samples its own 4 images); roofline: tensor-bound, GEMM + attention FLOPs of the denoiser forward against
    MEASURED_PEAKS bf16_tflops_sustained; e2e: er_dit_run_host (condition + noise uploaded, latents read back every step)."""
    rank = int(os.environ.get('RANK', '0')); world = int(os.environ.get('WORLD_SIZE', '1')); local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    import numpy as np
    from core.models_dit import DDIMScheduler
    from edgerunner_b200 import synth
    from edgerunner_b200.dit_engine import DiTEngine
    R, S, M = 4, 100, 257
    cfg = dict(hidden_dim=1024, num_heads=16, latent_size=2048, latent_dim=64, num_layers=24) if not args.tiny else \
        dict(hidden_dim=128, num_heads=2, latent_size=64, latent_dim=16, num_layers=2)
    eng = DiTEngine(dev, cfg['hidden_dim'], cfg['num_heads'], cfg['num_layers'], cfg['latent_size'], cfg['latent_dim'], M, 1280)
    eng.load_state_dict(synth.synth_dit_state_dict(**cfg, cond_dim=1280, seed=0))
    sched = DDIMScheduler(prediction_type='v_prediction')
    sched.set_timesteps(S)
    ts = sched.timesteps.numpy().astype(np.float32)
    coef = sched.step_coefficients(sched.timesteps).numpy()
    g = torch.Generator().manual_seed(200 + rank)
    cond_h = torch.randn(R, M, cfg['hidden_dim'], generator=g).pin_memory()
    noise_h = torch.randn(R, cfg['latent_size'], cfg['latent_dim'], generator=g).pin_memory()
    cond_d, noise_d = cond_h.to(dev), noise_h.to(dev)
    lat = torch.empty_like(noise_d)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def one():
        lat.copy_(noise_d)
        eng.run(cond_d, lat, ts, coef, 7.5, True, 'v_prediction')
    for _ in range(max(args.warmup, 1)):
        one()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    l0 = eng.kernel_launches()
    ev[0].record()
    for _ in range(args.steps):
        one()
    ev[1].record()
    barrier()
    launches = eng.kernel_launches() - l0
    ms = ev[0].elapsed_time(ev[1])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'latents': lat})
    # e2e: host buffers through the C ABI
    lat_h = np.empty_like(noise_h.numpy())
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    np.copyto(lat_h, noise_h.numpy()); eng.run_host(cond_h.numpy(), lat_h, ts, coef, 7.5, True, 'v_prediction')
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        np.copyto(lat_h, noise_h.numpy())
        eng.run_host(cond_h.numpy(), lat_h, ts, coef, 7.5, True, 'v_prediction')
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    finite = bool(np.isfinite(lat_h).all())
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms, e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_s = float(t[0].item()), float(t[1].item())
        dist.destroy_process_group()
    clocks = sampler.stop() if rank == 0 else None
    if rank != 0:
        return
    ms_step = ms / args.steps
    flops = eng.flops_per_forward(2 * R) * S
    peaks_path = os.path.join(REPO, 'MEASURED_PEAKS.json')
    peak = float(json.load(open(peaks_path)).get('bf16_tflops_sustained', 1400.0)) if os.path.exists(peaks_path) else 1400.0
    tf = flops / (ms_step * 1e-3) / 1e12
    line = {
        'metric': DIT_METRIC, 'value': world * S / (ms_step * 1e-3), 'unit': 'denoiser steps/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f16', 'data': 'synthetic',
        'config': {'workload': f'MDiT.run: {S} guided DDIM steps (v_prediction, guidance 7.5), {R} images/GPU -> denoiser batch {2 * R} x {cfg["latent_size"]} latents, '
                               f'{cfg["num_layers"]} layers x {cfg["hidden_dim"]}, {M} condition tokens; replicas x{world}',
                   'l2': 'activations (16384 rows x 1024..8192 fp16, 33..268 MB per tensor) exceed L2', 'latents_finite': finite},
        'clocks': clocks, 'gpu_launches': int(launches),
        'roofline': {'bound': 'tensor', 'achieved': tf, 'peak': peak, 'unit': 'TFLOP/s', 'frac': tf / peak, 'traffic': None,
                     'kernel': 'er::tc::gemm_tcgen05_kernel + er::fa::attention_tcgen05_kernel (inside one CUDA graph per step)',
                     'algorithmic_flops_per_step_per_gpu': flops, 'peak_source': 'MEASURED_PEAKS.json bf16_tflops_sustained (of measured)'},
        'e2e': {'value': world * S / e2e_s, 'unit': 'denoiser steps/s', 'h2d_bytes_per_step': int(cond_h.numel() * 4 + noise_h.numel() * 4),
                'd2h_bytes_per_step': int(noise_h.numel() * 4), 'note': 'er_dit_run_host: condition + noise uploaded, latents read back, synchronous'},
    }
    if not args.no_reference_gpu and not args.tiny:
        rg = ref_dit_leg('gpu', R, 3, 2)
        if rg and 's_per_forward' in rg:
            line['reference_gpu'] = {'value': 1.0 / rg['s_per_forward'], 'unit': 'denoiser steps/s', 'impl': rg.get('impl'), 'flash_attn': rg.get('flash_attn'),
                                     'sample': f"{rg['impl']} DiT module, .half() + autocast(fp16), denoiser batch {rg['batch']}, forward only (no scheduler / guidance)"}
        else:
            line['reference_gpu'] = rg
    if args.dit_pipeline and not args.tiny:
        line['pipeline'] = dit_pipeline_leg(dev)
    if not args.no_cpu_baseline and not args.tiny:
        rc = ref_dit_leg('cpu', 1, 1, 1)
        if rc and 's_per_forward' in rc:
            line['cpu_baseline'] = {'value': 1.0 / (rc['s_per_forward'] * R), 'unit': 'denoiser steps/s', 'cores': rc.get('cores'), 'kind': rc.get('impl'),
                                    'sample': f"1 denoiser forward of 1 image (batch 2), fp32 torch CPU ops, scaled x{R} to the 4-image step"}
        else:
            line['cpu_baseline'] = rc
    emit(json.dumps(line), flush=True)


def dit_pipeline_leg(dev):
    """BASELINE configs[4] end to end for ONE image at the preset sizes, through the public classes exactly as infer_dit.py:104-113 drives them:
    MDiT.run(image) [CLIP ViT-H/14 tower (library model, random weights) -> adaptor -> 100 guided DDIM steps] -> LMM.generate(latents,
    num_faces=4000, 16 000 new tokens, greedy) -> detokenise + clean.  Wall-clock seconds per stage (host-timed, synchronised)."""
    from dataclasses import replace
    from core.models import LMM
    from core.models_dit import MDiT
    from core.options import config_defaults
    from core.utils import get_tokenizer
    from edgerunner_b200 import synth
    opt = replace(config_defaults['DiT'], generate_mode='greedy')
    sd = synth.synth_state_dict(opt, seed=0, eos_logit=-30.0, dtype=torch.float16)
    with torch.device('meta'):
        lmm = LMM(opt)
    lmm.load_state_dict(sd, strict=True, assign=True)
    del sd
    lmm = lmm.half().eval().to(dev)
    opt.cond_mode = 'point_latent'                                   # infer_dit.py:55
    torch.manual_seed(0)
    mdit = MDiT(opt)
    mdit.load_state_dict(synth.synth_dit_state_dict(opt.dit_hidden_dim, opt.dit_num_heads, opt.point_latent_size, opt.point_latent_dim, opt.dit_num_layers,
                                                    cond_dim=1280, seed=0), strict=False)
    mdit = mdit.half().eval().to(dev)
    tok, _ = get_tokenizer(opt)
    img = torch.rand(1, 3, 512, 512, generator=torch.Generator().manual_seed(3)).to(dev)
    out = {}
    for rep in range(2):                                             # first pass warms up (engine creation, graph capture)
        torch.cuda.synchronize(); t0 = time.perf_counter()
        lat = mdit.run(img)
        torch.cuda.synchronize(); t1 = time.perf_counter()
        meshes, tokens = lmm.generate(lat, num_faces=4000, max_new_tokens=16000, tokenizer=tok, clean=True)
        torch.cuda.synchronize(); t2 = time.perf_counter()
        out = {'image_to_latents_s': t1 - t0, 'latents_to_mesh_s': t2 - t1, 'total_s': t2 - t0, 'new_tokens': int(len(tokens[0])), 'faces': int(len(meshes[0].faces)),
               'stages': 'MDiT.run (CLIP ViT-H/14 + adaptor + 100 guided DDIM steps, 1 image) | LMM.generate(point_latent, 4000 faces, 16000 tokens, greedy) + detokenise + clean'}
    return out


def run_dit_reference_arm(args):
    """`--impl reference --workload dit`: the reference's DiT module on the host cores (fp32, naive attention), bounded sample = one denoiser
    forward of one image (batch 2) per step, scaled to the 4-image step."""
    if int(os.environ.get('RANK', '0')) != 0:
        return
    R = 4
    rc = ref_dit_leg('cpu', 1, max(args.steps, 1), min(args.warmup, 1), timeout=1500)
    if not rc or 's_per_forward' not in rc:
        emit(json.dumps({'impl': 'reference', 'unavailable': str(rc)[:200]}), flush=True)
        return
    v = 1.0 / (rc['s_per_forward'] * R)
    cb = {'value': v, 'unit': 'denoiser steps/s', 'cores': rc.get('cores'), 'kind': rc.get('impl'),
          'sample': f"{args.steps} x one denoiser forward of 1 image (batch 2), fp32 torch CPU ops, scaled x{R} to the 4-image step"}
    emit(json.dumps({'impl': 'reference', 'metric': DIT_METRIC, 'value': v, 'unit': 'denoiser steps/s', 'n_gpus': args.gpus, 'steps': args.steps,
                      'warmup': args.warmup, 'ms_per_step': rc['s_per_forward'] * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                      'dtype': 'f32', 'data': 'synthetic', 'config': {'workload': 'reference DiT module forward, CPU', 'sample': cb['sample']},
                      'cpu_baseline': cb, 'e2e': {'value': v, 'unit': 'denoiser steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}), flush=True)


def run_train_reference_arm(args):
    """`--impl reference --workload train`: the reference's own training step on the host cores (oracle/ref_train_leg.py cpu): every bench step = one
    bounded sample (one sample of 128 tokens + 2049 condition rows through forward, backward, clip, AdamW), extrapolated to the configs[3] step by
    model FLOPs.  Rank 0 only."""
    if int(os.environ.get('RANK', '0')) != 0:
        return
    rc = ref_train_leg('cpu', max(args.steps, 1), min(args.warmup, 1), tiny=args.tiny, timeout=3000)
    if not rc or 'tok_s' not in rc:
        emit(json.dumps({'impl': 'reference', 'unavailable': str(rc)[:200]}), flush=True)
        return
    cb = {'value': rc['tok_s'], 'unit': 'tokens/s', 'cores': rc['threads'], 'kind': 'reference', 'sample': rc['sample'] + '; ' + rc['path']}
    emit(json.dumps({'impl': 'reference', 'metric': 'training tokens/sec, ArAE full step seq_len 8192 batch 4/GPU (BASELINE configs[3]; all parameters trained)',
                      'value': rc['tok_s'], 'unit': 'tokens/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
                      'ms_per_step': rc['s_per_step_sample'] * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
                      'data': 'synthetic', 'config': {'workload': 'reference LMM training step, CPU', 'sample': cb['sample'],
                                                      'note': 'ms_per_step is the measured bounded sample; value extrapolates it to the configs[3] step'},
                      'cpu_baseline': cb, 'e2e': {'value': rc['tok_s'], 'unit': 'tokens/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}), flush=True)


_STDOUT_FD = None


def emit(line, flush=True):
    """the bench line, on the process's ORIGINAL stdout (see main())"""
    if _STDOUT_FD is None:
        print(line, flush=True)
    else:
        os.write(_STDOUT_FD, (line + '\n').encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=2)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours')
    ap.add_argument('--max-new', type=int, default=16000)
    ap.add_argument('--tokens-per-launch', type=int, default=0)
    ap.add_argument('--tiny', action='store_true', help='debug: tiny model')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-reference-gpu', action='store_true')
    ap.add_argument('--e2e-steps', type=int, default=3, help='timed LMM.generate calls of the e2e leg (bounded: each is a full 16k request)')
    ap.add_argument('--grad-allreduce', action='store_true', help='--workload tf under torchrun: also all-reduce a flattened synthetic gradient buffer every step (SURVEY 8e)')
    ap.add_argument('--dit-pipeline', action='store_true', help='--workload dit: also time one image end to end (MDiT.run -> LMM.generate) at the preset sizes')
    ap.add_argument('--workload', default='decode', choices=['decode', 'tf', 'dit', 'train'],
                    help="decode = BASELINE configs[1] (the metric); tf = configs[3]: teacher-forced forward seq 8192 batch 4/GPU, loss all-reduced over NCCL")
    ap.add_argument('--freeze-encoder', action='store_true', help='--workload train: opt.freeze_encoder = True (the Options default) instead of the ArAE preset (encoder trained)')
    ap.add_argument('--debug', action='append', default=[], metavar='KEY=VALUE', help='process-wide experiment switch of the library (er_debug_set(NULL, KEY, VALUE)), e.g. attn_bwd_wmma=1')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps, write what the last one computed to DIR/<name>.npy (float64, '
                    'at most 64 MB in all; seeded inputs, so two builds can be compared output for output)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs records the CUDA path; the reference arm has none')
    # stdout carries exactly ONE JSON line: whatever libraries print there (NCCL's version banner under torchrun) is sent to stderr instead
    global _STDOUT_FD
    sys.stdout.flush()
    _STDOUT_FD = os.dup(1)
    os.dup2(2, 1)

    for kv in args.debug:
        from edgerunner_b200 import _lib
        k, v = kv.split('=')
        _lib.check(_lib.load().er_debug_set(None, k.encode(), int(v)))
    if args.impl == 'reference':
        {'dit': run_dit_reference_arm, 'train': run_train_reference_arm}.get(args.workload, run_reference_arm)(args)
        return
    if args.workload == 'dit':
        run_dit(args)
        return
    if args.workload == 'tf':
        run_teacher_forced(args)
        return
    if args.workload == 'train':
        run_train(args)
        return

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)

    from core.models import LMM
    from core.utils import get_tokenizer
    from edgerunner_b200 import synth

    opt, wl, T, nf = workload(args)
    # synthetic checkpoint straight into fp16 (model.half() of infer.py:56 is exact on it); the module is built on the meta device and
    # the tensors are assigned, so that N ranks do not each run a 766 M-parameter random init + a 3 GB fp32 copy on the shared host
    sd = synth.synth_state_dict(opt, seed=0, eos_logit=-30.0, dtype=torch.float16)
    with torch.device('meta'):
        model = LMM(opt)
    model.load_state_dict(sd, strict=True, assign=True)
    del sd
    model = model.half().eval().to(dev)
    tokenizer, _ = get_tokenizer(opt)
    eng = model.get_engine(max_new_tokens=T)
    cond_host = synth.synth_point_cloud(seed=rank, n=opt.point_num).pin_memory()      # independent request per replica
    cond_dev = cond_host.to(dev)
    L0 = opt.num_cond_tokens + 1

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    dec_ms = []

    def step_device():
        """inputs resident in HBM: encoder + prefill + decode on the device, ids stay on the device"""
        eng.encode_cond(cond_dev[0], nf)
        eng.prefill([opt.bos_token_id])
        ev[2].record()
        out = eng.decode(T, mode='greedy', tokens_per_launch=args.tokens_per_launch, sync=False)
        ev[3].record()
        return out

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([x], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    for _ in range(args.warmup):
        out = step_device()
    barrier()
    launches0 = eng.kernel_launches()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    ev[0].record()
    for _ in range(args.steps):
        out = step_device()
        torch.cuda.current_stream().synchronize()
        dec_ms.append(ev[2].elapsed_time(ev[3]))
    ev[1].record()
    barrier()
    ms_total = max_over_ranks(ev[0].elapsed_time(ev[1]))
    clocks = sampler.stop() if rank == 0 else None
    launches = eng.kernel_launches() - launches0
    n_tok = int(out['n'].item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'tokens': out['ids'][:n_tok]})
    value = world * args.steps * n_tok / (ms_total / 1e3)
    dec_ms_avg = float(np.mean(dec_ms))

    # ---- e2e: the public call (LMM.generate) with host buffers ---------------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        def step_e2e():
            c = cond_host.to(dev, non_blocking=True)            # H2D of this step's input from pinned memory
            with torch.no_grad():
                meshes, toks = model.generate(c, num_faces=nf, max_new_tokens=T, tokenizer=tokenizer, clean=True)   # D2H of ids inside
            return toks[0]
        import contextlib, io
        e2e_steps = max(1, min(args.steps, args.e2e_steps))
        with contextlib.redirect_stdout(io.StringIO()):
            step_e2e()
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                toks = step_e2e()
            torch.cuda.synchronize()
            dt = max_over_ranks(time.perf_counter() - t0)
        e2e = {'value': world * e2e_steps * len(toks) / dt, 'unit': UNIT, 'h2d_bytes_per_step': int(cond_host.numel() * 4),
               'd2h_bytes_per_step': int(len(toks) * 4 + 4), 'ms_per_step': dt / e2e_steps * 1e3, 'steps': e2e_steps,
               'api': 'core.models.LMM.generate(cond, num_faces, max_new_tokens, tokenizer, clean=True) incl. meto detokenize + mesh clean-up'}

    comm = {'world_size': world, 'backend': 'none (single process)', 'gpus_active': 1}
    if world > 1:
        import torch.distributed as dist
        # which GPUs actually ran a replica: one all_gather of (uuid, tokens generated) over the NCCL communicator used for the barriers
        props = torch.cuda.get_device_properties(dev)
        mine = {'rank': rank, 'gpu': props.name, 'uuid': str(getattr(props, 'uuid', local_rank)), 'tokens': int(n_tok)}
        allr = [None] * world
        dist.all_gather_object(allr, mine)
        comm = {'world_size': world, 'backend': dist.get_backend(), 'nccl_version': '.'.join(str(x) for x in torch.cuda.nccl.version()),
                'gpus_active': len({r['uuid'] for r in allr}), 'tokens_per_rank': [r['tokens'] for r in allr],
                'collectives_on_data_path': 0, 'note': 'replicas: NCCL carries only the timing barriers / max-reduce and this gather'}
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    # ---- roofline of the dominant kernel ------------------------------------------------------------------------------------------------
    peaks_path = os.path.join(REPO, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))['hbm_gbs']), 'MEASURED_PEAKS.json hbm_gbs (of measured)'
    else:
        peak, peak_src = 6650.0, 'B200_PROFILING.md fallback 6.65 TB/s (of fallback)'
    alg = algorithmic_decode_bytes(eng, L0, n_tok)
    achieved = alg / (dec_ms_avg / 1e3) / 1e9
    traffic, traffic_note = None, None
    tpath = os.path.join(REPO, 'profiles', 'decode_traffic.json')
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        # ncu cannot replay a 15 s launch: the captured launch is a short one of the same kernel; its measured
        # DRAM-bytes / algorithmic-bytes ratio is applied to this launch's algorithmic bytes
        traffic = tj['dram_over_algorithmic'] * alg if 'dram_over_algorithmic' in tj else None
        traffic_note = tj.get('note')
    roofline = {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic,
                'kernel': 'er::decode_persistent_kernel', 'algorithmic_bytes_per_launch': alg, 'launch_ms': dec_ms_avg,
                'peak_source': peak_src, 'frac_of_nominal_8TBs': achieved / 8000.0,
                'decode_only_tokens_per_s': (n_tok - 1) / (dec_ms_avg / 1e3), 'traffic_note': traffic_note}
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        cpu = cpu_baseline_leg(args, opt)
    ref_gpu = None
    if not args.no_reference_gpu and world == 1:
        del model, eng
        torch.cuda.empty_cache()
        r = ref_leg('gpu', 2, 1, tokens=32 if not args.tiny else 8, tiny=args.tiny, timeout=600)
        if r is not None and 'error' not in r:
            ref_gpu = {'value': r['tok_s'], 'unit': UNIT, 'kind': 'reference', 'path': r['path'], 'windows_tok_s': r['windows_tok_s'], 'sample': r['sample'],
                       'model': r['model'], 'ours_over_reference_gpu': value / r['tok_s']}
        else:
            ref_gpu = {'unavailable': 'oracle/_ref/py absent' if r is None else r['error']}
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms_total / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f16',
        'data': 'synthetic',
        'config': {'workload': wl, 'tokens_per_step_per_gpu': n_tok, 'prefix_rows': L0, 'parallelism': f'replicas x{world}',
                   'l2': 'inputs larger than L2: 1.36 GB weights + up to 2.66 GB KV cache streamed per token vs 126 MB L2',
                   'weights': 'seeded synthetic, fp16 (edgerunner_b200.synth)'},
        'clocks': clocks, 'e2e': e2e, 'gpu_launches': int(launches), 'roofline': roofline, 'cpu_baseline': cpu, 'reference_gpu': ref_gpu, 'comm': comm,
    }
    emit(json.dumps(line), flush=True)


if __name__ == '__main__':
    main()
