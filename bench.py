"""Headline benchmark: captions/sec at beam=5, seq_len=20 (BASELINE.json metric), UpDown, 36x2048 bottom-up features.

    python bench.py --gpus N --steps K --warmup W            # this engine (one process per GPU; torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # the UNMODIFIED reference (oracle/_ref copy) on the host cores
    python bench.py ... --dump-outputs DIR                   # also write what the timed path computed in its last step to DIR/*.npy

A "step" = one pass of the hot path (AttModel._sample_beam: prologue + 20 timesteps + beam bookkeeping) over one batch of
synthetic inputs (configs[1]: batch 256 per GPU).  Images are independent, so ranks shard the work with no data-path
collective ("scaling": "weak"); the only collectives are the timing barrier and the max-over-ranks reduction.

  value   captions/s with the step's inputs already resident in HBM (CUDA events, max over ranks)
  e2e     the same metric through the public model(...) call with HOST (pinned) inputs: H2D copy of the features and the
          D2H read of the caption ids are inside the timed region, every step
  roofline the dominant kernel (the persistent tcgen05 GEMM: CTA-pair kernel for the LSTM-gate and logit call sites): algorithmic
          FLOPs of all its launches / their CUDA-event time vs the measured bf16 tensor peak in MEASURED_PEAKS.json, the DRAM traffic
          of the largest call site from the committed ncu capture, and the fraction of the 3-pass ceiling (DESIGN.md section 3)
  cpu_baseline  the unmodified reference modules (oracle/_ref; "kind": "reference"), timed on this box's host cores on a bounded sample
  scst    the second half of BASELINE.json's metric in the SAME line: SCST samples/sec on configs[3] (AoANet, per-GPU batch 10 x 5
          samples, CIDEr-D reward, BPTT, NCCL gradient all-reduce, Adam), with per-rank times, the all-reduce time and its HBM roofline

Other workloads (--workload): transformer_beam / aoa_beam (BASELINE configs[2] shape and AoANet decode), updown_scst / aoa_scst (SCST
training step incl. H2D, the single NCCL gradient all-reduce and Adam; aoa_scst = BASELINE configs[3]).  The GPU arms build their
seeded random-init model and features from imagecaptioning.pytorch_b200.synthetic; only cpu_reference_rate() / cpu_reference_scst_rate() touch oracle/.

The benchmark runs the library __graft_entry__.build() made and writes nothing into the tree, which may be read-only.  With the same
arguments every run sees the same inputs and random draws, so the arrays --dump-outputs writes can be compared between two builds.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.dont_write_bytecode = True          # no __pycache__ in the tree

DUMP_LIMIT_BYTES = 64 << 20
DUMP_LOGPROB_ROWS = 32                  # seeded sample of the [rows, T, V+1] log-prob rows written by --dump-outputs
DUMP_GRAD_ENTRIES = 1 << 20             # seeded sample of the SCST step's gradient entries

CFG = dict(V=9487, E=1000, H=1000, A=512, F_fc=2048, F_att=2048, T=20)     # configs/updown/updown.yml + opts.py defaults
R = 36


def parse():
    p = argparse.ArgumentParser()
    p.add_argument('--gpus', type=int, default=1)
    p.add_argument('--steps', type=int, default=10)
    p.add_argument('--warmup', type=int, default=3)
    p.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    p.add_argument('--batch', type=int, default=None, help='images per GPU per step (default 256; 10 for updown_scst = BASELINE configs[3])')
    p.add_argument('--beam', type=int, default=5)
    p.add_argument('--mode', default='tc_f16x3', choices=['tc_f16x3', 'tc_f16x1', 'simt_fp32'])
    p.add_argument('--cpu-batch', type=int, default=32, help='images per CPU-baseline step (bounded sample)')
    p.add_argument('--no-cpu-baseline', action='store_true')
    p.add_argument('--workload', default='updown_beam', choices=['updown_beam', 'transformer_beam', 'aoa_beam', 'updown_scst', 'aoa_scst', 'transformer_scst'],
                   help='updown_beam = BASELINE.json configs[1] (the headline); transformer_beam = configs[2] (use --batch 64); aoa_beam = AoANet decode')
    p.add_argument('--dump-outputs', metavar='DIR', default=None,
                   help='after the timed steps, write what each timed path computed in its last step to DIR/<name>.npy (float32 / float64, '
                        'seeded samples of the large arrays, at most 64 MB in all)')
    args = p.parse_args()
    if args.steps < 1:
        p.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        p.error('--dump-outputs writes the outputs of the GPU arm (--impl b200)')
    if args.batch is None:
        args.batch = 10 if args.workload in ('updown_scst', 'aoa_scst', 'transformer_scst') else 256
    return args


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        names = {'hw_slowdown': 0x8, 'sw_power_cap': 0x4, 'hw_thermal_slowdown': 0x40, 'sw_thermal_slowdown': 0x20, 'hw_power_brake': 0x80}
        while not self.stop_flag:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                bits = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(self.nv, 'nvmlDeviceGetCurrentClocksEventReasons') \
                    else self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for n, b in names.items():
                    if bits & b:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(float(os.environ.get('CAPB200_CLOCK_SAMPLE_S', '0.05')))

    def summary(self):
        return {'sm_mhz': statistics.median(self.samples) if self.samples else None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons)}


def _calibrate_threads(run_once):
    """The reference's eager loop of small GEMMs, sorts and gathers scales badly past a few dozen threads (0.7 captions/s with 128 threads vs
    ~25 with 8 on the same code), so the thread count is calibrated on a small problem and the best one is used and reported."""
    import torch
    ncpu = os.cpu_count() or 1
    best = (None, float('inf'))
    for c in sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu}):
        torch.set_num_threads(c)
        run_once()
        t0 = time.perf_counter()
        run_once()
        dt = time.perf_counter() - t0
        if dt < best[1]:
            best = (c, dt)
    torch.set_num_threads(best[0])
    return best[0]


def cpu_reference_rate(batch, beam, steps, warmup):
    """captions/s of the reference's CPU path on this box's host cores: the UNMODIFIED reference modules (oracle/_ref, a verbatim copy made by
    oracle/build_ref.py) when the copy is present -- kind "reference" -- else the oracle port (kind "port").  Same model / feature shapes and
    seeds as the GPU arm.  Returns (captions/s, seconds per step, threads, kind)."""
    import torch
    from oracle import caption_oracle as co
    from oracle import ref_runtime as rr
    W = co.make_weights('updown', CFG['V'], CFG['E'], CFG['H'], CFG['A'], CFG['F_fc'], CFG['F_att'], seed=1234, logit_scale=12.0)
    use_ref = rr.available()
    opt = {'beam_size': beam, 'sample_n': 1}
    if use_ref:
        cwd = os.getcwd()
        m = rr.model('updown', W=W, **CFG)
        run = lambda fc, att: m(fc, att, None, opt=opt, mode='sample')
    else:
        fam = co.Family('updown', W, CFG['T'])
        run = lambda fc, att: co.sample_beam(fam, fc, att, beam_size=beam)
    fcc, attc = co.make_inputs(8, R, CFG['F_fc'], CFG['F_att'], seed=1)
    with torch.no_grad():
        cores = _calibrate_threads(lambda: run(fcc, attc))
        fc, att = co.make_inputs(batch, R, CFG['F_fc'], CFG['F_att'], seed=1234)
        times = []
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            run(fc, att)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    if use_ref:
        os.chdir(cwd)
    dt = statistics.median(times)
    return batch / dt, dt, cores, 'reference' if use_ref else 'port'


def cpu_reference_scst_rate(B, n, steps):
    """SCST samples/s of the reference on the host cores: LossWrapper(sc_flag=True).forward + backward of the unmodified AoANet modules
    (configs[3] shape: per-GPU batch 10, train_sample_n 5), CIDEr-D scorer fed from a synthetic document-frequency pickle."""
    import argparse as ap
    import torch
    from oracle import caption_oracle as co
    from oracle import ciderd_oracle as cdo
    from oracle import ref_runtime as rr
    if not rr.available():
        return None
    cwd = os.getcwd()
    cfg = dict(CFG, E=1024, H=1024)
    W = co.make_weights('aoa', cfg['V'], cfg['E'], cfg['H'], cfg['A'], cfg['F_fc'], cfg['F_att'], seed=1234, logit_scale=6.0)
    m = rr.model('aoa', W=W, **cfg, **dict(rr.FAMILY_EXTRA['aoa'], num_heads=8))
    from captioning.modules.loss_wrapper import LossWrapper
    gts = cdo.make_refs(B, cfg['V'], seed=5)
    df, ref_len = cdo.build_document_frequency(cdo.make_refs(1000, cfg['V'], seed=4))
    rr.write_df_pickle('bench-df', df, ref_len)
    rr.init_scorer('bench-df')
    opt = ap.Namespace(label_smoothing=0, structure_loss_type='seqnll', structure_loss_weight=1, train_sample_method='sample', train_beam_size=1,
                       train_sample_n=n, sc_sample_method='greedy', sc_beam_size=1, cider_reward_weight=1.0, bleu_reward_weight=0.0, use_ppo=0,
                       struc_use_logsoftmax=1)
    lw = LossWrapper(m, opt)
    fc, att = co.make_inputs(B, R, cfg['F_fc'], cfg['F_att'], seed=1234)
    import contextlib
    import io

    def step():
        m.zero_grad()
        with contextlib.redirect_stdout(io.StringIO()):          # rewards.py:65 prints the CIDEr score on every call
            out = lw(fc, att, None, None, None, gts, torch.arange(B), True, False, False)
        out['loss'].backward()
    cores = _calibrate_threads(step)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    os.chdir(cwd)
    dt = statistics.median(times)
    return {'value': B * n / dt, 'unit': 'samples/s', 'ms_per_step': dt * 1e3, 'cores': cores, 'kind': 'reference',
            'sample': '%d steps of LossWrapper(sc_flag=True).forward + backward, AoANet, batch %d x %d samples (no optimizer step)' % (steps, B, n)}


SCST_WEIGHT_BYTES = 110e6          # fp32 AoANet decoder weights touched by one time step (27.5 M parameters, SURVEY.md section 8d)


def _per_rank(ms, dev, world):
    """Every rank's own CUDA-event time of the timed region (list, rank order) and the max over ranks."""
    import torch
    import torch.distributed as dist
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        vals = [float(o.item()) for o in out]
    else:
        vals = [ms]
    return vals, max(vals)


def _seeded_subset(n, k, seed=0):
    """Sorted indices of a fixed, seeded choice of min(n, k) of range(n)."""
    import numpy as np
    import torch
    return torch.from_numpy(np.sort(np.random.default_rng(seed).choice(n, size=min(n, k), replace=False)))


def decode_outputs(prefix, seq, logprobs):
    """What a caller of the decode receives: the caption ids [B, T] and a seeded sample of the log-prob rows [B, T, V+1]."""
    out = {prefix + '_seq': seq.cpu()}
    if logprobs is not None:
        rows = _seeded_subset(logprobs.shape[0], DUMP_LOGPROB_ROWS)
        out[prefix + '_logprobs_sample'] = logprobs[rows.to(logprobs.device)].cpu()
        out[prefix + '_logprobs_sample_rows'] = rows
    return out


def write_outputs(out_dir, arrays):
    """DIR/<name>.npy per array: integer and float64 arrays as float64, the rest as float32."""
    import numpy as np
    host = {}
    for name, a in arrays.items():
        a = np.asarray(a.detach().cpu().numpy() if hasattr(a, 'detach') else a)
        host[name] = a.astype(np.float64 if a.dtype == np.float64 or np.issubdtype(a.dtype, np.integer) else np.float32)
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError('--dump-outputs: %d bytes exceed the %d byte limit' % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def bench_scst(args, rank, world, local_rank, dev, workload, batch):
    """SCST samples/sec (the second half of BASELINE.json's metric): AoANet (configs[3]) or UpDown, per-GPU batch `batch` images,
    train_sample_n = 5, CIDEr-D reward, greedy baseline, BPTT, gradient all-reduce over NCCL (overlapped with the backward pass when the loss
    wrapper supports it), value clipping and Adam.  Every step starts from pinned HOST features (H2D inside the timed region) and ends with
    the D2H read of the loss.  Returns the result dict on every rank (rank 0 prints) and, with --dump-outputs, the last step's outputs."""
    import argparse as ap
    import torch
    import torch.distributed as dist
    import imagecaptioning.pytorch_b200 as b200
    from imagecaptioning.pytorch_b200 import synthetic as syn
    B, n, T = batch, 5, CFG['T']
    aoa = workload == 'aoa_scst'
    if aoa:       # configs/aoa.yml: E = H = 1024, 8 heads, 6 refiner layers, ctx_drop, dropout_aoa 0.3 (BASELINE configs[3])
        model = syn.build_model('aoa', seed=1234, logit_scale=6.0, mode=args.mode, device=dev, heads=8, **dict(CFG, E=1024, H=1024, A=0))
    elif workload == 'transformer_scst':    # configs/transformer/transformer.yml: 6 + 6 layers, d_model 512, d_ff 2048, 8 heads
        model = syn.build_model('transformer', seed=1234, logit_scale=3.0, mode=args.mode, device=dev, heads=8, **dict(CFG, E=512, H=2048, A=6))
    else:
        model = syn.build_model('updown', seed=1234, logit_scale=12.0, mode=args.mode, device=dev, **CFG)
    fam_name = 'AoANet' if aoa else ('Transformer' if workload == 'transformer_scst' else 'UpDown')
    model.train()
    df, ref_len = syn.document_frequency(syn.make_refs(1000, CFG['V'], seed=4))              # synthetic DF table (format of prepro_ngrams.py)
    b200.rewards.reset_scorer()
    b200.rewards.init_scorer(b200.rewards.CiderDTable(df, ref_len))
    opt = ap.Namespace(sc_sample_method='greedy', sc_beam_size=1, train_sample_method='sample', train_beam_size=1, train_sample_n=n,
                       cider_reward_weight=1, bleu_reward_weight=0)
    lw = b200.B200LossWrapper(model, opt)
    fused_sync = world > 1 and hasattr(lw, 'enable_gradient_sync') and not os.environ.get('CAPB200_SCST_NO_OVERLAP')     # A/B switch
    if fused_sync:
        lw.enable_gradient_sync()            # the engine's flat gradient buffer is all-reduced in chunks while the backward pass still runs
    # tools/train.py:193-196: utils.clip_gradient(optimizer, 0.1) + Adam.step(), one launch of the engine's fused kernel (optim.py)
    optim = b200.optim.FusedAdam(model.parameters(), lr=5e-5, clip_value=0.1)
    host = [syn.make_inputs(B, R, CFG['F_fc'], CFG['F_att'], seed=99 + 13 * rank + i) for i in range(3)]
    host = [(a.pin_memory(), b.pin_memory()) for a, b in host]
    gts = syn.make_refs(B, CFG['V'], seed=5 + rank)
    idx = torch.arange(B)
    grad_bytes = [0]
    ar_events = []
    last = {}

    def step(i, timed=False):
        fc_h, att_h = host[i % 3]
        fc, att = fc_h.to(dev, non_blocking=True), att_h.to(dev, non_blocking=True)      # H2D every step (inputs start on the host)
        out = lw(fc, att, None, None, None, gts, idx, True, False, False)
        if args.dump_outputs:
            last.update(loss=out['loss'].detach(), reward=out['reward'].detach())
        optim.zero_grad(set_to_none=True)
        out['loss'].backward()
        if fused_sync:
            grad_bytes[0] = lw.last_sync_bytes
        else:
            if timed and world > 1:
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
            grad_bytes[0] = b200.parallel.allreduce_gradients(model.parameters())        # the one collective of the step
            if timed and world > 1:
                a1.record()
                ar_events.append((a0, a1))
        optim.step()
        return float(out['loss'].detach())                                                        # D2H read of the loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(3, args.warmup)):
        step(i)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = model.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    step_ms = []
    for i in range(args.steps):
        t_s = time.perf_counter()
        step(args.warmup + i, timed=True)
        step_ms.append((time.perf_counter() - t_s) * 1e3)
    e1.record()
    barrier()
    if os.environ.get('CAPB200_BENCH_STEP_TIMES'):
        print('rank %d per-step wall ms: %s' % (rank, ' '.join('%.1f' % v for v in step_ms)), file=sys.stderr, flush=True)
    sampler.stop_flag = True
    sampler.join()
    per_rank, ms = _per_rank(e0.elapsed_time(e1), dev, world)
    dump = None
    if args.dump_outputs:
        # the loss and mean reward the step returns, the captions it sampled, and a seeded sample of the gradients it left (clipped by the step)
        grads = torch.cat([p.grad.reshape(-1) for p in model.parameters() if p.grad is not None])
        pick = _seeded_subset(grads.numel(), DUMP_GRAD_ENTRIES)
        dump = {'scst_loss': last['loss'].reshape(1), 'scst_reward': last['reward'].reshape(1),
                'scst_sample_seq': lw.last_step['sample_seq'], 'scst_grad_sample': grads[pick.to(dev)], 'scst_grad_sample_index': pick}
        dump = {k: v.cpu() for k, v in dump.items()}
        del grads
    if fused_sync:
        allreduce_ms = getattr(lw, 'last_sync_exposed_ms', None)
    else:
        allreduce_ms = statistics.mean(a.elapsed_time(b) for a, b in ar_events) if ar_events else 0.0
    peaks_path = os.path.join(REPO, 'MEASURED_PEAKS.json')
    hbm = float(json.load(open(peaks_path))['hbm_gbs']) if os.path.exists(peaks_path) else 6650.0
    step_s = ms / args.steps / 1e3
    # algorithmic HBM bytes of one step (SURVEY.md 8d, AoANet): the 110 MB of fp32 decoder weights are streamed once per time step by the
    # sampling forward and about twice by the backward (input gradients read W, weight gradients write dW): 3 x T x 110 MB = 6.6 GB
    alg_bytes = 3 * T * SCST_WEIGHT_BYTES if aoa else None
    value = world * B * n * args.steps / (ms / 1e3)
    res = {'metric': 'SCST samples/sec (%s, train_sample_n=5, CIDEr-D reward, greedy baseline, BPTT, Adam)' % fam_name, 'value': value, 'unit': 'samples/s',
           'images_per_sec': value / n, 'n_gpus': world, 'steps': args.steps, 'ms_per_step': ms / args.steps, 'per_rank_ms_per_step': [v / args.steps for v in per_rank],
           'allreduce_ms': allreduce_ms, 'allreduce_bytes': grad_bytes[0], 'allreduce': 'chunked, overlapped with the backward pass' if fused_sync else ('one flat all-reduce after backward' if world > 1 else 'none (1 GPU)'),
           'launches': (model.launch_count - l0) // max(args.steps, 1), 'scaling': 'weak',
           'step_wall_ms': {'min': min(step_ms), 'median': statistics.median(step_ms), 'max': max(step_ms)},
           'config': {'workload': '%s SCST step (BASELINE configs[3]), per-GPU batch=%d images x %d samples, 36x2048 feats, seq_len=20, V=9487' % (fam_name, B, n),
                      'numeric_mode': 'greedy baseline %s (tcgen05 kind::f16 x3); sampling, backward and weight gradients on 3xTF32 tensor-core GEMMs over the fp32 weights' % args.mode},
           'clocks': sampler.summary(),
           'roofline': None if alg_bytes is None else {'bound': 'hbm', 'bytes': alg_bytes, 'achieved': alg_bytes / step_s / 1e9, 'peak': hbm, 'unit': 'GB/s',
                                                       'frac': alg_bytes / step_s / 1e9 / hbm,
                                                       'note': 'algorithmic bytes = 3 x T x 110 MB of decoder weights (SURVEY.md 8d); the step is latency/launch bound, not bandwidth bound'},
           'e2e': {'value': value, 'unit': 'samples/s', 'h2d_bytes_per_step': B * (CFG['F_fc'] + R * CFG['F_att']) * 4, 'd2h_bytes_per_step': 4,
                   'note': 'the timed region IS end to end: pinned host features copied H2D every step, loss read back D2H every step'}}
    del optim, lw, model
    torch.cuda.empty_cache()
    return res, dump


def main():
    args = parse()
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    names = {'updown_beam': 'UpDown', 'transformer_beam': 'Transformer 6+6/512/2048/8', 'aoa_beam': 'AoANet 1024', 'updown_scst': 'UpDown SCST',
             'aoa_scst': 'AoANet SCST', 'transformer_scst': 'Transformer 6+6/512/2048/8 SCST'}
    workload = '%s beam=%d, %dx2048 bottom-up feats, batch=%d per GPU, seq_len=20, V=9487' % (names[args.workload], args.beam, R, args.batch)

    if args.impl == 'reference':
        # The reference's own CPU implementation of the path on this box's host cores: the unmodified modules (oracle/_ref) at the
        # configured batch; rank 0 alone runs it.
        if rank != 0:
            return
        steps = args.steps
        batch = args.batch if args.workload == 'updown_beam' else args.cpu_batch
        rate, dt, cores, kind = cpu_reference_rate(batch, args.beam, steps, 1)
        line = {'impl': 'reference', 'metric': 'captions/sec at beam=5 seq_len=20', 'value': rate, 'unit': 'captions/s', 'n_gpus': args.gpus,
                'steps': steps, 'warmup': 1, 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
                'data': 'synthetic', 'config': {'workload': workload, 'sample': 'batch=%d per step on the host cores (the configured batch)' % batch},
                'cpu_baseline': {'value': rate, 'unit': 'captions/s', 'cores': cores, 'kind': kind, 'host_cpus': os.cpu_count(),
                                 'sample': '%d steps of batch %d through %s (torch fp32 CPU, best thread count of a calibration sweep)' %
                                           (steps, batch, 'the unmodified reference modules copied to oracle/_ref' if kind == 'reference' else 'the oracle port')},
                'e2e': {'value': rate, 'unit': 'captions/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}
        if args.workload == 'updown_beam' and not os.environ.get('CAPB200_BENCH_NO_SCST'):
            sc = cpu_reference_scst_rate(10, 5, 2)
            if sc is not None:
                line['scst'] = sc
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    import imagecaptioning.pytorch_b200 as b200
    b200._lib.load()                        # made by __graft_entry__.build(); a missing library is an error, not a rebuild
    torch.manual_seed(1234 + rank)          # the SCST steps draw their sampling / dropout seeds from torch's generator
    torch.cuda.set_device(local_rank)
    try:        # bind this rank to the CPU cores next to its GPU (NUMA): the SCST step is ~1300 launches of host-side work per step
        if os.environ.get('CAPB200_BENCH_NO_AFFINITY'):
            raise RuntimeError('disabled')
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local_rank))
    except Exception:
        pass
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
        dist.barrier()
    from imagecaptioning.pytorch_b200 import synthetic as syn      # seeded random-init weights / features: the GPU arm never touches oracle/
    dev = torch.device('cuda', local_rank)
    if args.workload in ('updown_scst', 'aoa_scst', 'transformer_scst'):
        res, dump = bench_scst(args, rank, world, local_rank, dev, args.workload, args.batch)
        if rank == 0:
            if dump is not None:
                write_outputs(args.dump_outputs, dump)
            line = dict(res, warmup=args.warmup, higher_is_better=True, vs_baseline=None, dtype='f32', data='synthetic', gpu_launches=res['launches'] * args.steps)
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return
    if args.workload == 'updown_beam':
        model = syn.build_model('updown', seed=1234, logit_scale=12.0, mode=args.mode, device=dev, **CFG)
    elif args.workload == 'transformer_beam':     # configs/transformer/transformer.yml: d_model 512, d_ff 2048, 6 + 6 layers, 8 heads
        model = syn.build_model('transformer', seed=1234, logit_scale=3.0, mode=args.mode, device=dev, heads=8,
                                **dict(CFG, E=512, H=2048, A=6))
    else:                                         # configs/aoa.yml: E = H = 1024, 8 heads, 6 refiner layers
        model = syn.build_model('aoa', seed=1234, logit_scale=6.0, mode=args.mode, device=dev, heads=8, **dict(CFG, E=1024, H=1024, A=0))
    B, T = args.batch, CFG['T']
    opt = {'beam_size': args.beam, 'sample_n': 1}
    n_rot = 3                                         # rotate input batches; per-step working set (features, weights, 1 GB slab) >> 126 MB L2
    host = [syn.make_inputs(B, R, CFG['F_fc'], CFG['F_att'], seed=1234 + 17 * rank + i) for i in range(n_rot)]
    host = [(a.pin_memory(), b.pin_memory()) for a, b in host]
    devin = [(a.to(dev), b.to(dev)) for a, b in host]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident(i):
        fc, att = devin[i % n_rot]
        with torch.no_grad():
            return model(fc, att, None, opt=opt, mode='sample')

    # End-to-end: features start in pinned HOST memory every step; the H2D copy of step i+1 is issued on a side stream while
    # step i decodes, and each step's caption ids are copied back to pinned host memory (D2H) and read one step later.
    copy_stream = torch.cuda.Stream(device=dev)
    pending = {}
    out_host = [torch.empty(B, T, dtype=torch.long).pin_memory() for _ in range(2)]
    out_events = [None, None]

    def prefetch(i):
        fc_h, att_h = host[i % n_rot]
        with torch.cuda.stream(copy_stream):
            fc = fc_h.to(dev, non_blocking=True)
            att = att_h.to(dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        pending[i] = (fc, att, ev)

    def step_e2e(i):
        if i not in pending:
            prefetch(i)
        fc, att, ev = pending.pop(i)
        cur = torch.cuda.current_stream()
        cur.wait_event(ev)
        fc.record_stream(cur)
        att.record_stream(cur)
        prefetch(i + 1)
        with torch.no_grad():
            seq, _ = model(fc, att, None, opt=opt, mode='sample')
        slot = i % 2
        if out_events[slot] is not None:
            out_events[slot].synchronize()                 # the ids of step i-2 are on the host now
            _ = int(out_host[slot][0, 0])
        out_host[slot].copy_(seq, non_blocking=True)       # the captions (ids) are the step's result
        out_events[slot] = torch.cuda.Event()
        out_events[slot].record(cur)
        return seq

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        l0 = model.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps - 1):
            fn(warmup + i)
        out = fn(warmup + steps - 1)         # kept for --dump-outputs; earlier outputs are freed as before
        e1.record()
        barrier()
        sampler.stop_flag = True
        sampler.join()
        per_rank, mx = _per_rank(e0.elapsed_time(e1), dev, world)
        return mx, sampler.summary(), model.launch_count - l0, per_rank, out

    dump = {}
    ms, clocks, launches, per_rank, out = timed(step_resident, args.steps, max(3, args.warmup))
    if args.dump_outputs:                   # copied before the next call of the model
        dump.update(decode_outputs('decode', *out))
    value = world * B * args.steps / (ms / 1e3)
    ms_e2e, _, _, per_rank_e2e, out = timed(step_e2e, args.steps, max(3, args.warmup))
    if args.dump_outputs:
        dump.update(decode_outputs('e2e', out, None))
    del out
    pending.clear()
    e2e = world * B * args.steps / (ms_e2e / 1e3)

    if args.workload != 'updown_beam':
        if rank == 0:
            line = {'metric': 'captions/sec at beam=5 seq_len=20', 'value': value, 'unit': 'captions/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
                    'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': args.mode, 'data': 'synthetic',
                    'config': {'workload': workload, 'numeric_mode': args.mode, 'global_batch': B * world}, 'clocks': clocks,
                    'per_rank_ms_per_step': [v / args.steps for v in per_rank],
                    'e2e': {'value': e2e, 'unit': 'captions/s', 'h2d_bytes_per_step': B * (CFG['F_fc'] + R * CFG['F_att']) * 4, 'd2h_bytes_per_step': B * T * 8},
                    'gpu_launches': launches, 'roofline': None}
            if args.dump_outputs:
                write_outputs(args.dump_outputs, dump)
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return

    # roofline of the dominant kernel, timed live with CUDA events on the launching stream over a few more steps
    model.set_profiling(True)
    for i in range(3):
        step_resident(i)
    prof = model.read_profile()
    model.set_profiling(False)
    peaks_path = os.path.join(REPO, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))['bf16_tflops_sustained']), 'MEASURED_PEAKS.json bf16_tflops_sustained (of measured)'
    else:
        peak, peak_src = 1400.0, 'fallback 1.4 PFLOP/s sustained (of fallback)'
    # The dominant kernel is the persistent tcgen05 GEMM (gemm_tc_kernel): every dense contraction of the step is a launch of it.
    # achieved = algorithmic FLOPs (2*M*N*K of the contraction actually executed) of ALL its launches / their summed CUDA-event time;
    # the largest single call site (language-LSTM gates, M=B*beam, N=4000, K=3000) is listed beside it.
    # DRAM bytes per launch of one of the three large call sites (the capture's own `kernel` field says which) from the committed
    # `ncu --set full` capture, when present
    traffic, traffic_src = None, None
    tpath = os.path.join(REPO, 'profiles', 'roofline_traffic.json')
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic, traffic_src = tj.get('dram_bytes_per_launch'), tj.get('source')
    all_ms = sum(v[0] for v in prof.values())
    all_fl = sum(v[1] for v in prof.values())
    all_calls = sum(v[2] for v in prof.values())
    achieved = all_fl / (all_ms / 1e3) / 1e12 if all_ms > 0 else 0.0
    big_ms, big_fl, big_calls = prof['lang_lstm']
    passes = 3 if args.mode == 'tc_f16x3' else 1
    roofline = {'bound': 'tensor', 'kernel': 'gemm_tc_pair_kernel<144,%d> / gemm_tc_kernel<64,..> (persistent tcgen05 GEMM, cta_group::2 pairs for the large call sites; all call sites of the step)' % passes,
                'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s', 'frac': achieved / peak, 'traffic': traffic, 'traffic_source': traffic_src, 'traffic_kernel': tj.get('kernel') if traffic is not None else None, 'peak_source': peak_src,
                'mma_passes': passes,
                'frac_of_pass_ceiling': achieved / (peak / passes),       # fp32-grade results cost 3 MMA passes per product
                'launches_timed': all_calls, 'avg_launch_ms': all_ms / max(all_calls, 1),
                'share_of_step': (all_ms / 3) / (ms / args.steps),
                'whole_step': {'algorithmic_tflop_per_batch': all_fl / 3 / 1e12, 'tflops': all_fl / 3 / (ms / args.steps / 1e3) / 1e12,
                               'frac': all_fl / 3 / (ms / args.steps / 1e3) / 1e12 / peak, 'frac_of_pass_ceiling': all_fl / 3 / (ms / args.steps / 1e3) / 1e12 / (peak / passes)},
                'largest_call_site': {'name': 'lang_lstm gates M=%d N=4000 K=3000 (fused LSTM cell epilogue)' % (B * args.beam),
                                      'tflops': big_fl / (big_ms / 1e3) / 1e12 if big_ms > 0 else 0.0, 'avg_launch_ms': big_ms / max(big_calls, 1),
                                      'frac': (big_fl / (big_ms / 1e3) / 1e12 if big_ms > 0 else 0.0) / peak},
                'per_gemm_ms_per_step': {k: v[0] / 3 for k, v in prof.items() if v[2] > 0},
                'per_gemm_tflops': {k: v[1] / (v[0] / 1e3) / 1e12 for k, v in prof.items() if v[0] > 0}}
    del model
    devin = None
    torch.cuda.empty_cache()

    # the second half of BASELINE.json's metric, in the same line: SCST samples/sec on configs[3] (AoANet, per-GPU batch 10 x 5 samples)
    scst = None
    if not os.environ.get('CAPB200_BENCH_NO_SCST'):
        scst, scst_dump = bench_scst(args, rank, world, local_rank, dev, 'aoa_scst', 10)
        if scst_dump is not None:
            dump.update(scst_dump)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = {'metric': 'captions/sec at beam=5 seq_len=20', 'value': value, 'unit': 'captions/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32 (fp32-grade: split-fp16 x3 tensor-core passes, fp32 accumulate)' if args.mode == 'tc_f16x3' else args.mode, 'data': 'synthetic',
            'config': {'workload': workload, 'numeric_mode': args.mode, 'global_batch': B * world, 'parallelism': 'dp%d (independent images, no collective)' % world,
                       'l2': 'inputs rotated over %d batches; per-step working set ~1.3 GB >> 126 MB L2' % n_rot},
            'clocks': clocks, 'per_rank_ms_per_step': [v / args.steps for v in per_rank],
            'e2e': {'value': e2e, 'unit': 'captions/s', 'h2d_bytes_per_step': B * (CFG['F_fc'] + R * CFG['F_att']) * 4, 'd2h_bytes_per_step': B * T * 8,
                    'ms_per_step': ms_e2e / args.steps, 'per_rank_ms_per_step': [v / args.steps for v in per_rank_e2e]},
            'gpu_launches': launches, 'roofline': roofline}
    if scst is not None:
        line['scst'] = scst
    if not args.no_cpu_baseline and world == 1:
        rate, dt, cores, kind = cpu_reference_rate(args.cpu_batch, args.beam, 2, 1)
        line['cpu_baseline'] = {'value': rate, 'unit': 'captions/s', 'cores': cores, 'kind': kind, 'host_cpus': os.cpu_count(),
                                'sample': '2 steps of batch %d through %s (torch fp32 CPU, best thread count of a calibration sweep)' %
                                          (args.cpu_batch, 'the unmodified reference modules copied to oracle/_ref' if kind == 'reference' else 'the oracle port')}
    if args.dump_outputs:
        write_outputs(args.dump_outputs, dump)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
