#!/usr/bin/env python
"""bench.py -- one JSON line per run (see the round contract).

Default workload (`--workload dense`, BASELINE.json configs[1]): one STEP = one pass of `fp8_gemm_nt` over the four
DeepSeek-V3 dense shapes M in {64,128,512,4096}, N=4096, K=7168 (synthetic BF16 randn, quantised like the
reference's tests: 1x128 UE8M0 token scales, 128x128 UE8M0 weight scales). `value` = sum(2MNK) / sum(device time) in
TFLOPS with operands resident in HBM and packed scale factors prepared (kernel-only, cold L2: a 512 MB flush
precedes every timed launch, timed with CUDA events on the launching stream). `e2e` = the same step through the
public API from PINNED HOST buffers: H2D of BF16 activations and FP8 weights + scales, the CUDA activation quantiser,
scale packing, the GEMMs, D2H of D.

Outside the timed regions the same line also carries (every block degrades to {"unavailable": reason}):
  * `vs_reference_kernel` -- the UNMODIFIED reference SM100 kernel (oracle/_ref, JIT-compiled on the box) timed beside
    ours on the same tensors with the same flush + CUDA-event method, interleaved launch by launch, per dense shape;
    `bitwise_equal` compares the two outputs with split-K off (north_star: ">= the reference on every listed shape").
  * `grouped` -- BASELINE configs 3 (contiguous, 256 experts, mean M 128) and 4 (masked decode under a CUDA graph, mean M 64)
    with their HBM roofline and the same A/B.
  * `ep` -- BASELINE config 5 at THIS run's --gpus N: the expert-sharded step (peer-memory dispatch + grouped GEMM +
    weighted top-k combine) with dispatch / GEMM / combine split and, for N > 1, the 1-GPU step run on rank 0 so that
    `efficiency_vs_n1` is in the line. `value` stays the dense metric (replicas), so the driver's scaling table keeps one
    metric across N.
  * `decode_chain` -- the M = 64 GEMM inside a chain of 12 layers (stream order / PDL / CUDA graph), ours and the reference's.
  * `fp8_peak` -- the issue-only tcgen05.mma block-scaled FP8 probe (burst and 2 s sustained); `roofline.peak` uses it.

`--impl reference` runs the UNMODIFIED reference through its own public API (`deep_gemm.fp8_gemm_nt` from oracle/_ref) on
the same four shapes with the same method (value kernel-only, e2e from pinned host buffers), as replicas on every rank;
when the reference cannot be imported it falls back to the torch-CPU BF16-emulated GEMM (oracle port) on a bounded sample.
Its `cpu_baseline` block is that CPU port in both cases (the reference has no CPU implementation of this path).

`--dump-outputs DIR` (dense workload) writes D of the four shapes as the last timed step left them, as float32 .npy files
(see `dump_outputs`). The inputs come from fixed seeds, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

DENSE_SHAPES = [(64, 4096, 7168), (128, 4096, 7168), (512, 4096, 7168), (4096, 4096, 7168)]
NOMINAL_FP8_TFLOPS = 4500.0
FALLBACK_PEAKS = {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}


def load_peaks():
    path = os.path.join(REPO, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), 'measured'
    return dict(FALLBACK_PEAKS), 'fallback'


def committed_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed `ncu --set full` capture
    (profiles/traffic.json, written by tools/ncu_summary.py); None if that kernel has no capture."""
    path = os.path.join(REPO, 'profiles', 'traffic.json')
    if not os.path.exists(path):
        return None
    with open(path) as f:
        t = json.load(f).get(key)
    return None if t is None else int(t['dram_read_bytes'] + t['dram_write_bytes'])


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clocks / throttle reasons while the timed region runs: NVML in-process every ~2 ms (the timed region of
    the default run lasts ~10 ms, one `nvidia-smi` fork takes longer than that); falls back to forking nvidia-smi."""
    QUERY = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = int(visible.split(',')[index]) if visible and visible.split(',')[index].isdigit() else index
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._max = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self._nvml = pynvml
        except Exception:  # noqa: BLE001
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        sm = float(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM))
        try:
            mask = n.nvmlDeviceGetCurrentClocksEventReasons(self._h)
        except Exception:  # noqa: BLE001
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        flag = lambda bit: 'Active' if mask & bit else 'Not Active'   # noqa: E731
        try:
            watts = n.nvmlDeviceGetPowerUsage(self._h) / 1000.0
        except Exception:  # noqa: BLE001
            watts = 0.0
        return [str(sm), str(self._max), f'{watts:.0f}', flag(0x8), flag(0x40), flag(0x20), flag(0x4)]

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nvml is not None:
                    self.rows.append(self._sample_nvml())
                else:
                    out = subprocess.run(['nvidia-smi', f'--query-gpu={self.QUERY}', '--format=csv,noheader,nounits',
                                          '-i', str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.rows.append([c.strip() for c in out.split(',')])
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.002 if self._nvml is not None else 0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        mx = max((float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()), default=None)
        watts = sorted(float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace('.', '').isdigit())
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_min_mhz': sm[0] if sm else None, 'sm_max_mhz': mx,
                'reasons': sorted(reasons), 'samples': len(self.rows), 'power_w_median': watts[len(watts) // 2] if watts else None,
                'source': 'nvml' if self._nvml is not None else 'nvidia-smi'}


# ------------------------------------------------------------------------------------------------ the reference install
_REF = None


def import_reference():
    """The UNMODIFIED reference (oracle/_ref, built by oracle/build_ref.sh). `deep_gemm` inside this repository is our alias
    package, so the reference is imported from its install directory first and stays registered under its own name (bench.py
    itself only uses `deepgemm_b200`). Raises if it is not there (the caller reports `unavailable`)."""
    global _REF
    if _REF is not None:
        return _REF
    ref_root = os.path.join(REPO, 'oracle', '_ref')
    if not os.path.isdir(os.path.join(ref_root, 'deep_gemm')):
        raise RuntimeError('oracle/_ref is not built (oracle/build_ref.sh needs /root/reference)')
    os.environ.setdefault('DG_JIT_CACHE_DIR', f'/tmp/dg_ref_cache_{os.environ.get("LOCAL_RANK", "0")}')
    os.environ.setdefault('CUDA_HOME', '/usr/local/cuda')
    for k in [k for k in sys.modules if k == 'deep_gemm' or k.startswith('deep_gemm.')]:
        del sys.modules[k]
    sys.path.insert(0, ref_root)
    import deep_gemm as ref
    assert ref_root in ref.__file__, ref.__file__
    _REF = ref
    return _REF


def time_ab(fn_a, fn_b, iters, warmup=3):
    """Device time of two callables on the same stream, interleaved launch by launch (the order alternates every
    iteration), each preceded by an L2 flush and bracketed by CUDA events.
    Returns (median_a_ms, median_b_ms, min_a_ms, min_b_ms); fn_b may be None."""
    from deepgemm_b200.testing import flush_l2
    fns = [f for f in (fn_a, fn_b) if f is not None]
    for _ in range(warmup):
        for f in fns:
            f()
    torch.cuda.synchronize()
    evs = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in fns] for _ in range(iters)]
    for it in range(iters):
        order = range(len(fns)) if it % 2 == 0 else reversed(range(len(fns)))
        for j in order:
            flush_l2()
            evs[it][j][0].record()
            fns[j]()
            evs[it][j][1].record()
    torch.cuda.synchronize()
    out = []
    for j in range(len(fns)):
        ts = sorted(e[j][0].elapsed_time(e[j][1]) for e in evs)
        out.append((ts[len(ts) // 2], ts[0]))
    if fn_b is None:
        return out[0][0], None, out[0][1], None
    return out[0][0], out[1][0], out[0][1], out[1][1]


def kineto_us(fn, name, num_tests=10):
    """Mean kernel time by the profiler, the reference's own method (deep_gemm/testing/bench.py:79-146), in us."""
    from deepgemm_b200.testing import bench_kineto
    return round(bench_kineto(fn, name, num_tests=num_tests) * 1e6, 2)


# ------------------------------------------------------------------------------------------------ FP8 tensor peak
def fp8_peak_block(device):
    """Issue-only tcgen05.mma block-scaled FP8 probe (csrc/peak_probe.cuh): burst = best of 10 launches of ~1 ms,
    sustained = back-to-back launches for ~2 s with the SM clock sampled meanwhile."""
    from deepgemm_b200 import _lib
    lib = _lib.lib()
    sms = torch.cuda.get_device_properties(device).multi_processor_count & ~1
    stream = torch.cuda.current_stream().cuda_stream
    out = {}
    for n_, iters in ((256, 4096), (240, 4096)):
        flops = (sms // 2) * iters * 4 * 2.0 * 256 * n_ * 32
        for _ in range(3):
            _lib.check(lib.dgb200_debug_fp8_peak(n_, iters, sms, stream))
        torch.cuda.synchronize()
        best = float('inf')
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.check(lib.dgb200_debug_fp8_peak(n_, iters, sms, stream))
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        out[f'burst_tflops_n{n_}'] = round(flops / (best * 1e-3) / 1e12, 1)
        if n_ == 256:
            reps = max(1, int(2000.0 / best))
            with ClockSampler(torch.cuda.current_device()) as clocks:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    _lib.check(lib.dgb200_debug_fp8_peak(n_, iters, sms, stream))
                e1.record()
                torch.cuda.synchronize()
            out['sustained_tflops_n256'] = round(flops * reps / (e0.elapsed_time(e1) * 1e-3) / 1e12, 1)
            out['sustained_seconds'] = round(e0.elapsed_time(e1) * 1e-3, 2)
            out['sustained_clocks'] = clocks.summary()
    out['method'] = ('tcgen05.mma.cta_group::2.kind::mxf8f6f4.block_scale, UMMA 256xNx32, operands resident in shared memory '
                     '(random finite E4M3), one CTA pair per 2 SMs, no TMA / epilogue; FLOPs = pairs*iters*4*2*256*N*32')
    return out


# ------------------------------------------------------------------------------------------------ workloads
def make_dense_problem(m, n, k, device, seed):
    from deepgemm_b200.utils import per_block_cast_to_fp8, per_token_cast_to_fp8
    g = torch.Generator(device=device).manual_seed(seed)
    a = torch.randn((m, k), device=device, dtype=torch.bfloat16, generator=g)
    b = torch.randn((n, k), device=device, dtype=torch.bfloat16, generator=g)
    qa, qb = per_token_cast_to_fp8(a, True), per_block_cast_to_fp8(b, True)
    return a, qa, qb


def dense_step_setup(device, gemm, transform):
    """The four DeepSeek-V3 dense problems with packed scale factors for the implementation behind `gemm` / `transform`."""
    probs = []
    for i, (m, n, k) in enumerate(DENSE_SHAPES):
        a, qa, qb = make_dense_problem(m, n, k, device, seed=i)
        sfa = transform(qa[1], m, k, (1, 128, 128), None, True)
        sfb = transform(qb[1], n, k, (1, 128, 128), None, False)
        d = torch.empty((m, n), device=device, dtype=torch.bfloat16)
        probs.append(dict(m=m, n=n, k=k, a=a, qa=qa, qb=qb, sfa=sfa, sfb=sfb, d=d))
    return probs


RETIMED = None   # set by time_dense_step when the timed region had to be measured a second time


def time_dense_step(args, world, device, probs, gemm, on_first_call=None):
    """W warm-up steps, then exactly K timed steps; every launch preceded by an L2 flush and bracketed by CUDA events.
    Returns (per-shape mean ms, per-step ms lists, clock summary, wall seconds)."""
    from deepgemm_b200.testing import flush_l2

    def step(record=None):
        for i, p in enumerate(probs):
            flush_l2()
            if record is not None:
                record[i][0].record()
            gemm((p['qa'][0], p['sfa']), (p['qb'][0], p['sfb']), p['d'])
            if record is not None:
                record[i][1].record()
            elif on_first_call is not None:
                on_first_call(p)

    def timed_region(clocks):
        torch.cuda.synchronize()
        barrier(world)
        events = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in probs]
                  for _ in range(args.steps)]
        clocks.rows.clear()
        t0 = time.perf_counter()
        for s in range(args.steps):
            step(events[s])
        torch.cuda.synchronize()
        wall_ = time.perf_counter() - t0
        ms = [[e[i][0].elapsed_time(e[i][1]) for i in range(len(probs))] for e in events]
        return ms, wall_

    def stalled(ms):
        """A launch that took more than 3x the median of its shape: the host stalled between the event and the launch (the
        events bracket one kernel each, so the GPU sat idle inside the bracket). Seen once with 4 ranks on one box."""
        worst = 0.0
        for i in range(len(probs)):
            col = sorted(st[i] for st in ms)
            worst = max(worst, col[-1] / max(col[len(col) // 2], 1e-9))
        return worst

    global RETIMED
    RETIMED = None
    # the clock sampler starts before the warm-up: its start-up noise and the idle->busy clock ramp fall outside the timed region
    with ClockSampler(torch.cuda.current_device()) as clocks:
        for _ in range(args.warmup):
            step()
        per_step_ms, wall = timed_region(clocks)
        ratio = allreduce_max(stalled(per_step_ms), world, device)
        if os.environ.get('BENCH_FORCE_RETIME'):      # (test hook for the second-attempt path)
            ratio = 99.0
        if ratio > 3.0:
            # like a throttled run: rejected and re-measured ONCE, by every rank together; both attempts are reported
            first = sum(sum(st[i] for st in per_step_ms) / args.steps for i in range(len(probs)))
            per_step_ms, wall = timed_region(clocks)
            RETIMED = {'reason': 'a launch took %.1fx the median of its shape on some rank (host stall inside an event bracket); the K timed '
                                 'steps were measured again once' % ratio,
                       'first_attempt_ms_per_step_this_rank': round(first, 4),
                       'second_attempt_worst_over_median': round(allreduce_max(stalled(per_step_ms), world, device), 2)}
    barrier(world)
    per_shape_ms = [sum(st[i] for st in per_step_ms) / args.steps for i in range(len(probs))]
    return per_shape_ms, per_step_ms, clocks.summary(), wall


DUMP_LIMIT_BYTES = 64_000_000      # all files together, .npy headers included
NPY_HEADER_BYTES = 4096            # an upper bound of the header np.save writes for a 2-D array


def dump_outputs(out_dir, probs):
    """D of every dense problem to `out_dir`/d_<M>x<N>x<K>.npy in float32 (BF16 widens exactly). Smallest first, each file
    gets an equal share of what is left of 64 MB, so small outputs are written whole and what they leave goes to the larger
    ones; a D larger than its share keeps the rows of a sorted sample drawn with a fixed seed, the same rows in every run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_LIMIT_BYTES
    for i, p in enumerate(sorted(probs, key=lambda p_: p_['d'].numel())):
        d = p['d'].float().cpu()
        rows = (left // (len(probs) - i) - NPY_HEADER_BYTES) // (d.shape[1] * d.element_size())
        if rows < d.shape[0]:
            d = d[torch.randperm(d.shape[0], generator=torch.Generator().manual_seed(0))[:rows].sort().values]
        path = os.path.join(out_dir, f"d_{p['m']}x{p['n']}x{p['k']}.npy")
        np.save(path, d.numpy())
        left -= os.path.getsize(path)


def dense_ab_block(probs, dg, iters=20):
    """Per dense shape: ours vs the unmodified reference kernel, same tensors, same flush + CUDA-event method, interleaved."""
    try:
        ref = import_reference()
    except Exception as e:  # noqa: BLE001
        return {'unavailable': f'{type(e).__name__}: {e}'[:300]}
    rows = []
    for p in probs:
        m, n, k = p['m'], p['n'], p['k']
        try:
            sfa_r = ref.transform_sf_into_required_layout(p['qa'][1], m, k, (1, 128, 128), None, True)
            sfb_r = ref.transform_sf_into_required_layout(p['qb'][1], n, k, (1, 128, 128), None, False)
            d_ref, d_our = torch.empty_like(p['d']), torch.empty_like(p['d'])
            f_ref = lambda: ref.fp8_gemm_nt((p['qa'][0], sfa_r), (p['qb'][0], sfb_r), d_ref)   # noqa: E731
            f_our = lambda: dg.fp8_gemm_nt((p['qa'][0], p['sfa']), (p['qb'][0], p['sfb']), d_our)   # noqa: E731
            f_ref()                                                       # JIT compile (seconds, once per shape)
            torch.cuda.synchronize()
            dg.set_split_k(False)
            try:
                f_our()
                torch.cuda.synchronize()
                bitwise = bool(torch.equal(d_ref, d_our))
            finally:
                dg.set_split_k(True)
            f_our()
            torch.cuda.synchronize()
            default_mismatch = int((d_ref != d_our).sum())
            ours, refk, ours_min, ref_min = time_ab(f_our, f_ref, iters)
            k_our, k_ref = kineto_us(f_our, 'fp8_gemm_kernel'), kineto_us(f_ref, 'gemm_')
            rows.append({'m': m, 'n': n, 'k': k, 'ours_us': round(ours * 1e3, 2), 'ref_kernel_us': round(refk * 1e3, 2),
                         'speedup': round(refk / ours, 4), 'ours_min_us': round(ours_min * 1e3, 2), 'ref_min_us': round(ref_min * 1e3, 2),
                         'ours_kineto_us': k_our, 'ref_kineto_us': k_ref, 'speedup_kineto': round(k_ref / k_our, 4) if k_our else None,
                         'ours_tflops': round(2.0 * m * n * k / (ours * 1e-3) / 1e12, 1),
                         'ref_tflops': round(2.0 * m * n * k / (refk * 1e-3) / 1e12, 1),
                         'bitwise_equal': bitwise, 'default_config_mismatching_elements': default_mismatch})
        except Exception as e:  # noqa: BLE001
            rows.append({'m': m, 'n': n, 'k': k, 'unavailable': f'{type(e).__name__}: {e}'[:300]})
    ok = [r for r in rows if 'speedup' in r]
    return {'method': 'median of %d interleaved launches each (order alternating), L2 flushed (512 MB write) before every launch, CUDA events '
                      '(*_us: includes the launch gaps around one kernel); *_kineto_us: mean kernel time by torch.profiler, the reference\'s own '
                      'bench_kineto method; bitwise_equal with set_split_k(False), default_config_mismatching_elements with the default '
                      '(cluster split-K for M <= 256)' % iters,
            'reference': 'deepseek-ai/DeepGEMM sm100_fp8_fp4_gemm_1d1d (oracle/_ref, unmodified, NVCC JIT on this box)',
            'per_shape': rows, 'ours_ge_reference_on_every_shape': bool(ok) and all(r['speedup'] >= 1.0 for r in ok) and len(ok) == len(rows),
            'ours_ge_reference_on_every_shape_kineto': bool(ok) and all((r.get('speedup_kineto') or 0) >= 1.0 for r in ok) and len(ok) == len(rows)}


def run_dense(args, rank, world, device):
    import deepgemm_b200 as dg
    from deepgemm_b200 import _lib
    peaks, peak_kind = load_peaks()
    probs = dense_step_setup(device, dg.fp8_gemm_nt, dg.transform_sf_into_required_layout)

    def note_tile(p):
        if 'tile' not in p:
            cfg = _lib.last_config()
            p['tile'] = {k_: cfg[k_] for k_ in ('block_m', 'cluster', 'num_stages', 'num_splits', 'cluster_split', 'tma_store')}

    launches0 = _lib.launch_count()
    per_shape_ms, per_step_ms, clock_summary, t_wall = time_dense_step(args, world, device, probs, dg.fp8_gemm_nt, note_tile)
    retimed = RETIMED
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, probs)
    launches = (_lib.launch_count() - launches0) * args.steps // (args.steps + args.warmup)
    step_ms = allreduce_max(sum(per_shape_ms), world, device)
    flops = sum(2.0 * p['m'] * p['n'] * p['k'] for p in probs)
    value = flops * world / (step_ms * 1e-3) / 1e12

    # ---- FP8 tensor peak: the measured issue-only probe; the 2 x BF16 cuBLAS proxy stays beside it
    proxy_peak = 2.0 * peaks['bf16_tflops']
    try:
        peak_probe = fp8_peak_block(device) if rank == 0 or world == 1 else None
    except Exception as e:  # noqa: BLE001
        peak_probe = {'unavailable': f'{type(e).__name__}: {e}'[:300]}
    fp8_peak, peak_source = proxy_peak, f'2 x {peak_kind} bf16_tflops (MEASURED_PEAKS.json): FP8 probe unavailable'
    if peak_probe and 'burst_tflops_n256' in peak_probe:
        fp8_peak = peak_probe['burst_tflops_n256']
        peak_source = ('measured issue-only tcgen05.mma FP8 block-scaled burst on this GPU (fp8_peak.burst_tflops_n256); '
                       f'proxy 2 x {peak_kind} bf16_tflops = {proxy_peak:.1f}; nominal dense FP8 = {NOMINAL_FP8_TFLOPS}')
    if world > 1:
        fp8_peak = allreduce_max(fp8_peak if rank == 0 else 0.0, world, device)
    per_shape = []
    for p, ms in zip(probs, per_shape_ms):
        m, n, k = p['m'], p['n'], p['k']
        fl = 2.0 * m * n * k
        byts = m * k + n * k + m * n * 2 + (m + n) * ((k + 511) // 512) * 4
        tf, gbs = fl / (ms * 1e-3) / 1e12, byts / (ms * 1e-3) / 1e9
        bound = 'tensor' if fl / byts > fp8_peak * 1e12 / (peaks['hbm_gbs'] * 1e9) else 'hbm'
        frac = tf / fp8_peak if bound == 'tensor' else gbs / peaks['hbm_gbs']
        per_shape.append({'m': m, 'n': n, 'k': k, 'us': round(ms * 1e3, 2), 'tflops': round(tf, 1), 'gbs': round(gbs, 1),
                          'bound': bound, 'frac_of_' + peak_kind: round(frac, 4), 'tile': p['tile']})

    # dominant kernel of the step = the M=4096 launch (tensor bound)
    dom = per_shape[-1]
    roofline = {'bound': 'tensor', 'kernel': 'fp8_gemm_kernel<dense> M=4096 N=4096 K=7168',
                'achieved': dom['tflops'], 'peak': round(fp8_peak, 1), 'unit': 'TFLOP/s',
                'frac': round(dom['tflops'] / fp8_peak, 4), 'peak_source': peak_source,
                'frac_of_2x_bf16_proxy': round(dom['tflops'] / proxy_peak, 4),
                'frac_of_nominal': round(dom['tflops'] / NOMINAL_FP8_TFLOPS, 4), 'traffic': committed_traffic('dense_m4096'),
                'algorithmic_bytes': int(4096 * 7168 + 4096 * 7168 + 4096 * 4096 * 2 + 2 * 4096 * 14 * 4),
                'share_of_step': round(per_shape_ms[-1] / sum(per_shape_ms), 4)}

    # ---- end to end: pinned host buffers -> H2D -> quantise / pack -> GEMM -> D2H ---------------------------------
    e2e_ms, h2d, d2h = time_dense_e2e(args, world, device, probs,
                                      quantise=dg.per_token_cast_to_fp8_packed,
                                      pack_b=lambda sf, n, k: dg.transform_sf_into_required_layout(sf, n, k, (1, 128, 128), None, False),
                                      gemm=dg.fp8_gemm_nt)
    e2e_value = flops * world / (e2e_ms * 1e-3) / 1e12

    out = {
        'metric': 'FP8 TFLOPS over the DeepSeek-V3 dense shapes (sum 2MNK / sum kernel time)', 'value': round(value, 2),
        'unit': 'TFLOPS', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': round(step_ms, 4),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'fp8_e4m3 (fp32 accumulate, bf16 out)',
        'data': 'synthetic', 'impl': 'deepgemm_b200',
        'config': {'workload': 'dense fp8_gemm_nt M in {64,128,512,4096} N=4096 K=7168, 1x128/128x128 UE8M0 SF',
                   'l2': 'flushed (512 MB write) before every timed launch', 'parallelism': f'replicas x{world}',
                   **({'retimed': retimed} if retimed else {})},
        'per_shape': per_shape, 'roofline': roofline, 'clocks': clock_summary,
        'e2e': {'value': round(e2e_value, 3), 'unit': 'TFLOPS', 'ms_per_step': round(e2e_ms, 4),
                'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                'path': 'pinned host BF16 activations + FP8 weights/FP32 scales -> H2D -> CUDA quantiser (packed UE8M0) + weight-scale pack -> fp8_gemm_nt -> D2H'},
        'gpu_launches': int(launches), 'wall_ms_per_step_incl_flush': round(t_wall * 1e3 / args.steps, 3),
        'per_step_us': [[round(x * 1e3, 1) for x in st] for st in per_step_ms[:8]],
    }
    if peak_probe is not None:
        out['fp8_peak'] = peak_probe
    return out, probs


def next_rows_block(device, dg):
    """SURVEY section 8(f4) and the k-grouped row beside the reference's own kernels (same tensors, kernel time by the profiler):
    BF16-operand dense GEMMs, the k-grouped weight-gradient form for both operand types."""
    from deepgemm_b200.utils import per_channel_cast_to_fp8
    try:
        ref = import_reference()
    except Exception as e:  # noqa: BLE001
        return {'unavailable': f'{type(e).__name__}: {e}'[:300]}
    rows = []
    gen = torch.Generator(device=device).manual_seed(7)
    for (m, n, k) in [(64, 4096, 7168), (4096, 4096, 7168)]:
        a = torch.randn((m, k), device=device, dtype=torch.bfloat16, generator=gen)
        b = torch.randn((n, k), device=device, dtype=torch.bfloat16, generator=gen)
        d0, d1 = torch.empty((m, n), device=device, dtype=torch.bfloat16), torch.empty((m, n), device=device, dtype=torch.bfloat16)
        ref.bf16_gemm_nt(a, b, d0)
        dg.set_split_k(False)
        try:
            dg.bf16_gemm_nt(a, b, d1)
            torch.cuda.synchronize()
            bitwise = bool(torch.equal(d0, d1))
        finally:
            dg.set_split_k(True)
        rows.append({'op': 'bf16_gemm_nt', 'm': m, 'n': n, 'k': k, 'bitwise_equal': bitwise,
                     'ours_kineto_us': kineto_us(lambda: dg.bf16_gemm_nt(a, b, d1), 'fp8_gemm_kernel'),
                     'ref_kineto_us': kineto_us(lambda: ref.bf16_gemm_nt(a, b, d0), 'sm100_bf16')})
    g, m, n, ks = 4, 4096, 7168, [1024, 2048, 512, 4096]
    a = torch.randn((sum(ks), m), device=device, dtype=torch.bfloat16, generator=gen)
    b = torch.randn((sum(ks), n), device=device, dtype=torch.bfloat16, generator=gen)
    c = torch.randn((g, m, n), device=device, dtype=torch.float32, generator=gen)
    layout = torch.tensor(ks, device=device, dtype=torch.int32)
    d0, d1 = c.clone(), c.clone()
    ref.k_grouped_bf16_gemm_tn_contiguous(a, b, d0, ks, layout, c=d0)
    dg.k_grouped_bf16_gemm_tn_contiguous(a, b, d1, ks, layout, c=d1)
    torch.cuda.synchronize()
    rows.append({'op': 'k_grouped_bf16_gemm_tn_contiguous', 'groups': g, 'm': m, 'n': n, 'ks': ks, 'bitwise_equal': bool(torch.equal(d0, d1)),
                 'ours_kineto_us': kineto_us(lambda: dg.k_grouped_bf16_gemm_tn_contiguous(a, b, d1, ks, layout, c=d1), 'fp8_gemm_kernel', 5),
                 'ref_kineto_us': kineto_us(lambda: ref.k_grouped_bf16_gemm_tn_contiguous(a, b, d0, ks, layout, c=d0), 'sm100_bf16', 5)})
    qa, qb = per_channel_cast_to_fp8(a, True), per_channel_cast_to_fp8(b, True)
    del a, b
    d0.copy_(c), d1.copy_(c)
    ref.k_grouped_fp8_gemm_tn_contiguous(qa, qb, d0, ks, layout, c=d0)
    dg.k_grouped_fp8_gemm_tn_contiguous(qa, qb, d1, ks, layout, c=d1)
    torch.cuda.synchronize()
    rows.append({'op': 'k_grouped_fp8_gemm_tn_contiguous', 'groups': g, 'm': m, 'n': n, 'ks': ks, 'bitwise_equal': bool(torch.equal(d0, d1)),
                 'ours_kineto_us': kineto_us(lambda: dg.k_grouped_fp8_gemm_tn_contiguous(qa, qb, d1, ks, layout, c=d1), 'fp8_gemm_kernel', 5),
                 'ref_kineto_us': kineto_us(lambda: ref.k_grouped_fp8_gemm_tn_contiguous(qa, qb, d0, ks, layout, c=d0), 'sm100_fp8', 5)})
    return {'method': 'kernel time by torch.profiler (GEMM kernels selected by name; the k-grouped FP8 calls also run their scale-factor packing '
                      'kernels, not counted), L2 flushed before every launch; bitwise_equal with set_split_k(False)', 'rows': rows}


def add_dense_extras(out, probs, args, rank, world, device):
    """Outside the timed regions: the comparisons the north star is about (reference-kernel A/B, configs 3 / 4, config 5)."""
    import deepgemm_b200 as dg
    if rank == 0:
        out['vs_reference_kernel'] = guarded(lambda: dense_ab_block(probs, dg))
        try:    # the dominant kernel's share of the step by KERNEL time (what an ncu launch list shows: no event gaps)
            ks = [r['ours_kineto_us'] for r in out['vs_reference_kernel']['per_shape']]
            out['roofline']['share_of_step_by_kernel_time'] = round(ks[-1] / sum(ks), 4)
            out['roofline']['achieved_by_kernel_time'] = round(2.0 * 4096 * 4096 * 7168 / (ks[-1] * 1e-6) / 1e12, 1)
            out['roofline']['frac_by_kernel_time'] = round(out['roofline']['achieved_by_kernel_time'] / out['roofline']['peak'], 4)
        except Exception:  # noqa: BLE001
            pass
    probs.clear()
    torch.cuda.empty_cache()
    if rank == 0:
        out['decode_chain'] = guarded(lambda: decode_chain_block(device, dg))
    torch.cuda.empty_cache()
    if rank == 0:
        out['next_rows'] = guarded(lambda: next_rows_block(device, dg))
    torch.cuda.empty_cache()
    barrier(world)
    weights = None
    if rank == 0:
        out['grouped'], weights = grouped_blocks(device, dg)
    barrier(world)
    out_ep = guarded(lambda: ep_block(args, rank, world, device, dg, weights))
    if rank == 0:
        out['ep'] = out_ep


def time_dense_e2e(args, world, device, probs, quantise, pack_b, gemm):
    """The dense step through the public API from pinned HOST buffers: BF16 activations, FP8 weights + FP32 block scales.
    Every step copies them to the device, quantises the activations (packed UE8M0 out), packs the weight scales, runs the
    four GEMMs and reads every D back."""
    host = []
    for p in probs:
        host.append({'a': p['a'].cpu().pin_memory(), 'd': torch.empty((p['m'], p['n']), dtype=torch.bfloat16).pin_memory()})
    hb = probs[0]['qb'][0].view(torch.uint8).cpu().pin_memory()        # all four shapes share N, K: the weight matrix travels once per step
    hsfb = probs[0]['qb'][1].cpu().pin_memory()
    dev_a = [torch.empty_like(p['a']) for p in probs]
    dev_b, dev_sfb = torch.empty_like(probs[0]['qb'][0].view(torch.uint8)), torch.empty_like(probs[0]['qb'][1])
    h2d = hb.numel() + hsfb.numel() * 4 + sum(h['a'].numel() * 2 for h in host)
    d2h = sum(h['d'].numel() * 2 for h in host)
    n, k = probs[0]['n'], probs[0]['k']

    def step():
        dev_b.copy_(hb, non_blocking=True)
        dev_sfb.copy_(hsfb, non_blocking=True)
        sfb = pack_b(dev_sfb, n, k)
        for i, p in enumerate(probs):
            dev_a[i].copy_(host[i]['a'], non_blocking=True)
            qa = quantise(dev_a[i])
            gemm(qa, (dev_b.view(torch.float8_e4m3fn), sfb), p['d'])
            host[i]['d'].copy_(p['d'], non_blocking=True)

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    barrier(world)
    return allreduce_max(e0.elapsed_time(e1) / args.steps, world, device), h2d, d2h


def decode_chain_block(device, dg, layers=12, m=64, n=4096, k=7168, reps=8):
    """A decode micro-step: `layers` different weight matrices (12 x 29 MB > L2, so every GEMM streams its weights from HBM)
    applied back to back with M = 64 tokens, no flush and no event between the launches -- what the small-M kernel looks like
    inside a real step, where the ~4-5 us of launch gap around an isolated, event-timed launch disappear: plain stream order,
    programmatic dependent launch (set_pdl: the next GEMM's prologue and weight prefetch overlap this one's tail), and one CUDA
    graph of the chain. Per-GEMM time = total / launches; the reference's kernel runs the same chain."""
    from deepgemm_b200.utils import per_block_cast_to_fp8, per_token_cast_to_fp8
    peaks, peak_kind = load_peaks()
    gen = torch.Generator(device=device).manual_seed(5)
    a = torch.randn((m, k), device=device, dtype=torch.bfloat16, generator=gen)
    qa = per_token_cast_to_fp8(a, True)
    ws = [per_block_cast_to_fp8(torch.randn((n, k), device=device, dtype=torch.bfloat16, generator=gen), True) for _ in range(layers)]
    byts = m * k + n * k + m * n * 2 + (m + n) * ((k + 511) // 512) * 4
    out = {'workload': f'{layers} layers of fp8_gemm_nt {m}x{n}x{k} back to back ({layers * n * k / 1e6:.0f} MB of weights cycling through a 126 MB L2)',
           'hbm_roofline_us': round(byts / peaks['hbm_gbs'] / 1e3, 2)}

    def run(lib_mod, tag):
        sfa = lib_mod.transform_sf_into_required_layout(qa[1], m, k, (1, 128, 128), None, True)
        sfbs = [lib_mod.transform_sf_into_required_layout(w[1], n, k, (1, 128, 128), None, False) for w in ws]
        ds = [torch.empty((m, n), device=device, dtype=torch.bfloat16) for _ in range(layers)]

        def chain():
            for i in range(layers):
                lib_mod.fp8_gemm_nt((qa[0], sfa), (ws[i][0], sfbs[i]), ds[i])

        def timed(fn):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return round(e0.elapsed_time(e1) * 1e3 / (reps * layers), 2)

        res = {}
        for pdl in (False, True):
            lib_mod.set_pdl(pdl)
            try:
                res['pdl_us' if pdl else 'stream_us'] = timed(chain)
                chain()
                torch.cuda.synchronize()
                graph, side = torch.cuda.CUDAGraph(), torch.cuda.Stream()
                with torch.cuda.stream(side):
                    with torch.cuda.graph(graph, stream=side):
                        chain()
                res['graph_pdl_us' if pdl else 'graph_us'] = timed(graph.replay)
                del graph
            except Exception as e:  # noqa: BLE001
                res['pdl_error' if pdl else 'error'] = f'{type(e).__name__}: {e}'[:200]
            finally:
                lib_mod.set_pdl(False)
        best = min(v for v in res.values() if isinstance(v, float))
        res['best_us'] = best
        res['best_frac_of_hbm_roofline'] = round(out['hbm_roofline_us'] / best, 4)
        out[tag] = res

    run(dg, 'ours')
    try:
        run(import_reference(), 'reference')
        out['speedup_best'] = round(out['reference']['best_us'] / out['ours']['best_us'], 4)
    except Exception as e:  # noqa: BLE001
        out['reference'] = {'unavailable': f'{type(e).__name__}: {e}'[:300]}
    out['method'] = f'CUDA events around {reps} x {layers} launches, per-GEMM time = total / launches; no L2 flush needed: the weights exceed L2'
    return out


def guarded(fn):
    try:
        return fn()
    except Exception as e:  # noqa: BLE001
        import traceback
        return {'unavailable': f'{type(e).__name__}: {e}'[:300], 'where': traceback.format_exc().strip().splitlines()[-3:]}


# ------------------------------------------------------------------------------------------------ grouped workloads
def _grouped_weights(g, n, k, device, seed):
    """[G,N,K] FP8 weights + 128x128 scales, generated expert by expert to bound memory."""
    from deepgemm_b200.utils import per_block_cast_to_fp8
    gen = torch.Generator(device=device).manual_seed(seed)
    b = torch.empty((g, n, k), device=device, dtype=torch.float8_e4m3fn)
    sfb = torch.empty((g, (n + 127) // 128, (k + 127) // 128), device=device, dtype=torch.float32)
    for i in range(g):
        b[i], sfb[i] = per_block_cast_to_fp8(torch.randn((n, k), device=device, dtype=torch.bfloat16, generator=gen), True)
    return b, sfb


def _time_events(fn, steps, warmup, world):
    from deepgemm_b200.testing import flush_l2
    for _ in range(warmup):
        fn()
    barrier(world)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for s0, s1 in evs:
        flush_l2()
        s0.record()
        fn()
        s1.record()
    barrier(world)
    return sum(a.elapsed_time(b) for a, b in evs) / steps


def build_grouped_problem(kind, device, dg, mean_m, weights=None, seed=0):
    """BASELINE config 3 (`contiguous`) / 4 (`masked`). Returns a dict with `ours` (callable), the tensors the reference
    needs, and the algorithmic work."""
    import random
    from deepgemm_b200.utils import per_token_cast_to_fp8
    rnd = random.Random(seed)
    g = 256
    if kind == 'masked':
        m_max, n, k = 128, 7168, 2048
    else:
        n, k = 4096, 7168
    b, sfb = weights if weights is not None else _grouped_weights(g, n, k, device, seed=0)
    sfb_p = dg.transform_sf_into_required_layout(sfb, n, k, (1, 128, 128), g, False)
    if kind == 'masked':
        a = torch.randn((g * m_max, k), device=device, dtype=torch.bfloat16)
        q = per_token_cast_to_fp8(a, True)
        del a
        qa = (q[0].view(g, m_max, k), q[1].view(g, m_max, -1))
        sfa = dg.transform_sf_into_required_layout(qa[1], m_max, k, (1, 128, 128), g, True)
        counts = torch.tensor([min(m_max, int(mean_m * rnd.uniform(0.7, 1.3))) for _ in range(g)], device=device, dtype=torch.int32)
        d = torch.zeros((g, m_max, n), device=device, dtype=torch.bfloat16)
        valid = int(counts.sum())
        expected_m = int(1.2 * mean_m)
        call = lambda: dg.m_grouped_fp8_gemm_nt_masked((qa[0], sfa), (b, sfb_p), d, counts, expected_m)  # noqa: E731
        call()
        graph, side = torch.cuda.CUDAGraph(), torch.cuda.Stream()
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                call()
        return dict(kind=kind, ours=graph.replay, ours_eager=call, qa=qa, b=b, sfb=sfb, d=d, counts=counts, expected_m=expected_m,
                    valid=valid, rows_total=valid, g=g, n=n, k=k, m_max=m_max, _graph=graph,
                    name=f'masked grouped decode (CUDA graph replay), G=256 M_max=128 N=7168 K=2048 mean_m={mean_m}')
    alignment = dg.get_mk_alignment_for_contiguous_layout()
    ms = [int(mean_m * rnd.uniform(0.7, 1.3)) for _ in range(g)]
    aligned = [(x + alignment - 1) // alignment * alignment for x in ms]
    m = sum(aligned)
    a = torch.randn((m, k), device=device, dtype=torch.bfloat16)
    layout = torch.empty(m, dtype=torch.int32)
    s0 = 0
    for i, (mi, ai) in enumerate(zip(ms, aligned)):
        layout[s0:s0 + mi] = i
        layout[s0 + mi:s0 + ai] = -1
        s0 += ai
    layout = layout.to(device)
    a[layout < 0] = 0
    qa = per_token_cast_to_fp8(a, True)
    del a
    sfa = dg.transform_sf_into_required_layout(qa[1], m, k, (1, 128, 128), None, True)
    d = torch.empty((m, n), device=device, dtype=torch.bfloat16)
    fn = lambda: dg.m_grouped_fp8_gemm_nt_contiguous((qa[0], sfa), (b, sfb_p), d, layout)  # noqa: E731
    return dict(kind=kind, ours=fn, qa=qa, b=b, sfb=sfb, d=d, layout=layout, valid=sum(ms), rows_total=m, g=g, n=n, k=k,
                name=f'm_grouped contiguous prefill, G=256 N=4096 K=7168 mean_m={mean_m} (sum M={m}, valid {sum(ms)}, alignment {alignment})')


def grouped_reference_fn(p):
    """The unmodified reference on the same tensors (its own SF transform; masked: under its own CUDA graph)."""
    ref = import_reference()
    g, n, k = p['g'], p['n'], p['k']
    sfb_r = ref.transform_sf_into_required_layout(p['sfb'], n, k, (1, 128, 128), g, False)
    d_ref = torch.zeros_like(p['d'])
    if p['kind'] == 'masked':
        sfa_r = ref.transform_sf_into_required_layout(p['qa'][1], p['m_max'], k, (1, 128, 128), g, True)
        call = lambda: ref.m_grouped_fp8_gemm_nt_masked((p['qa'][0], sfa_r), (p['b'], sfb_r), d_ref, p['counts'], p['expected_m'])  # noqa: E731
        call()
        torch.cuda.synchronize()
        graph, side = torch.cuda.CUDAGraph(), torch.cuda.Stream()
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                call()
        p['_ref_graph'] = graph
        return graph.replay, d_ref
    sfa_r = ref.transform_sf_into_required_layout(p['qa'][1], p['rows_total'], k, (1, 128, 128), None, True)
    ref.set_mk_alignment_for_contiguous_layout(128)
    call = lambda: ref.m_grouped_fp8_gemm_nt_contiguous((p['qa'][0], sfa_r), (p['b'], sfb_r), d_ref, p['layout'])  # noqa: E731
    call()
    torch.cuda.synchronize()
    return call, d_ref


def grouped_line(p, ms_step, peaks, peak_kind):
    g, n, k = p['g'], p['n'], p['k']
    rows = p['rows_total']
    flops = 2.0 * p['valid'] * n * k
    # A (as laid out, padding included: it is loaded with its tile) + weights + D rows actually written (valid rows: the
    # contiguous kernel leaves padding groups alone, the masked one never touches rows >= masked_m) + packed scale factors
    byts = rows * k + g * n * k + p['valid'] * n * 2 + (rows + g * n) * ((k + 511) // 512) * 4
    gbs = byts / (ms_step * 1e-3) / 1e9
    return {'workload': p['name'], 'us': round(ms_step * 1e3, 1), 'tokens_per_s': round(p['valid'] / (ms_step * 1e-3), 1),
            'tflops': round(flops / (ms_step * 1e-3) / 1e12, 1),
            'roofline': {'bound': 'hbm', 'achieved': round(gbs, 1), 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                         'frac': round(gbs / peaks['hbm_gbs'], 4), 'peak_source': peak_kind + ' hbm_gbs (MEASURED_PEAKS.json)',
                         'algorithmic_bytes': int(byts), 'traffic': committed_traffic('contiguous_g256_m128' if p['kind'] != 'masked' else 'masked_g256_m64')}}


def grouped_blocks(device, dg, iters=10):
    """Configs 3 and 4 beside the reference kernel (rank 0, outside the dense timed region). Returns (block, weights of the
    contiguous problem for reuse by the 1-GPU EP step)."""
    from deepgemm_b200 import _lib
    peaks, peak_kind = load_peaks()
    out, keep = {}, None
    for kind, mean_m in (('contiguous', 128), ('masked', 64)):
        try:
            p = build_grouped_problem(kind, device, dg, mean_m)
            p['ours']()
            torch.cuda.synchronize()
            tile = _lib.last_config()
            try:
                f_ref, d_ref = grouped_reference_fn(p)
                ref_err = None
            except Exception as e:  # noqa: BLE001
                f_ref, d_ref, ref_err = None, None, f'{type(e).__name__}: {e}'[:300]
            ours, refk, ours_min, ref_min = time_ab(p['ours'], f_ref, iters)
            line = grouped_line(p, ours, peaks, peak_kind)
            line['tile'] = tile
            if f_ref is not None:
                p['ours']()
                f_ref()
                torch.cuda.synchronize()
                if kind == 'masked':
                    rows = torch.arange(p['m_max'], device=device).unsqueeze(0) < p['counts'].unsqueeze(1)
                    same = bool(torch.equal(p['d'][rows], d_ref[rows]))
                else:
                    same = bool(torch.equal(p['d'][p['layout'] >= 0], d_ref[p['layout'] >= 0]))
                k_our, k_ref = kineto_us(p['ours'], 'fp8_gemm_kernel', 5), kineto_us(f_ref, 'gemm_', 5)
                line.update({'ref_kernel_us': round(refk * 1e3, 1), 'speedup': round(refk / ours, 4), 'ours_min_us': round(ours_min * 1e3, 1),
                             'ref_min_us': round(ref_min * 1e3, 1), 'ours_kineto_us': k_our, 'ref_kineto_us': k_ref,
                             'speedup_kineto': round(k_ref / k_our, 4) if k_our else None, 'bitwise_equal_valid_rows': same})
            else:
                line['reference'] = {'unavailable': ref_err}
            out[kind] = line
            if kind == 'contiguous':
                keep = (p['b'], p['sfb'])
            p.pop('_graph', None), p.pop('_ref_graph', None)
            del p, d_ref, f_ref
        except Exception as e:  # noqa: BLE001
            out[kind] = {'unavailable': f'{type(e).__name__}: {e}'[:300]}
        torch.cuda.empty_cache()
    out['method'] = f'median of {iters} interleaved launches each (ours, reference), L2 flushed before every launch, CUDA events'
    return out, keep


def run_grouped(args, rank, world, device):
    """`--workload contiguous|masked`: BASELINE configs 3 / 4 as the headline line (HBM-bound: roofline = algorithmic bytes /
    measured HBM copy bandwidth)."""
    import deepgemm_b200 as dg
    from deepgemm_b200 import _lib
    peaks, peak_kind = load_peaks()
    masked = args.workload == 'masked'
    p = build_grouped_problem(args.workload, device, dg, args.mean_m or (64 if masked else 128))
    launches0 = _lib.launch_count()
    with ClockSampler(torch.cuda.current_device()) as clocks:
        ms_step = _time_events(p['ours'], args.steps, args.warmup, world)
    ms_step = allreduce_max(ms_step, world, device)
    launches = (_lib.launch_count() - launches0) if not masked else args.steps + args.warmup  # graph replays relaunch the kernel
    line = grouped_line(p, ms_step, peaks, peak_kind)
    return {
        'metric': 'grouped FP8 GEMM tokens/s (valid rows / kernel time)', 'value': round(p['valid'] * world / (ms_step * 1e-3), 1),
        'unit': 'tokens/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': round(ms_step, 4),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'fp8_e4m3 (fp32 accumulate, bf16 out)',
        'data': 'synthetic', 'impl': 'deepgemm_b200', 'tflops': line['tflops'],
        'config': {'workload': p['name'], 'l2': 'flushed (512 MB write) before every timed launch', 'parallelism': f'replicas x{world}',
                   'tile': _lib.last_config()},
        'roofline': line['roofline'], 'clocks': clocks.summary(), 'gpu_launches': int(launches),
        'e2e': {'value': None, 'unit': 'tokens/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0,
                'note': 'grouped workloads keep the 7.5 / 3.8 GB of expert weights resident; see the dense workload for e2e'},
    }


# ------------------------------------------------------------------------------------------------ expert-sharded step
def ep_step_timing(steps, warmup, world, device, dg, buf, xq, sf_packed, ids, wq, sfb_p, n, group_world):
    """dispatch -> grouped GEMM -> weighted combine on `buf`; per-phase CUDA-event times, max over the ranks of
    `group_world` (1 = this rank alone)."""
    t_local = xq.shape[0]
    d = buf.output(n)
    token_row = torch.empty(t_local, dtype=torch.int32, device=device)
    out_tokens = torch.empty((t_local, n), device=device, dtype=torch.bfloat16)

    def step(ev=None):
        if ev:
            ev[0].record()
        r = buf.dispatch(xq, sf_packed, ids, token_row)
        if ev:
            ev[1].record()
        buf.grouped_gemm((wq, sfb_p), d, r.expected_m, overlap=False)
        if ev:
            ev[2].record()
        buf.combine(token_row, ids, out_tokens)
        if ev:
            ev[3].record()

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    assert not buf.overflowed(), 'dispatch buffer capacity exceeded'
    barrier(group_world)
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(steps)]
    for e in evs:
        step(e)
    torch.cuda.synchronize()
    barrier(group_world)
    mean = lambda i, j: sum(e[i].elapsed_time(e[j]) for e in evs) / steps  # noqa: E731
    res = {'dispatch_ms': mean(0, 1), 'gemm_ms': mean(1, 2), 'combine_ms': mean(2, 3), 'step_ms': mean(0, 3)}
    if group_world > 1:
        res = {k_: allreduce_max(v, group_world, device) for k_, v in res.items()}
    return res


def ep_problem(rank, world, device, dg, g, n, k, tokens_total, weights=None):
    from deepgemm_b200.utils import per_token_cast_to_fp8
    epr, t_local = g // world, tokens_total // world
    if weights is not None and weights[0].shape[0] == epr:
        b, sfb = weights
    else:
        b, sfb = _grouped_weights(epr, n, k, device, seed=1000 + rank)
    sfb_p = dg.transform_sf_into_required_layout(sfb, n, k, (1, 128, 128), epr, False)
    gen = torch.Generator(device=device).manual_seed(rank)
    x = torch.randn((t_local, k), device=device, dtype=torch.bfloat16, generator=gen)
    xq, sf_packed = per_token_cast_to_fp8(x, True, 128, use_packed_ue8m0=True)
    ids = torch.randint(0, g, (t_local,), device=device, generator=gen)
    align = dg.get_mk_alignment_for_contiguous_layout()
    # capacity: balanced routing + 25% head room + alignment padding (a production caller sizes for its worst case)
    capacity = (int(t_local * 1.25) + epr * align + 127) // 128 * 128
    return b, sfb_p, xq, sf_packed, ids, capacity


def ep_block(args, rank, world, device, dg, weights_1gpu=None, steps=10, warmup=3):
    """BASELINE config 5 at this run's world size: 256 experts sharded over the ranks, 32768 tokens (top-1), N=4096, K=7168.
    One step = peer-memory dispatch (one persistent kernel) + local grouped GEMM + combine over NVLink. For world > 1 rank 0
    also runs the same 32768 tokens on one GPU so that the strong-scaling efficiency is in the line."""
    from deepgemm_b200 import ep
    g, n, k, tokens_total = 256, 4096, 7168, 32768
    res = {'workload': f'expert-sharded grouped GEMM: 256 experts over {world} GPU(s), 32768 tokens top-1, N=4096 K=7168; '
                       'step = dispatch (NVLink peer stores into the owner\'s GEMM buffer) + grouped GEMM + combine',
           'steps': steps, 'warmup': warmup, 'parallelism': f'ep{world}', 'scaling': 'strong'}
    b, sfb_p, xq, sf_packed, ids, capacity = ep_problem(rank, world, device, dg, g, n, k, tokens_total, weights_1gpu if world == 1 else None)
    buf = ep.EpBuffer(g, capacity, k)
    try:
        t = ep_step_timing(steps, warmup, world, device, dg, buf, xq, sf_packed, ids, b, sfb_p, n, world)
    finally:
        buf.close()
    del b, sfb_p, xq, sf_packed, ids
    torch.cuda.empty_cache()
    res.update({k_: round(v, 4) for k_, v in t.items()})
    res['tokens_per_s'] = round(tokens_total / (t['step_ms'] * 1e-3), 1)
    res['tflops'] = round(2.0 * tokens_total * n * k / (t['step_ms'] * 1e-3) / 1e12, 1)
    row_bytes = k + 4 * ((k + 511) // 512)
    res['dispatch_wire_bytes_per_rank'] = int(tokens_total // world * row_bytes)
    res['dispatch_remote_bytes_per_rank'] = int(tokens_total // world * row_bytes * (world - 1) / world)
    if world > 1:
        # the 1-GPU step of the same problem, on rank 0 alone (the others wait at the barrier below)
        one = None
        if rank == 0:
            b1, sfb1, xq1, sf1, ids1, cap1 = ep_problem(0, 1, device, dg, g, n, k, tokens_total)
            buf1 = ep.EpBuffer(g, cap1, k, local_only=True)
            try:
                one = ep_step_timing(steps, warmup, 1, device, dg, buf1, xq1, sf1, ids1, b1, sfb1, n, 1)
            finally:
                buf1.close()
            del b1, sfb1, xq1, sf1, ids1
            torch.cuda.empty_cache()
        barrier(world)
        if rank == 0:
            res['n1'] = {k_: round(v, 4) for k_, v in one.items()}
            res['speedup_vs_n1'] = round(one['step_ms'] / t['step_ms'], 3)
            res['efficiency_vs_n1'] = round(one['step_ms'] / t['step_ms'] / world, 4)
            res['gemm_efficiency_vs_n1'] = round(one['gemm_ms'] / t['gemm_ms'] / world, 4)
    else:
        res['speedup_vs_n1'], res['efficiency_vs_n1'] = 1.0, 1.0
    return res


def run_ep(args, rank, world, device):
    """`--workload ep`: BASELINE config 5 as the headline line."""
    import deepgemm_b200 as dg
    from deepgemm_b200 import _lib
    launches0 = _lib.launch_count()
    with ClockSampler(torch.cuda.current_device()) as clocks:
        blk = ep_block(args, rank, world, device, dg, None, steps=args.steps, warmup=args.warmup)
    launches = _lib.launch_count() - launches0
    peaks, peak_kind = load_peaks()
    total = blk['step_ms']
    gbs = 2.0 * blk['dispatch_wire_bytes_per_rank'] / (blk['dispatch_ms'] * 1e-3) / 1e9 if blk['dispatch_ms'] > 0 else 0.0
    return {
        'metric': 'expert-sharded grouped FP8 GEMM tokens/s (dispatch + GEMM + combine)', 'value': blk['tokens_per_s'],
        'unit': 'tokens/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': round(total, 4),
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'fp8_e4m3 (fp32 accumulate, bf16 out)',
        'data': 'synthetic', 'impl': 'deepgemm_b200',
        'config': {'workload': blk['workload'], 'parallelism': f'ep{world}', 'l2': 'inputs (>= 0.9 GB of expert weights per rank) exceed L2'},
        'ep': blk,
        'roofline': {'kernel': 'ep::dispatch_fused_kernel', 'bound': 'hbm', 'achieved': round(gbs, 1),
                     'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': round(gbs / peaks['hbm_gbs'], 4),
                     'peak_source': peak_kind + ' hbm_gbs (MEASURED_PEAKS.json)', 'traffic': None,
                     'note': 'algorithmic bytes = read + write of every local token row once; the remote share crosses NVLink (770 GB/s per direction measured)'},
        'clocks': clocks.summary(), 'gpu_launches': int(launches),
        'e2e': {'value': blk['tokens_per_s'], 'unit': 'tokens/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0,
                'note': 'tokens originate on the GPUs (output of the previous layer); nothing crosses PCIe in this path'},
    }


# ------------------------------------------------------------------------------------------------ reference arm
def cpu_reference_step(shapes, threads):
    """torch-CPU BF16-emulated blockwise GEMM (oracle port) over `shapes`; returns (seconds, flops)."""
    from deepgemm_b200.utils import per_block_cast_to_fp8, per_token_cast_to_fp8
    from oracle import blockwise
    torch.set_num_threads(threads)
    total, flops = 0.0, 0.0
    for i, (m, n, k) in enumerate(shapes):
        g = torch.Generator().manual_seed(i)
        a = torch.randn((m, k), generator=g).to(torch.bfloat16)
        b = torch.randn((n, k), generator=g).to(torch.bfloat16)
        qa, qb = per_token_cast_to_fp8(a, True), per_block_cast_to_fp8(b, True)
        best = float('inf')
        for _ in range(2):
            t0 = time.perf_counter()
            blockwise.bf16_emulated_gemm_nt(qa, qb)
            best = min(best, time.perf_counter() - t0)
        total += best
        flops += 2.0 * m * n * k
    return total, flops


def cpu_baseline_block():
    threads = os.cpu_count() or 1
    sample = DENSE_SHAPES[:3]
    saved = None
    try:        # the process is bound to the GPU's NUMA node for the end-to-end leg; the CPU baseline gets every core back
        saved = os.sched_getaffinity(0)
        os.sched_setaffinity(0, range(threads))
    except Exception:  # noqa: BLE001
        saved = None
    try:
        sec, fl = cpu_reference_step(sample, threads)
    finally:
        if saved:
            try:
                os.sched_setaffinity(0, saved)
            except Exception:  # noqa: BLE001
                pass
    return {'value': round(fl / sec / 1e12, 4), 'unit': 'TFLOPS', 'cores': threads, 'kind': 'port',
            'sample': 'M in {64,128,512} of the dense step (N=4096, K=7168), dequantise-to-BF16 + torch.matmul, best of 2',
            'seconds': round(sec, 3)}


def run_reference_arm_gpu(args, rank, world, device):
    """The UNMODIFIED reference (oracle/_ref) through its own public API on the same step, same method: kernel-only `value`
    (its SM100 kernel with its own packed scale factors) and `e2e` from pinned host buffers (its Python quantiser path:
    FP8 + FP32 scales on the host -> H2D -> its own SF transform + GEMM -> D2H)."""
    ref = import_reference()
    probs = dense_step_setup(device, ref.fp8_gemm_nt, ref.transform_sf_into_required_layout)
    per_shape_ms, per_step_ms, clock_summary, _ = time_dense_step(args, world, device, probs, ref.fp8_gemm_nt)
    retimed = RETIMED
    step_ms = allreduce_max(sum(per_shape_ms), world, device)
    flops = sum(2.0 * p['m'] * p['n'] * p['k'] for p in probs)
    value = flops * world / (step_ms * 1e-3) / 1e12
    # e2e: the reference has no CUDA activation quantiser; its callers quantise with the torch helpers of deep_gemm.utils.
    from deepgemm_b200.utils import per_token_cast_to_fp8 as torch_quantiser   # bit-identical restatement of the reference's helper
    e2e_ms, h2d, d2h = time_dense_e2e(args, world, device, probs,
                                      quantise=lambda a: torch_quantiser(a, True),
                                      pack_b=lambda sf, n, k: sf, gemm=ref.fp8_gemm_nt)
    return {
        'impl': 'reference', 'metric': 'FP8 TFLOPS over the DeepSeek-V3 dense shapes (sum 2MNK / sum kernel time)',
        'value': round(value, 2), 'unit': 'TFLOPS', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': round(step_ms, 4), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'fp8_e4m3 (fp32 accumulate, bf16 out)', 'data': 'synthetic',
        'reference': 'deepseek-ai/DeepGEMM, unmodified, oracle/_ref: deep_gemm.fp8_gemm_nt -> sm100_fp8_fp4_gemm_1d1d (NVCC JIT on this box)',
        'config': {'workload': 'dense fp8_gemm_nt M in {64,128,512,4096} N=4096 K=7168, 1x128/128x128 UE8M0 SF',
                   'l2': 'flushed (512 MB write) before every timed launch', 'parallelism': f'replicas x{world}',
                   **({'retimed': retimed} if retimed else {})},
        'per_shape': [{'m': p['m'], 'n': p['n'], 'k': p['k'], 'us': round(ms * 1e3, 2),
                       'tflops': round(2.0 * p['m'] * p['n'] * p['k'] / (ms * 1e-3) / 1e12, 1)} for p, ms in zip(probs, per_shape_ms)],
        'clocks': clock_summary,
        'e2e': {'value': round(flops * world / (e2e_ms * 1e-3) / 1e12, 3), 'unit': 'TFLOPS', 'ms_per_step': round(e2e_ms, 4),
                'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                'path': 'pinned host BF16 activations + FP8 weights/FP32 scales -> H2D -> torch quantiser (deep_gemm.utils.per_token_cast_to_fp8) -> deep_gemm.fp8_gemm_nt (its own SF transform) -> D2H'},
        'gpu_launches': 0,
    }


def run_reference_arm_cpu(args, why):
    threads = os.cpu_count() or 1
    sample = DENSE_SHAPES[:3]
    for _ in range(min(args.warmup, 1)):
        cpu_reference_step(sample[:1], threads)
    times = []
    fl = 0.0
    for _ in range(args.steps):
        sec, fl = cpu_reference_step(sample, threads)
        times.append(sec)
    sec = sum(times) / len(times)
    v = round(fl / sec / 1e12, 4)
    return {
        'impl': 'reference', 'metric': 'FP8 TFLOPS over the DeepSeek-V3 dense shapes (sum 2MNK / sum kernel time)',
        'value': v, 'unit': 'TFLOPS', 'n_gpus': 1, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': round(sec * 1e3, 3), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'bf16 emulation of fp8_e4m3 x ue8m0 (fp32 accumulate)', 'data': 'synthetic',
        'config': {'workload': 'dense fp8_gemm_nt M in {64,128,512,4096} N=4096 K=7168, 1x128/128x128 UE8M0 SF',
                   'sample': 'bounded: M in {64,128,512} per step'},
        'reference_kernel_unavailable': why,
        'cpu_baseline': {'value': v, 'unit': 'TFLOPS', 'cores': threads, 'kind': 'port',
                         'sample': 'M in {64,128,512} of the dense step, torch CPU BF16 matmul of the dequantised operands'},
        'e2e': {'value': v, 'unit': 'TFLOPS', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }


# ------------------------------------------------------------------------------------------------ distributed glue
def barrier(world):
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()


def allreduce_max(x, world, device):
    if world == 1:
        return x
    t = torch.tensor([x], device=device, dtype=torch.float64)
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item())


def bind_to_gpu_numa_node(local_rank):
    """Run this process on the CPUs next to its GPU (NVML's ideal affinity) before any pinned host buffer is allocated: the end-to-
    end leg is PCIe-bound, and the same 137 MB per step took 2.8 ms on one box and 4.3 ms on another depending on where the
    process and its pinned pages happened to sit. Both arms do this; failures are ignored (it only steadies the measurement)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get('CUDA_VISIBLE_DEVICES')
        phys = int(vis.split(',')[local_rank]) if vis and all(v.strip().isdigit() for v in vis.split(',')) else local_rank
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(phys))
        return True
    except Exception:  # noqa: BLE001
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='dense', choices=['dense', 'contiguous', 'masked', 'ep'])
    ap.add_argument('--mean-m', type=int, default=0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='dense workload: skip the reference A/B, grouped and EP blocks')
    ap.add_argument('--extras-timeout', type=float, default=420.0)
    ap.add_argument('--dump-outputs', metavar='DIR', help='dense workload: write what the last timed step computed to DIR')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.workload != 'dense' or args.impl != 'ours'):
        ap.error('--dump-outputs covers the dense workload of --impl ours')
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))

    if args.impl == 'reference' and not torch.cuda.is_available():
        if rank == 0:
            print(json.dumps(run_reference_arm_cpu(args, 'no CUDA device')), flush=True)
        return
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (the FP8 GEMM path has no CPU fallback)')
    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    bind_to_gpu_numa_node(local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        torch.distributed.init_process_group(backend='nccl', device_id=device)

    if args.impl == 'reference':
        try:
            import_reference()
            why = None
        except Exception as e:  # noqa: BLE001
            why = f'{type(e).__name__}: {e}'[:300]
        if why is None:
            out = run_reference_arm_gpu(args, rank, world, device)
            if rank == 0 and not args.no_cpu_baseline:
                out['cpu_baseline'] = cpu_baseline_block()
        else:
            out = run_reference_arm_cpu(args, why) if rank == 0 else None
    else:
        if args.workload == 'dense':
            out, probs = run_dense(args, rank, world, device)
            if rank == 0 and not args.no_cpu_baseline:
                out['cpu_baseline'] = cpu_baseline_block()
            if not args.no_extras:
                # The extra blocks JIT-compile the reference and run multi-rank handshakes: if any of it wedges, the line
                # measured above must still come out. A watchdog prints it and leaves.
                def bail():
                    if rank == 0:
                        out.setdefault('extras', {'unavailable': f'watchdog: extra blocks exceeded {args.extras_timeout} s'})
                        print(json.dumps(out), flush=True)
                    os._exit(0)
                dog = threading.Timer(args.extras_timeout, bail)
                dog.daemon = True
                dog.start()
                add_dense_extras(out, probs, args, rank, world, device)
                dog.cancel()
        else:
            out = {'contiguous': run_grouped, 'masked': run_grouped, 'ep': run_ep}[args.workload](args, rank, world, device)
    if rank == 0 and out is not None:
        print(json.dumps(out), flush=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == '__main__':
    main()
