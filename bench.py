#!/usr/bin/env python
"""bench.py — the scoring hot path of DeepRecommendation on B200, measured per BASELINE.json.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload all|attention|graph|basic] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Prints ONE JSON line (rank 0).  Headline = BASELINE.json configs[1]: AttentionNCF scoring on the MovieLens-latest-small
shape, one step = one batch of 512 (user, item) pairs through `AttentionNCF.forward(candidate_items, rated_items,
user_matrix)`; `value` = pairs/s with inputs resident in HBM, `e2e` = the same call fed from pinned host buffers with
the result read back.  `also` carries the other two metric legs: GraphNCF propagation (configs[2], MovieLens-25M shape,
directed-edge messages/s = 2·E·L / time) and BasicNCF scoring (configs[0] shape).  Everything is fp32 ("parity mode",
rel <= 1e-5 vs the reference).  Data is synthetic (deeprecommendation_b200/synth.py) — no dataset ships with the
reference and there is no network.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 512
F = 2094


def _peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return {'hbm_gbs': d['hbm_gbs'], 'bf16_tflops': d.get('bf16_tflops', 1590.0), 'bf16_tflops_sustained': d.get('bf16_tflops_sustained', 1400.0),
                'src': 'measured (MEASURED_PEAKS.json)'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'src': 'fallback (B200_PROFILING.md)'}


def _traffic(name):
    p = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(p):
        return json.load(open(p)).get(name)
    return None


# ----------------------------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, gpu_index):
        self.gpu, self.f, self.p = gpu_index, None, None

    def __enter__(self):
        if int(os.environ.get('RANK', '0')) != 0:      # NVML queries take driver locks: one sampler per job, not per rank
            return self
        try:
            self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
            self.p = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '200', '-i',
                                       str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        return self

    def __exit__(self, *exc):
        if self.p is not None:
            time.sleep(0.15)
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except Exception:
                self.p.kill()
        return False

    def summary(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        if self.f is None:
            return out
        try:
            self.f.flush()
            rows = [r.strip().split(', ') for r in open(self.f.name).read().strip().splitlines() if r.strip()]
            os.unlink(self.f.name)
            sm = [float(r[1]) for r in rows]
            power = [float(r[3]) for r in rows if r[3].replace('.', '', 1).isdigit()]
            busy = [s for s, r in zip(sm, rows) if (not power) or float(r[3]) > 0.5 * max(power)] or sm
            out['sm_mhz'] = float(np.median(busy)) if busy else None
            out['sm_max_mhz'] = float(rows[0][2]) if rows else None
            out['samples'] = len(rows)
            names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
            out['reasons'] = [n for k, n in enumerate(names) if any(r[4 + k].strip().lower().startswith('active') for r in rows)]
        except Exception as e:   # clocks are evidence, never a reason to lose the measurement
            out['error'] = repr(e)
        return out


def bind_to_gpu_numa(gpu_index):
    """Pin this process to the CPUs NVML names as local to its GPU BEFORE any pinned host buffer is allocated: first-touch then places the
    staging buffers of the end-to-end legs on the GPU's own NUMA node, so that N ranks feed N GPUs through N root complexes instead of
    crossing the socket interconnect (round 1: the dense-contract e2e of 8 ranks reached 0.47 of 8x one rank).  Returns what it did."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = [64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1 and 64 * w + b < n_cpu]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {'cpus': f'{cpus[0]}-{cpus[-1]} ({len(cpus)})', 'source': 'nvmlDeviceGetCpuAffinity'}
    except Exception as e:
        return {'error': repr(e)[:120]}
    return {'cpus': 'unchanged'}


# ----------------------------------------------------------------------------------------------------------------------
# timing helpers
# ----------------------------------------------------------------------------------------------------------------------
def _barrier(dist):
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()


def _max_over_ranks(dist, ms, dev):
    if dist is None:
        return ms
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def timed_steps(step_fn, steps, warmup, dist, dev, keep=None):
    """W untimed steps, then exactly K steps between CUDA events on the launching stream, barrier + synchronize on both
    sides, max over ranks.  Returns (ms_total, launches).  `keep`, a list, receives host copies of what step_fn returned
    in the last timed step (a tensor or a list / tuple of tensors), taken after the timed region."""
    from deeprecommendation_b200 import ops
    for i in range(warmup):
        step_fn(i)
    _barrier(dist)
    l0 = ops.launch_count()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = None
    for i in range(steps):
        out = step_fn(warmup + i)
    b.record()
    _barrier(dist)
    launches = ops.launch_count() - l0
    if keep is not None:
        keep.extend(t.detach().cpu() for t in (out if isinstance(out, (list, tuple)) else [out]))
    return _max_over_ranks(dist, a.elapsed_time(b), dev), launches


def op_breakdown(step_fn, steps, start_index):
    """Per-op device time inside a (separate, untimed-for-the-headline) pass of the same steps."""
    from deeprecommendation_b200 import ops
    timer = ops.OpTimer()
    ops.set_timer(timer)
    try:
        for i in range(steps):
            # keep the device busy for ~1 ms first, so that the whole step is queued behind it and the events bracket
            # device time only (not the CPU's launch latency, which is what an idle GPU would make them measure)
            torch.cuda._sleep(2_000_000)
            step_fn(start_index + i)
        torch.cuda.synchronize()
    finally:
        ops.set_timer(None)
    # batches differ slightly in their row counts (I = size of the rated-item union): group by op and inner dims
    groups = {}
    for (name, meta), ms in timer.summary().items():
        if name in ('linear', 'linear_tc', 'linear_tc_batch'):        # (M, K, N): M varies with I
            key, var = (name, tuple(meta[1:])), meta[0]
        elif name == 'attention_pool':             # (B, I, H, U): I varies
            key, var = (name, (meta[0],) + tuple(meta[2:])), meta[1]
        else:
            key, var = (name, tuple(meta)), None
        g = groups.setdefault(key, {'ms': [], 'var': []})
        g['ms'] += ms
        g['var'] += [var] * len(ms)
    agg = {}
    for (name, inner), g in groups.items():
        if name in ('linear', 'linear_tc', 'linear_tc_batch'):
            meta = (int(np.max(g['var'])),) + inner
        elif name == 'attention_pool':
            meta = (inner[0], int(np.max(g['var']))) + inner[1:]
        else:
            meta = inner
        agg[(name, meta)] = (float(np.median(g['ms'])), len(g['ms']) / steps)
    return agg


# ----------------------------------------------------------------------------------------------------------------------
# workload A — AttentionNCF, BASELINE configs[1]
# ----------------------------------------------------------------------------------------------------------------------
def build_attention(dev, rank, n_batches=None):
    n_batches = N_ROTATING if n_batches is None else n_batches
    from deeprecommendation_b200 import synth
    from deeprecommendation_b200.content_providers import ArrayDynamicProvider, DeviceCollateProvider, ResidentRows
    from deeprecommendation_b200.neural_collaborative_filtering.models import AttentionNCF
    users_raw, items_raw, ratings = synth.interactions_small(610, 9724, 100_836, seed=42)
    _, u = synth.dense_ids(users_raw)
    item_ids, it = synth.dense_ids(items_raw)
    n_items = len(item_ids)
    profiles = synth.item_profiles(n_items, seed=43)
    row_ptr, idx, rr, _ = synth.user_rating_lists(u, it, ratings, 610)
    prov = ArrayDynamicProvider(np.arange(n_items), profiles, np.arange(610), row_ptr, idx, rr)
    kw = dict(item_dim=F, item_emb=128, user_emb=128, att_dense=128, mlp_dense_layers=[256, 128], dropout_rate=0.2)
    sd = synth.to_torch(synth.attention_ncf_weights(seed=1, **kw))
    model = AttentionNCF(**kw).to(dev).eval()
    model.load_state_dict(sd)
    rprov = None
    if dev.type == 'cuda':        # device-resident provider (SURVEY.md §8 f-4): same batches as row numbers + CSR
        rprov = DeviceCollateProvider(np.arange(n_items), profiles, np.arange(610), row_ptr, idx, rr, device=dev)    # (a ResidentDynamicProvider + K6)
    rng = np.random.default_rng(1000 + rank)           # every rank scores its own shard of the pairs (data-parallel)
    host, nnz, resident_form, picks = [], [], [], []
    for _ in range(n_batches):
        pick = rng.permutation(len(u))[:BATCH]
        rated_idx, um = prov.collate_indices(u[pick])
        if rprov is not None:
            r_idx, um_csr = rprov.collate_csr(u[pick])
            resident_form.append((ResidentRows(rprov.table, it[pick]), ResidentRows(rprov.table, r_idx), um_csr))
            picks.append((torch.from_numpy(u[pick].astype(np.int64)).pin_memory(), resident_form[-1][0]))
        cand = torch.from_numpy(profiles[it[pick]]).pin_memory()
        rated = torch.from_numpy(profiles[rated_idx]).pin_memory()
        host.append((cand, rated, torch.from_numpy(um).pin_memory()))
        nnz.append(int((um != 0).sum()))
    # the reference's serving call (src/webapp/backend.py:78-121): ONE user, every unseen item of the catalogue a candidate
    counts = np.diff(row_ptr)
    su = int(np.argsort(counts)[len(counts) // 2])                       # the user with the median number of rated items
    serving = dict(profiles=profiles, positions=idx[row_ptr[su]:row_ptr[su + 1]].astype(np.int64), ratings=rr[row_ptr[su]:row_ptr[su + 1]].astype(np.float64),
                   table=(rprov.table if rprov is not None else None))
    return dict(model=model, sd=sd, host=host, nnz=nnz, kw=kw, resident_form=resident_form, serving=serving, picks=picks, device_provider=rprov)


def run_attention(w, steps, warmup, dist, dev, peaks):
    from deeprecommendation_b200 import ops
    from deeprecommendation_b200.graphed import GraphedForward
    model, host = w['model'], w['host']
    resident = [tuple(t.to(dev) for t in b) for b in host]
    nb = len(resident)

    def step_eager(i):
        with torch.no_grad():
            return model(*resident[i % nb])

    # one CUDA graph per rotating batch (their rated-item unions differ in size, i.e. in shape): the ~12 launches of a
    # forward are replayed without Python / launch overhead.  The captured inputs are the graphs' own resident copies.
    graphs = None
    if not w.get('eager'):
        try:
            graphs = [GraphedForward(lambda c, r, um: model(c, r, um), *b) for b in resident]
            resident = None                                  # the graphs own the device copies now
        except Exception as e:
            w['graph_capture_error'] = repr(e)[:300]
            graphs = None
    if graphs is None and resident is None:
        resident = [tuple(t.to(dev) for t in b) for b in host]

    def step(i):
        # ONE timed step = all `nb` rotating batches (nb x 512 pairs, ~105 MB of inputs each: the working set of a step is far
        # larger than L2, and K steps make a timed region of tens of milliseconds)
        return [step_eager(k) if graphs is None else graphs[k].replay() for k in range(nb)]

    dump = [] if w.get('dump') else None
    ms, launches = timed_steps(step, steps, warmup, dist, dev, dump)
    if graphs is not None:                                   # replays do not pass through the launch counter
        resident = [tuple(g.static_in) for g in graphs]
        l0 = ops.launch_count()
        for k in range(nb):
            step_eager(k)
        launches = (ops.launch_count() - l0) * steps
    with torch.no_grad():
        out0 = model(*resident[0]).float().cpu()             # batch 0 through the same call: compared with the oracle's output (`parity`)

    # end to end: pinned host buffers in, scores out, every step (H2D straight into the captured input buffers)
    from deeprecommendation_b200.graphed import PipelinedScoring
    pipe = PipelinedScoring(graphs) if graphs is not None else None   # H2D of batch k + 1 under the kernels of batch k, one sync per step

    def step_e2e(i):
        res = None
        if pipe is not None:
            return pipe(host)[-1]
        for k in range(nb):
            if graphs is not None:
                res = graphs[k](*host[k]).cpu()
            else:
                with torch.no_grad():
                    c, r, um = (t.to(dev, non_blocking=True) for t in host[k])
                    res = model(c, r, um).cpu()
        return res

    for i in range(min(warmup, 3)):
        step_e2e(i)
    _barrier(dist)
    t0 = time.perf_counter()
    for i in range(steps):
        step_e2e(i)
    torch.cuda.synchronize()
    e2e_ms = _max_over_ranks(dist, (time.perf_counter() - t0) * 1e3, dev)
    h2d = int(np.sum([sum(t.numel() * 4 for t in b) for b in host]))

    # the same batches through the device-resident provider: row numbers + CSR cross PCIe, the profile table stays in HBM
    rf = w.get('resident_form') or []
    e2e_res = None
    if rf:
        pin_res = torch.empty((nb, BATCH, 1), dtype=torch.float32).pin_memory()

        def step_res(i):                       # scores of every batch land in pinned memory, one synchronize per step
            for k in range(nb):
                c, r, um = rf[k]
                with torch.no_grad():
                    pin_res[k].copy_(model.forward_resident(c, r, um), non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return pin_res[-1]
        for i in range(min(warmup, 3)):
            step_res(i)
        _barrier(dist)
        t0 = time.perf_counter()
        for i in range(steps):
            step_res(i)
        torch.cuda.synchronize()
        res_ms = _max_over_ranks(dist, (time.perf_counter() - t0) * 1e3, dev)
        e2e_res = {'ms': res_ms, 'h2d': int(np.sum([c.pos.numel() * 8 + r.pos.numel() * 8 + um.nbytes() for c, r, um in rf]))}

    # the same (user, item) samples with the collate itself on the device (K6, SURVEY.md §8 a-8 / f-4): per batch 2 x 512 row numbers go up,
    # the size of the rated-item union (4 B) and the scores come back; sort / unique / multi-hot of the reference's collate are inside the timed region
    e2e_ids = None
    dprov, picks = w.get('device_provider'), w.get('picks') or []
    if dprov is not None and picks:
        from deeprecommendation_b200.content_providers import ResidentRows

        pin_ids = torch.empty((len(picks), BATCH, 1), dtype=torch.float32).pin_memory()

        def step_ids(i):
            # K6 of batch k + 1 is enqueued AHEAD of the forward of batch k: its counts are on the host by the time forward k has been launched,
            # so learning I never drains the stream; scores land in pinned memory, one synchronize per step
            pend = dprov.collate_launch(picks[0][0])
            for k, (users, cand) in enumerate(picks):
                rated_rows, um = dprov.collate_finish(pend)
                if k + 1 < len(picks):
                    pend = dprov.collate_launch(picks[k + 1][0])
                with torch.no_grad():
                    pin_ids[k].copy_(model.forward_resident(cand, ResidentRows(dprov.table, rated_rows), um), non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return pin_ids[-1]
        try:
            for i in range(min(warmup, 3)):
                step_ids(i)
            _barrier(dist)
            t0 = time.perf_counter()
            for i in range(steps):
                step_ids(i)
            torch.cuda.synchronize()
            ids_ms = _max_over_ranks(dist, (time.perf_counter() - t0) * 1e3, dev)
            rated0, um0 = dprov.collate_device(picks[0][0])
            with torch.no_grad():
                ids_out0 = model.forward_resident(picks[0][1], ResidentRows(dprov.table, rated0), um0).float().cpu()
            t0 = time.perf_counter()
            for users, _ in picks:
                dprov.collate_csr(users.numpy())
            host_collate_ms = (time.perf_counter() - t0) * 1e3 / len(picks)
            e2e_ids = {'ms': ids_ms, 'h2d': int(sum(u_.numel() * 8 + c.pos.numel() * 8 for u_, c in picks)), 'd2h_extra': 4 * len(picks),
                       'bit_equal_to_dense_contract': bool(torch.equal(ids_out0, out0)), 'host_collate_ms_per_batch': host_collate_ms}
        except Exception as e:
            e2e_ids = {'error': repr(e)[:300]}

    ops_ms = op_breakdown(step_eager, nb, 0)

    # training step of the same batches (NCF/train.py:99-105): forward in train mode (dropout 0.2, isclose target mask), sum-MSE loss,
    # backward (K2's own backward kernel, gradient GEMMs on K1a) and Adam; eager launches — the rated-item union differs per batch
    train = None
    if not w.get('no_train'):
        try:
            model.train()
            ys = [torch.rand(BATCH, 1, device=dev) * 4.5 + 0.5 for _ in range(nb)]

            def one_step(opt, k):
                opt.zero_grad(set_to_none=True)
                (model(*resident[k]) - ys[k]).square().sum().backward()
                opt.step()

            # The rated-item union differs per batch (one shape bucket per rotating batch): ONE CUDA graph per batch holds forward, backward and Adam.
            # The inner-dropout seed is drawn on the device inside the capture, so every replay applies a new mask; the Adam state is shared.
            tgraphs, train_mode = None, 'eager'
            if not w.get('eager'):
                try:
                    opt = torch.optim.Adam(model.parameters(), lr=1e-4, capturable=True)
                    side = torch.cuda.Stream()
                    side.wait_stream(torch.cuda.current_stream())
                    with torch.cuda.stream(side):
                        for k in range(nb):
                            one_step(opt, k)
                    torch.cuda.current_stream().wait_stream(side)
                    torch.cuda.synchronize()
                    tgraphs = []
                    pool = None
                    for k in range(nb):
                        gk = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(gk, pool=pool):
                            one_step(opt, k)
                        pool = gk.pool()
                        tgraphs.append(gk)
                    train_mode = 'cuda_graph (one per rotating batch: forward + backward + Adam)'
                except Exception as e:
                    tgraphs, train_mode = None, 'eager: ' + repr(e)[:200]
                    torch.cuda.synchronize()
            if tgraphs is None:
                opt = torch.optim.Adam(model.parameters(), lr=1e-4, fused=True)

            def train_step(i):
                if tgraphs is not None:
                    tgraphs[i % nb].replay()
                else:
                    one_step(opt, i % nb)

            def train_step_eager(i):
                one_step(opt, i % nb)

            n_train = max(3, steps // 2)
            # warm-up walks every batch shape once: the caching allocator otherwise answers first-seen sizes with cudaMalloc (3 ms each)
            train_ms, _ = timed_steps(train_step, n_train, nb + 2, dist, dev)
            t_ops = op_breakdown(train_step_eager, min(n_train, nb), 0)
            train = {'ms': train_ms / n_train, 'steps': n_train, 'launch_mode': train_mode,
                     'op_ms_per_step': {f'{n}{list(m)}': round(v[0] * v[1], 4) for (n, m), v in sorted(t_ops.items(), key=lambda kv: -kv[1][0] * kv[1][1])[:8]}}
        except Exception as e:
            train = {'error': repr(e)[:300]}
        finally:
            model.eval()
            model.load_state_dict(w['sd'])
    # serving pattern: recommend_for_user = one user x the whole catalogue (+ top-10 + attention-threshold explanations), eager call
    serving = None
    sv = w.get('serving')
    if sv is not None and sv.get('table') is not None:
        try:
            pos, rat = torch.from_numpy(sv['positions']).to(dev), torch.from_numpy(sv['ratings']).to(dev)
            for _ in range(3):
                model.recommend_for_user(sv['table'], pos, rat, k=10)
            torch.cuda.synchronize()
            n_req = 10
            t0 = time.perf_counter()
            for _ in range(n_req):
                rec = model.recommend_for_user(sv['table'], pos, rat, k=10)
                rec['scores'].cpu()
            torch.cuda.synchronize()
            req_ms = (time.perf_counter() - t0) * 1e3 / n_req
            n_cand = sv['table'].shape[0] - len(sv['positions'])
            serving = {'ms_per_request': req_ms, 'candidates': int(n_cand), 'rated_items': int(len(sv['positions'])), 'value': n_cand / (req_ms * 1e-3),
                       'unit': 'pairs/s', 'what': 'AttentionNCF.recommend_for_user (src/webapp/backend.py:78-121): every unseen catalogue item scored for one '
                                                  'user, top-10, explanations by attention threshold; wall clock per request incl. the D2H of the result'}
        except Exception as e:
            serving = {'error': repr(e)[:300]}
    I_mean = float(np.mean([b[1].shape[0] for b in host]))
    TS = 'profiles/traffic.json (static: one `ncu --set full` capture of this kernel per round, not measured in this run)'

    def k1a_roof(opname, meta, kms):
        """SURVEY.md §8d: roofline_time = max(bytes / HBM_peak, flops / pipe_peak), frac = roofline_time / measured time, with the ALGORITHMIC
        flops 2·M·K·N.  fp32 parity runs on the TF32 pipe (dense rate = half the measured bf16 rate; MEASURED_PEAKS.json has no TF32 figure).
        The 3 MMAs per product of the 3xTF32 split are emulation overhead, not useful work: they only show in `issued_frac`, never in `frac`."""
        M, K, N = meta
        ab = 4.0 * (M * K + N * K + M * N)                  # read X and W once, write Y once
        ach = ab / (kms * 1e-3) / 1e9 if kms > 0 else 0.0
        if opname == 'linear':
            return {'bound': 'hbm', 'kernel': f'gemm_tn_kernel (K1a linear {M}x{K}->{N}, fp32 FFMA)', 'achieved': round(ach, 1), 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                    'frac': round(ach / peaks['hbm_gbs'], 4), 'traffic': _traffic('attention'), 'traffic_source': TS, 'peak_source': peaks['src'],
                    'kernel_ms': round(kms, 4), 'algorithmic_bytes': int(ab)}
        flops = 2.0 * M * K * N
        tf32 = w.get('gemm', 'bf16x3') == 'tf32x3'
        issue = 1.0 if w.get('gemm') == 'bf16' else 3.0             # hi.hi + hi.lo + lo.hi in both split engines
        pipe = peaks['bf16_tflops'] / 2.0 if tf32 else peaks['bf16_tflops']
        t_hbm, t_pipe = ab / (peaks['hbm_gbs'] * 1e9), flops / (pipe * 1e12)
        t_roof = max(t_hbm, t_pipe)
        ach_tf = flops / (kms * 1e-3) / 1e12 if kms > 0 else 0.0
        tensor = t_pipe > t_hbm
        return {'bound': 'tensor' if tensor else 'hbm',
                'kernel': f'gemm_tc_kernel + tc_splitk_reduce_kernel (K1a linear {M}x{K}->{N}, tcgen05 {w.get("gemm", "bf16x3")}, 128x256 tiles + split-K)',
                'achieved': round(ach_tf, 1) if tensor else round(ach, 1), 'peak': round(pipe, 1) if tensor else peaks['hbm_gbs'],
                'unit': 'TFLOP/s' if tensor else 'GB/s', 'frac': round(t_roof / (kms * 1e-3), 4) if kms > 0 else 0.0, 'roofline_us': round(t_roof * 1e6, 2),
                'traffic': _traffic('attention'), 'traffic_source': TS, 'peak_source': peaks['src'], 'kernel_ms': round(kms, 4), 'algorithmic_bytes': int(ab),
                'hbm_view': {'achieved': round(ach, 1), 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'roofline_us': round(t_hbm * 1e6, 2)},
                'tensor_view': {'achieved': round(ach_tf, 1), 'peak': round(pipe, 1), 'unit': 'TFLOP/s', 'roofline_us': round(t_pipe * 1e6, 2), 'algorithmic_flops': int(flops),
                                'peak_source': peaks['src'] + (': bf16 burst %.0f TFLOP/s / 2 = dense TF32' % peaks['bf16_tflops'] if tf32 else ': bf16 burst')},
                'issued_tflops': round(ach_tf * issue, 1), 'issued_frac': round(ach_tf * issue / pipe, 4),
                'issued_note': '3 TF32 MMAs per product (hi*hi + hi*lo + lo*hi) for fp32 parity' if tf32 else 'one bf16 MMA per product'}

    def k2_roof(kms):
        ab = float(np.mean(w['nnz'])) * (2 * 128 * 4 + 8) + BATCH * (128 * 4 + 4)     # SURVEY.md §8d, K2
        ach = ab / (kms * 1e-3) / 1e9 if kms > 0 else 0.0
        tr = _traffic('attention_pool')
        r = {'bound': 'hbm', 'kernel': 'um_compact_kernel + attention_wseg_kernel + attention_merge_kernel (K2)', 'achieved': round(ach, 1), 'peak': peaks['hbm_gbs'],
             'unit': 'GB/s', 'frac': round(ach / peaks['hbm_gbs'], 4), 'traffic': tr, 'traffic_source': TS, 'peak_source': peaks['src'], 'kernel_ms': round(kms, 4),
             'algorithmic_bytes': int(ab),
             'regime': 'the two gathered tables are 2 x 9.7 MB at this config: L2-resident.  `frac` is SURVEY.md §8d\'s formula (algorithmic gather bytes / time / HBM '
                       'peak) and measures L2 + latency here, not HBM — the DRAM pins move `traffic` bytes (`dram_frac`); the HBM-regime leg of K2 (`also`, tables 4 GB) is the '
                       'honest HBM figure'}
        if tr:
            r['dram_frac'] = round(tr / (kms * 1e-3) / 1e9 / peaks['hbm_gbs'], 4)
        return r

    def roof_of(opname, meta, kms):
        if opname in ('linear', 'linear_tc', 'linear_tc_batch') and meta[1] >= 512:
            return k1a_roof(opname, meta, kms)
        if opname == 'attention_pool':
            return k2_roof(kms)
        return None

    ranked = sorted(ops_ms.items(), key=lambda kv: -kv[1][0] * kv[1][1])
    roofs = [(n_, roof_of(n_, m_, v_[0])) for (n_, m_), v_ in ranked]
    roofs = [r_ for _, r_ in roofs if r_ is not None]
    roof = roofs[0] if roofs else {'bound': 'hbm', 'kernel': ranked[0][0][0], 'achieved': 0.0, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': 0.0, 'traffic': None}
    roof['op_ms_per_batch'] = {f'{n_}{list(m_)}': round(v_[0] * v_[1], 4) for (n_, m_), v_ in ranked}
    roof['dominance_note'] = ('K1a (rated-item projection) and K2 (attention pooling) take about the same time per batch at this config; whichever is larger in this run is '
                              'the object above, the other is `other_kernels[0]` with the same fields')
    if len(roofs) > 1:
        roof['other_kernels'] = roofs[1:]
    return dict(ms=ms, launches=launches, e2e_ms=e2e_ms, h2d=h2d, d2h=BATCH * 4 * nb, roofline=roof, I_mean=I_mean, out0=out0, nb=nb,
                nnz_mean=float(np.mean(w['nnz'])), e2e_res=e2e_res, e2e_ids=e2e_ids, train=train, serving=serving, dump=dump,
                launch_mode='cuda_graph' if graphs is not None else 'eager: ' + w.get('graph_capture_error', 'requested'))


def cpu_attention(w, sample_pairs=BATCH, repeats=3):
    """the reference's own algorithm (oracle port, literal op order incl. the (B*I, E) materialisation) on host cores"""
    from oracle import restatement as R
    torch.set_num_threads(os.cpu_count() or 1)
    cand, rated, um = (t.clone() for t in w['host'][0])
    cand, um = cand[:sample_pairs], um[:sample_pairs]
    with torch.no_grad():
        out = R.attention_ncf_forward(w['sd'], cand, rated, um)
        ts = []
        for _ in range(repeats):
            t0 = time.perf_counter()
            R.attention_ncf_forward(w['sd'], cand, rated, um)
            ts.append(time.perf_counter() - t0)
    return sample_pairs / float(np.median(ts)), torch.get_num_threads(), \
        f'{sample_pairs} pairs of batch 0 (I={rated.shape[0]} rated items, F={F}), median of {repeats} forwards, oracle/restatement.py', out


def _parity(gpu_out, cpu_out, what, tol=1e-5):
    """max-norm relative error of the CUDA path against the oracle on the SAME benchmarked inputs (the bar of north_star)"""
    a, b = gpu_out.detach().double().cpu().reshape(-1), cpu_out.detach().double().cpu().reshape(-1)
    n = min(a.numel(), b.numel())
    e = float((a[:n] - b[:n]).abs().max() / b[:n].abs().max())
    return {'max_rel': e, 'tolerance': tol, 'ok': bool(e <= tol), 'n': int(n), 'vs': what}


def cpu_serving(w, repeats=2):
    """the reference's per-user serving forward on host cores (backend.py:96-99: one forward over every unseen candidate)"""
    from oracle import restatement as R
    torch.set_num_threads(os.cpu_count() or 1)
    sv = w['serving']
    pos = np.sort(sv['positions'])
    order = np.argsort(sv['positions'])
    ratings = sv['ratings'][order]
    centred = (ratings - (ratings.mean() + 2.5) / 2).astype(np.float32)
    keep = np.ones(sv['profiles'].shape[0], dtype=bool)
    keep[pos] = False
    cand = torch.from_numpy(sv['profiles'][keep])
    rated = torch.from_numpy(sv['profiles'][pos])
    um = torch.from_numpy(np.tile(centred, (cand.shape[0], 1)))
    ts = []
    with torch.no_grad():
        for _ in range(repeats + 1):
            t0 = time.perf_counter()
            R.attention_ncf_forward(w['sd'], cand, rated, um)
            ts.append(time.perf_counter() - t0)
    return float(np.median(ts[1:])) * 1e3


def cpu_attention_train(w, sample_pairs=64, repeats=3):
    """the reference's train step on host cores: forward in train mode (oracle port, dropouts 0) + sum-MSE backward + Adam
    (NCF/train.py:99-105) on the first `sample_pairs` pairs of batch 0 — a whole batch would hold ~40 GB of autograd state"""
    from oracle import restatement as R
    torch.set_num_threads(os.cpu_count() or 1)
    cand, rated, um = (t.clone() for t in w['host'][0])
    cand, um = cand[:sample_pairs], um[:sample_pairs]
    sd = {k: v.clone().requires_grad_(True) for k, v in w['sd'].items()}
    opt = torch.optim.Adam(list(sd.values()), lr=1e-4)
    y = torch.rand(sample_pairs, 1) * 4.5 + 0.5
    ts = []
    for _ in range(repeats + 1):
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        (R.attention_ncf_forward(sd, cand, rated, um, training=True) - y).square().sum().backward()
        opt.step()
        ts.append(time.perf_counter() - t0)
    return sample_pairs / float(np.median(ts[1:])), f'{sample_pairs} pairs of batch 0, median of {repeats} steps'


# ----------------------------------------------------------------------------------------------------------------------
# workload B — GraphNCF propagation, BASELINE configs[2]
# ----------------------------------------------------------------------------------------------------------------------
def zipf_edges_gpu(n_users, n_items, n_edges, dev, seed=42, a_user=0.55, a_item=0.95, active_items=0.946):
    """synth.interactions_zipf with torch on the device (25M unique pairs in well under a second)"""
    g = torch.Generator(device=dev).manual_seed(seed)
    n_act = max(1, int(round(n_items * active_items)))
    cu = torch.cumsum(1.0 / torch.arange(1, n_users + 1, device=dev, dtype=torch.float64) ** a_user, 0)
    ci = torch.cumsum(1.0 / torch.arange(1, n_act + 1, device=dev, dtype=torch.float64) ** a_item, 0)
    cu, ci = cu / cu[-1], ci / ci[-1]
    up = torch.randperm(n_users, device=dev, generator=g)
    ip = torch.randperm(n_items, device=dev, generator=g)[:n_act]
    keys = torch.empty(0, dtype=torch.int64, device=dev)
    while keys.numel() < n_edges:
        m = int((n_edges - keys.numel()) * 1.3) + 1024
        u = torch.searchsorted(cu, torch.rand(m, device=dev, dtype=torch.float64, generator=g)).clamp_(max=n_users - 1)
        i = torch.searchsorted(ci, torch.rand(m, device=dev, dtype=torch.float64, generator=g)).clamp_(max=n_act - 1)
        keys = torch.unique(torch.cat((keys, up[u] * n_items + ip[i])))
    keys = keys[torch.randperm(keys.numel(), device=dev, generator=g)[:n_edges]]
    ratings = torch.randint(1, 11, (n_edges,), device=dev, generator=g).double() * 0.5
    return keys // n_items, keys % n_items, ratings


def build_graph(dev, scale=1.0, world=1, scheme='reduce'):
    from deeprecommendation_b200 import synth
    from deeprecommendation_b200.graph import IdTable, create_graph, get_index
    from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF
    nU, nI, E = int(162_541 * scale), int(62_423 * scale), int(25_000_095 * scale)
    d, L_ = 128, 2
    users, items, ratings = zipf_edges_gpu(nU, nI, E, dev)
    g = torch.Generator(device=dev).manual_seed(7)
    fi = torch.randn(nI, d, device=dev, generator=g)
    fu = torch.randn(nU, d, device=dev, generator=g)
    t0 = time.perf_counter()
    graph = create_graph(users, items, ratings, fi, fu, IdTable(torch.arange(nU, device=dev)), IdTable(torch.arange(nI, device=dev)))
    index = get_index(graph)
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    kw = dict(item_dim=d, user_dim=d, num_gnn_layers=L_, hetero=True, node_emb=d, mlp_dense_layers=[256, 128], dropout_rate=0.2)
    sd = synth.to_torch(synth.graph_ncf_weights(seed=2, **kw))
    model = GraphNCF(**kw).to(dev).eval()
    model.load_state_dict(sd)
    pick = torch.randint(0, E, (64, BATCH), device=dev, generator=g)
    if world > 1:                       # users 1-D nnz-partitioned; exchange = own kernels over peer memory (peer.py) or NCCL (parallel.py)
        from deeprecommendation_b200.parallel import partition_graph
        partition_graph(graph, scheme=scheme, d_max=d, batch_max=BATCH)
    return dict(model=model, sd=sd, graph=graph, index=index, E=E, nU=nU, nI=nI, d=d, L=L_, pick=pick, build_s=build_s, kw=kw,
                edges=(users, items, ratings))


def run_graph(w, steps, warmup, dist, dev, peaks):
    model, graph, index, pick = w['model'], w['graph'], w['index'], w['pick']
    u2i = graph.user2item_edge_index
    ids = [(u2i[0][pick[k]].contiguous(), u2i[1][pick[k]].contiguous()) for k in range(pick.shape[0])]
    ids_host = [(a.cpu().pin_memory(), b.cpu().pin_memory()) for a, b in ids]

    def step_eager(i):
        with torch.no_grad():
            a, b = ids[i % len(ids)]
            return model(graph, a, b, dev)

    # the whole forward (~25 launches + collectives) is captured once and replayed: deeprecommendation_b200/graphed.py
    from deeprecommendation_b200.graphed import GraphedForward
    graphed = None
    if not w.get('eager'):
        try:
            graphed = GraphedForward(lambda a, b: model(graph, a, b, dev), *ids[0])
        except Exception as e:                               # keep the measurement, say what happened
            w['graph_capture_error'] = repr(e)[:300]
            graphed = None

    def step(i):
        if graphed is None:
            return step_eager(i)
        return graphed(*ids[i % len(ids)])

    dump = [] if w.get('dump') else None
    ms, launches = timed_steps(step, steps, warmup, dist, dev, dump)
    if graphed is not None:                                  # replays do not pass through the launch counter
        l0 = __import__('deeprecommendation_b200.ops', fromlist=['x']).launch_count()
        step_eager(0)
        launches = (__import__('deeprecommendation_b200.ops', fromlist=['x']).launch_count() - l0) * steps

    def step_e2e(i):
        a, b = ids_host[i % len(ids)]
        a, b = a.to(dev, non_blocking=True), b.to(dev, non_blocking=True)
        if graphed is None:
            with torch.no_grad():
                return model(graph, a, b, dev).cpu()
        return graphed(a, b).cpu()

    for i in range(min(warmup, 3)):
        step_e2e(i)
    _barrier(dist)
    t0 = time.perf_counter()
    for i in range(steps):
        step_e2e(i)
    torch.cuda.synchronize()
    e2e_ms = _max_over_ranks(dist, (time.perf_counter() - t0) * 1e3, dev)

    ops_ms = op_breakdown(step_eager, min(steps, 4), 0)
    trace = None
    if hasattr(getattr(graph, '_b200rec_partition', None), 'check'):
        torch.cuda.synchronize()
        graph._b200rec_partition.check()                     # a peer wait that timed out would have produced garbage: fail loudly
        if graphed is not None and os.environ.get('B200REC_PEER_TRACE') == '1':
            graphed.replay()
            graphed.replay()
            torch.cuda.synchronize()
            trace = graph._b200rec_partition.trace()         # %globaltimer markers of the last replayed step of this rank

    # training step on the same graph (NCF/train.py:99-105 through gnn_ncf.py:298-367): target edges of the batch masked out of the
    # propagation (pair hash + skip bitmap), conv / MLP dropout, sum-MSE backward (K3 on the reverse-edge weights, gradient GEMMs on
    # K1a) and Adam; eager launches
    train = None
    if w.get('train_leg') and getattr(graph, '_b200rec_partition', None) is None:
        try:
            model.train()
            opt = torch.optim.Adam(model.parameters(), lr=1e-4, fused=True)
            ys = torch.rand(BATCH, 1, device=dev) * 4.5 + 0.5

            def train_step(i):
                a, b = ids[i % len(ids)]
                opt.zero_grad(set_to_none=True)
                (model(graph, a, b, dev) - ys).square().sum().backward()
                opt.step()

            n_train = max(3, steps // 4)
            train_ms, _ = timed_steps(train_step, n_train, 3, dist, dev)
            train = {'ms': train_ms / n_train, 'steps': n_train}
        except Exception as e:
            train = {'error': repr(e)[:300]}
        finally:
            model.eval()
            model.load_state_dict(w['sd'])
            torch.cuda.empty_cache()
    spmm = [(k, v) for k, v in ops_ms.items() if k[0] == 'spmm']
    kms = spmm[0][1][0] if spmm else 0.0
    N, d, E2 = index.num_nodes, w['d'], index.e1 + index.e2
    pg = getattr(graph, '_b200rec_partition', None)
    if pg is not None:                  # rank 0's share of the rows
        E2 = pg.edges_own
    l2 = torch.cuda.get_device_properties(dev).L2_cache_size
    ts = 2 if getattr(model, 'message_dtype', 'fp32') == 'bf16' else 4        # bytes per gathered feature (t); outputs stay fp32
    feat = N * d * ts
    alg_bytes = E2 * 8 + (E2 * d * ts + N * d * 4 if feat > l2 else feat + N * d * 4)       # SURVEY.md §8d, K3
    achieved = alg_bytes / (kms * 1e-3) / 1e9 if kms > 0 else 0.0
    roof = {'bound': 'hbm', 'kernel': 'spmm_chunk_kernel (K3, per layer)', 'achieved': round(achieved, 1), 'peak': peaks['hbm_gbs'],
            'unit': 'GB/s', 'frac': round(achieved / peaks['hbm_gbs'], 4), 'traffic': _traffic('graph'), 'peak_source': peaks['src'],
            'kernel_ms': round(kms, 4), 'algorithmic_bytes': int(alg_bytes), 'features_fit_l2': bool(feat <= l2),
            'gather_inclusive_gbs': round((E2 * 8 + E2 * d * ts) / (kms * 1e-3) / 1e9, 1) if kms > 0 else 0.0,
            'op_ms_per_step': {f'{n}{list(m)}': round(v[0] * v[1], 4) for (n, m), v in sorted(ops_ms.items(), key=lambda kv: -kv[1][0] * kv[1][1])}}
    tf = os.path.join(ROOT, 'profiles', 'tf32_peak.json')
    if kms > 0 and os.path.exists(tf):
        # SURVEY.md §8d: roofline_time = max(bytes / HBM, flops / FP32 peak); at config 3 (features ~ L2) the FP32 side is the larger one
        fp32 = json.load(open(tf)).get('fp32_simt_tflops')
        if fp32:
            flops = 2.0 * E2 * d
            t_fp32 = flops / (fp32 * 1e12) * 1e3
            roof['fp32_view'] = {'algorithmic_flops': int(flops), 'peak': fp32, 'unit': 'TFLOP/s', 'roofline_ms': round(t_fp32, 4),
                                 'frac': round(t_fp32 / kms, 4), 'what': 'cuBLAS fp32 SIMT rate of this GPU (profiles/tf32_peak.json); the kernel itself '
                                 'is bound by the L1 data path (ncu l1tex 81 %), see DESIGN.md'}
    return dict(ms=ms, launches=launches, e2e_ms=e2e_ms, h2d=2 * BATCH * 8, d2h=BATCH * 4, roofline=roof, train=train, trace=trace, dump=dump,
                launch_mode='cuda_graph' if graphed is not None else 'eager: ' + w.get('graph_capture_error', 'requested'))


def cpu_graph(w, sample_frac=0.04, repeats=2):
    """reference algorithm (per-edge Linear + index_add_) on an edge sample of the same graph, host cores"""
    from oracle import restatement as R
    torch.set_num_threads(os.cpu_count() or 1)
    users, items, ratings = (t.cpu().numpy() for t in w['edges'])
    n = int(len(users) * sample_frac)
    users, items, ratings = users[:n], items[:n], ratings[:n]
    g = R.create_graph(users, items, ratings, np.arange(w['nU']), np.arange(w['nI']))
    gd = {k: (torch.from_numpy(v) if v is not None else None) for k, v in g.items()}
    uid = torch.from_numpy(g['user2item_edge_index'][0][:BATCH])
    iid = torch.from_numpy(g['user2item_edge_index'][1][:BATCH])
    gd['item_features'], gd['user_features'] = w['graph'].item_features.cpu(), w['graph'].user_features.cpu()
    ts = []
    with torch.no_grad():
        for _ in range(repeats + 1):
            t0 = time.perf_counter()
            out = R.graph_ncf_forward(w['sd'], gd, uid, iid, w['L'])
            ts.append(time.perf_counter() - t0)
    # the CUDA path on the SAME sampled graph (K4 build + K1c + K3 + K1b), for the `parity` figure of the line
    gpu_out = None
    try:
        from deeprecommendation_b200.graph import IdTable, create_graph
        dev = w['graph'].item_features.device
        eu, ei, er = (t[:n] for t in w['edges'])
        g2 = create_graph(eu, ei, er, w['graph'].item_features, w['graph'].user_features, IdTable(torch.arange(w['nU'], device=dev)),
                          IdTable(torch.arange(w['nI'], device=dev)))
        with torch.no_grad():
            gpu_out = w['model'](g2, uid.to(dev), iid.to(dev), dev).float().cpu()
        del g2
    except Exception as e:
        gpu_out = repr(e)[:300]
    return 2 * n * w['L'] / float(np.median(ts[1:])), torch.get_num_threads(), \
        f'first {n} of {len(w["edges"][0])} interactions ({sample_frac:.0%} edge sample, same node set), median of {repeats} forwards, oracle/restatement.py', \
        out, gpu_out


def run_k3_hbm_regime(dev, peaks, n_users=8_000_000, n_items=1_000_000, n_edges=100_000_000, d=64, reps=5):
    """K3 where the roofline formula is meaningful: node features (2.3 GB) >> L2, so every gathered row comes from HBM.
    Shape = one GPU's share of BASELINE configs[4] (10M users x 1M items x 1B edges, d=64, 8 GPUs), propagation only."""
    from deeprecommendation_b200 import ops
    from deeprecommendation_b200.graph import IdTable, create_graph, get_index
    users, items, ratings = zipf_edges_gpu(n_users, n_items, n_edges, dev, seed=11, a_user=0.5, a_item=0.9)
    graph = create_graph(users, items, ratings, torch.empty(n_items, 1, device=dev), torch.empty(n_users, 1, device=dev),
                         IdTable(torch.arange(n_users, device=dev)), IdTable(torch.arange(n_items, device=dev)))
    del users, items, ratings
    index = get_index(graph)
    N, E2 = index.num_nodes, index.e1 + index.e2
    t = torch.randn(N, d, device=dev)
    x_next, acc = torch.empty(N, d, device=dev), torch.zeros(N, d, device=dev)

    def timed(**kw):
        ts = []
        for r in range(reps + 2):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            ops.spmm_raw(index, t, w=index.w, dinv=index.dinv, **kw)
            b.record()
            torch.cuda.synchronize()
            if r >= 2:
                ts.append(a.elapsed_time(b))
        return float(np.median(ts))

    ms = timed(x_next=x_next)                                               # the layer as SURVEY.md §8d counts it: one (N, d) output
    ms_fused = timed(x_next=x_next, acc_in=acc, acc_out=acc, acc_scale=1.0)     # + the fused running mean (reads and writes one more (N, d))
    alg = E2 * 8 + E2 * d * 4 + N * d * 4                   # SURVEY.md §8d K3, features larger than L2
    achieved = alg / (ms * 1e-3) / 1e9
    alg_fused = alg + 2 * N * d * 4
    probe = _gather_probe()
    roof = {'bound': 'hbm', 'kernel': 'spmm_chunk_kernel + spmm_fixup_kernel (K3)', 'achieved': round(achieved, 1), 'peak': peaks['hbm_gbs'],
            'unit': 'GB/s', 'frac': round(achieved / peaks['hbm_gbs'], 4), 'traffic': _traffic('k3_hbm'),
            'peak_source': peaks['src'], 'kernel_ms': round(ms, 4), 'algorithmic_bytes': int(alg),
            'with_fused_combine': {'kernel_ms': round(ms_fused, 4), 'algorithmic_bytes': int(alg_fused),
                                   'achieved': round(alg_fused / (ms_fused * 1e-3) / 1e9, 1), 'frac': round(alg_fused / (ms_fused * 1e-3) / 1e9 / peaks['hbm_gbs'], 4)}}
    if probe and probe.get(f'gather_{d * 4}B_GBs'):
        roof['random_gather_ceiling'] = {'GB/s': probe[f'gather_{d * 4}B_GBs'], 'frac_of_it': round(achieved / probe[f'gather_{d * 4}B_GBs'], 4),
                                         'what': f'tools/gather_probe.cu: independent random {d * 4}-byte rows of a 4 GiB table, no arithmetic, same GPU, same run'}
    roof['traffic_source'] = 'profiles/traffic.json (static: one `ncu --set full` capture of this kernel per round, not measured in this run)'
    if roof.get('traffic'):
        # `frac` follows SURVEY.md §8d's gather-inclusive formula (every gathered row counted as HBM bytes); the popular rows of the Zipf graph hit
        # in L2, so the DRAM pins move fewer bytes: dram_frac = measured DRAM bytes per launch / kernel time / HBM peak is the honest HBM figure
        roof['dram_gbs'] = round(roof['traffic'] / (ms * 1e-3) / 1e9, 1)
        roof['dram_frac'] = round(roof['traffic'] / (ms * 1e-3) / 1e9 / peaks['hbm_gbs'], 4)
    out = {'metric': 'K3 SpMM directed-edge messages/sec, HBM regime (features >> L2)', 'value': E2 / (ms * 1e-3), 'unit': 'edges/s',
           'ms_per_step': ms, 'dtype': 'f32',
           'config': {'workload': f'one layer of K3 on nU={n_users}, nI={n_items}, E={n_edges} (2E={E2} directed), d={d}: one GPU share of '
                      f'configs[4]; features {N * d * 4 / 1e9:.2f} GB, CSR {E2 * 8 / 1e9:.2f} GB', 'l2': 'working set >> L2'},
           'roofline': roof}
    del graph, index, t, x_next, acc
    torch.cuda.empty_cache()
    return out


_PROBE = None


def _gather_probe():
    """tools/gather_probe.cu (prebuilt by __graft_entry__.build()): the random-row gather bandwidth of this GPU, run once per bench"""
    global _PROBE
    if _PROBE is None:
        exe = os.path.join(ROOT, 'tools', 'build', 'gather_probe')
        _PROBE = {}
        if os.path.exists(exe):
            try:
                r = subprocess.run([exe, '4', '48'], capture_output=True, text=True, timeout=120)
                _PROBE = json.loads(r.stdout.strip().splitlines()[-1])
            except Exception as e:
                _PROBE = {'error': repr(e)[:200]}
    return _PROBE


def run_k2_hbm_regime(dev, peaks, n_items=4_000_000, n_rows=8192, H=128, reps=5, seed=5):
    """K2 where its roofline formula measures HBM (SURVEY.md §8d asks for it): the Pr / Q tables (2 x 2 GB) >> L2, ragged rated lists
    with the config-2 length law (log-normal, mean ~165, clipped to [20, 2698]) over a 4 M-item catalogue, CSR front-end."""
    from deeprecommendation_b200 import ops
    from deeprecommendation_b200 import _lib as L
    g = torch.Generator(device=dev).manual_seed(seed)
    lens = torch.exp(torch.randn(n_rows, device=dev, generator=g) * 1.0 + 4.6).clamp_(20, 2698).long()
    row_ptr = torch.zeros(n_rows + 1, dtype=torch.int64, device=dev)
    row_ptr[1:] = torch.cumsum(lens, 0)
    nnz = int(row_ptr[-1])
    rows = torch.repeat_interleave(torch.arange(n_rows, device=dev), lens)
    col = torch.randint(0, n_items, (nnz,), device=dev, generator=g)
    col = torch.sort(rows * n_items + col).values % n_items                  # ascending inside a row, like the reference's collate
    val = (torch.randint(1, 11, (nnz,), device=dev, generator=g).float() * 0.5 - 2.75)
    csr = (row_ptr.int(), col.int(), val)
    Pr, Q = torch.randn(n_items, H, device=dev), torch.randn(n_items, H, device=dev)
    Pc, a2 = torch.randn(n_rows, H, device=dev), torch.randn(H, device=dev)
    a20, bU = torch.zeros(1, device=dev), torch.zeros(H, device=dev)
    mx = int(lens.max())
    ts = []
    inner = 8                      # calls per timed region, queued back to back: the ~50 us of host-side launch work per call hides behind the GPU
    for r in range(reps + 2):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(inner):
            ops.attention_pool_raw(Pc, Pr, Q, mode=L.ATT_NET, a2=a2, a20=a20, bU=bU, csr=csr, max_row_nnz=mx)
        b.record()
        torch.cuda.synchronize()
        if r >= 2:
            ts.append(a.elapsed_time(b) / inner)
    ms = float(np.median(ts))
    alg = nnz * (2 * H * 4 + 8) + n_rows * (H * 4 + 4)                       # SURVEY.md §8d, K2
    achieved = alg / (ms * 1e-3) / 1e9
    probe = _gather_probe()
    roof = {'bound': 'hbm', 'kernel': 'att_worklist_kernel + attention_wseg_tma_kernel + attention_merge_kernel (K2, CSR front-end)', 'achieved': round(achieved, 1),
            'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': round(achieved / peaks['hbm_gbs'], 4), 'traffic': _traffic('k2_hbm'),
            'traffic_source': 'profiles/traffic.json (static: one `ncu --set full` capture of this kernel per round, not measured in this run)',
            'peak_source': peaks['src'], 'kernel_ms': round(ms, 4), 'algorithmic_bytes': int(alg)}
    if probe and probe.get(f'gather_{H * 4}B_GBs'):
        roof['random_gather_ceiling'] = {'GB/s': probe[f'gather_{H * 4}B_GBs'], 'frac_of_it': round(achieved / probe[f'gather_{H * 4}B_GBs'], 4),
                                         'what': f'tools/gather_probe.cu: independent random {H * 4}-byte rows of a 4 GiB table, no arithmetic, same GPU, same run'}
    out = {'metric': 'K2 attention pooling (candidate, rated-item) interactions/sec, HBM regime (tables >> L2)', 'value': nnz / (ms * 1e-3),
           'unit': 'interactions/s', 'ms_per_step': ms, 'dtype': 'f32',
           'config': {'workload': f'K2 on {n_rows} candidate rows x {n_items} catalogue items, {nnz} non-zeros (mean {nnz / n_rows:.0f}, max {mx} per row), '
                      f'H=U={H}: Pr and Q tables {2 * n_items * H * 4 / 1e9:.1f} GB', 'l2': 'tables >> L2, random rows'},
           'roofline': roof}
    del Pr, Q, Pc, csr, col, val, rows
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------------------------------------------------
# workload C — BasicNCF, BASELINE configs[0] shape
# ----------------------------------------------------------------------------------------------------------------------
def build_basic(dev, rank, n_batches=32):
    from deeprecommendation_b200 import synth
    from deeprecommendation_b200.neural_collaborative_filtering.models import BasicNCF
    users_raw, items_raw, ratings = synth.interactions_small(610, 9724, 100_836, seed=42)
    _, u = synth.dense_ids(users_raw)
    item_ids, it = synth.dense_ids(items_raw)
    profiles = synth.item_profiles(len(item_ids), seed=43)
    uprof = synth.fixed_user_profiles(u, it, ratings, profiles, 610)
    kw = dict(item_dim=F, user_dim=F, item_emb=128, user_emb=128, mlp_dense_layers=[256], dropout_rate=0.2)
    sd = synth.to_torch(synth.basic_ncf_weights(seed=1, **kw))
    model = BasicNCF(**kw).to(dev).eval()
    model.load_state_dict(sd)
    rng = np.random.default_rng(2000 + rank)
    host, resident_form = [], []
    rprov = None
    if dev.type == 'cuda':        # both profile tables resident in HBM (SURVEY.md §8 f-4): the same batches as row numbers
        from deeprecommendation_b200.content_providers import ResidentProfilesProvider
        rprov = ResidentProfilesProvider(np.arange(len(item_ids)), profiles, np.arange(610), uprof, device=dev)
    for _ in range(n_batches):
        pick = rng.permutation(len(u))[:BATCH]
        host.append((torch.from_numpy(uprof[u[pick]]).pin_memory(), torch.from_numpy(profiles[it[pick]]).pin_memory()))
        if rprov is not None:
            resident_form.append((rprov.get_user_profile(u[pick]), rprov.get_item_profile(it[pick])))
    return dict(model=model, sd=sd, host=host, resident_form=resident_form)


def run_basic(w, steps, warmup, dist, dev, peaks):
    model, host = w['model'], w['host']
    resident = [tuple(t.to(dev) for t in b) for b in host]
    nb = len(resident)

    def step_eager(i):
        with torch.no_grad():
            return model(*resident[i % nb])

    from deeprecommendation_b200 import ops
    from deeprecommendation_b200.graphed import GraphedForward
    graphed = None
    if not w.get('eager'):
        try:                                   # all batches share one shape: one captured forward, inputs copied in
            graphed = GraphedForward(lambda a, b: model(a, b), *resident[0])
        except Exception as e:
            w['graph_capture_error'] = repr(e)[:300]

    def step(i):                                 # ONE timed step = all `nb` rotating batches (nb x 512 pairs, 275 MB of inputs > L2)
        out = None
        for k in range(nb):
            out = step_eager(k) if graphed is None else graphed(*resident[k])
        return out

    # the captured forward overwrites its one output buffer per batch: a step leaves the scores of its last batch
    dump = [] if w.get('dump') else None
    ms, launches = timed_steps(step, steps, warmup, dist, dev, dump)
    if graphed is not None:
        l0 = ops.launch_count()
        step_eager(0)
        launches = (ops.launch_count() - l0) * steps * nb
    with torch.no_grad():
        out0 = model(*resident[0]).float().cpu()

    def step_e2e(i):
        res = None
        for k in range(nb):
            if graphed is not None:
                res = graphed(*host[k]).cpu()
            else:
                with torch.no_grad():
                    xu, xi = (t.to(dev, non_blocking=True) for t in host[k])
                    res = model(xu, xi).cpu()
        return res

    for i in range(min(warmup, 3)):
        step_e2e(i)
    _barrier(dist)
    t0 = time.perf_counter()
    for i in range(steps):
        step_e2e(i)
    torch.cuda.synchronize()
    e2e_ms = _max_over_ranks(dist, (time.perf_counter() - t0) * 1e3, dev)
    # the same batches as row numbers into profile tables resident in HBM (ResidentProfilesProvider): per batch 2 x 512 x 8 B go up.
    # `e2e_resident`: rows gathered on the device, then the same kernels as the dense contract (identical bits);
    # `e2e_resident_cached`: every table row projected once per weight version, a batch = the MLP tower over gathered embedding rows
    res_legs = {}
    rf = w.get('resident_form') or []
    if rf:
        for name, cached in (('e2e_resident', False), ('e2e_resident_cached', True)):
            try:
                model.cache_eval_embeddings = cached

                pin_res = torch.empty((len(rf), BATCH, 1), dtype=torch.float32).pin_memory()

                def step_res(i):               # scores of every batch land in pinned memory, one synchronize per step
                    for k, (xu, xi) in enumerate(rf):
                        with torch.no_grad():
                            pin_res[k].copy_(model(xu, xi), non_blocking=True)
                    torch.cuda.current_stream().synchronize()
                    return pin_res[-1]
                for i in range(min(warmup, 3)):
                    step_res(i)
                _barrier(dist)
                t0 = time.perf_counter()
                for i in range(steps):
                    step_res(i)
                torch.cuda.synchronize()
                res_ms = _max_over_ranks(dist, (time.perf_counter() - t0) * 1e3, dev)
                with torch.no_grad():
                    o = model(*rf[0]).float().cpu()
                res_legs[name] = {'ms': res_ms, 'h2d': int(sum(a.pos.numel() * 8 + b.pos.numel() * 8 for a, b in rf)),
                                  'max_rel_vs_dense_contract': float((o - out0).abs().max() / out0.abs().max().clamp_min(1e-30)),
                                  'bit_equal_to_dense_contract': bool(torch.equal(o, out0))}
            except Exception as e:
                res_legs[name] = {'error': repr(e)[:300]}
            finally:
                model.cache_eval_embeddings = False
                model.invalidate_caches()

    # configs[0] names a TRAIN step: forward (dropout 0.2 active) + sum-MSE backward + Adam, gradients of every GEMM on K1a
    train_ms, train_mode = None, 'eager'
    try:
        model.train()
        ys = [torch.rand(BATCH, 1, device=dev) * 4.5 + 0.5 for _ in range(nb)]
        sx = [t.clone() for t in resident[0]] + [ys[0].clone()]           # static inputs of the captured step

        def one_step(opt):
            opt.zero_grad(set_to_none=True)
            loss = (model(sx[0], sx[1]) - sx[2]).square().sum()
            loss.backward()
            opt.step()

        graph = None
        if not w.get('eager'):
            try:                                                          # whole train step (fwd + bwd + Adam) as ONE CUDA graph
                opt = torch.optim.Adam(model.parameters(), lr=1e-4, capturable=True)
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    for _ in range(3):
                        one_step(opt)
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    one_step(opt)
                train_mode = 'cuda_graph'
            except Exception as e:
                graph, train_mode = None, 'eager: ' + repr(e)[:200]
                torch.cuda.synchronize()
        if graph is None:
            opt = torch.optim.Adam(model.parameters(), lr=1e-4)

        def train_step(i):
            for dst, src in zip(sx, resident[i % nb] + (ys[i % nb],)):
                dst.copy_(src, non_blocking=True)
            if graph is not None:
                graph.replay()
            else:
                one_step(opt)

        train_ms, _ = timed_steps(train_step, steps * 4, warmup, dist, dev)
        train_ms /= 4.0                                                   # (ms of `steps` single-batch train steps)
    finally:
        model.eval()
        model.load_state_dict(w['sd'])
    ops_ms = op_breakdown(step_eager, min(steps, nb), 0)
    lin = [(k, v) for k, v in ops_ms.items() if k[0] in ('linear', 'linear_tc_splitk', 'linear_tc_splitk_batch')]
    kms = float(np.mean([v[0] for _, v in lin])) if lin else 0.0
    batched = any(k[0] == 'linear_tc_splitk_batch' for k, _ in lin)           # both projections of the batch in one launch
    alg_bytes = 4.0 * (BATCH * F + 128 * F + BATCH * 128) * (2 if batched else 1)
    achieved = alg_bytes / (kms * 1e-3) / 1e9 if kms > 0 else 0.0
    roof = {'bound': 'hbm', 'kernel': (f'gemm_tc_kernel + 2 x tc_splitk_reduce_kernel (K1a: user and item projections {BATCH}x{F}->128 in one split-K launch, tcgen05)' if batched else f'gemm_tc_kernel + tc_splitk_reduce_kernel (K1a linear {BATCH}x{F}->128, tcgen05 split-K)' if any(k[0] == 'linear_tc_splitk' for k, _ in lin) else f'gemm_tn_kernel (K1a linear {BATCH}x{F}->128, fp32 FFMA, split-K)'), 'achieved': round(achieved, 1),
            'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': round(achieved / peaks['hbm_gbs'], 4), 'traffic': _traffic('basic'),
            'peak_source': peaks['src'], 'kernel_ms': round(kms, 4), 'algorithmic_bytes': int(alg_bytes),
            'op_ms_per_step': {f'{n}{list(m)}': round(v[0] * v[1], 4) for (n, m), v in sorted(ops_ms.items(), key=lambda kv: -kv[1][0] * kv[1][1])}}
    return dict(ms=ms, launches=launches, e2e_ms=e2e_ms, h2d=2 * BATCH * F * 4 * nb, d2h=BATCH * 4 * nb, roofline=roof, train_ms=train_ms, train_mode=train_mode, out0=out0, nb=nb, res_legs=res_legs, dump=dump,
                launch_mode='cuda_graph' if graphed is not None else 'eager: ' + w.get('graph_capture_error', 'requested'))


def cpu_basic(w, repeats=10):
    from oracle import restatement as R
    torch.set_num_threads(os.cpu_count() or 1)
    xu, xi = (t.clone() for t in w['host'][0])
    with torch.no_grad():
        out = R.basic_ncf_forward(w['sd'], xu, xi)
        ts = []
        for _ in range(repeats):
            t0 = time.perf_counter()
            R.basic_ncf_forward(w['sd'], xu, xi)
            ts.append(time.perf_counter() - t0)
    return BATCH / float(np.median(ts)), torch.get_num_threads(), f'batch 0 ({BATCH} pairs, F={F}), median of {repeats} forwards, oracle/restatement.py', out


def cpu_basic_train(w, repeats=10):
    """the reference's train step on host cores: forward (oracle port) + sum-MSE backward + Adam (NCF/train.py:99-105)"""
    from oracle import restatement as R
    torch.set_num_threads(os.cpu_count() or 1)
    xu, xi = (t.clone() for t in w['host'][0])
    sd = {k: v.clone().requires_grad_(True) for k, v in w['sd'].items()}
    opt = torch.optim.Adam(list(sd.values()), lr=1e-4)
    y = torch.rand(BATCH, 1) * 4.5 + 0.5
    ts = []
    for _ in range(repeats + 1):
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        (R.basic_ncf_forward(sd, xu, xi) - y).square().sum().backward()
        opt.step()
        ts.append(time.perf_counter() - t0)
    return BATCH / float(np.median(ts[1:]))


# ----------------------------------------------------------------------------------------------------------------------
# workload D — BasicNCF all-pairs top-K, BASELINE configs[3] (one slab of users per GPU against the whole catalogue)
# ----------------------------------------------------------------------------------------------------------------------
AP_USERS, AP_ITEMS, AP_K = 4736, 100_000, 10          # 148 CTAs x 32 users; configs[3] has 10^6 users x 10^5 items = 211 such slabs


def build_allpairs(dev, rank):
    from deeprecommendation_b200 import synth
    from deeprecommendation_b200.neural_collaborative_filtering.models import BasicNCF
    kw = dict(item_dim=F, user_dim=F, item_emb=128, user_emb=128, mlp_dense_layers=[256, 128], dropout_rate=0.2)
    sd = synth.to_torch(synth.basic_ncf_weights(seed=1, **kw))
    model = BasicNCF(**kw).to(dev).eval()
    model.load_state_dict(sd)
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    # dense F=2094 profiles like synth.item_profiles (966 Bernoulli(0.01) columns + 1128 U[0,1) columns), generated on the device
    def profiles(n):
        x = torch.rand(n, F, device=dev, generator=g)
        x[:, :966] = (x[:, :966] < 0.01).float()
        return x
    items = profiles(AP_ITEMS)
    users = [((profiles(AP_USERS) - 0.3) * 0.1) for _ in range(2)]          # two rotating slabs (40 MB each)
    users_host = [u.cpu().pin_memory() for u in users]
    return dict(model=model, sd=sd, items=items, users=users, users_host=users_host)


def run_allpairs(w, steps, warmup, dist, dev, peaks, precision='fp32'):
    from deeprecommendation_b200 import ops
    model, items, users = w['model'], w['items'], w['users']

    def step(i):
        return model.recommend(users[i % 2], items, k=AP_K, precision=precision)

    dump = [] if w.get('dump') else None
    ms, launches = timed_steps(step, steps, warmup, dist, dev, dump)

    def step_e2e(i):
        xu = w['users_host'][i % 2].to(dev, non_blocking=True)
        val, idx = model.recommend(xu, items, k=AP_K, precision=precision)
        return val.cpu(), idx.cpu()

    for i in range(2):
        step_e2e(i)
    _barrier(dist)
    t0 = time.perf_counter()
    for i in range(steps):
        step_e2e(i)
    torch.cuda.synchronize()
    e2e_ms = _max_over_ranks(dist, (time.perf_counter() - t0) * 1e3, dev)
    ops_ms = op_breakdown(step, min(steps, 3), 0)
    ap = [(k, v) for k, v in ops_ms.items() if k[0] == 'allpairs']
    kms = ap[0][1][0] if ap else 0.0
    pairs = AP_USERS * AP_ITEMS
    flop = pairs * (2.0 * 256 * 128 + 2 * 128)                     # SURVEY.md §8d: 65,792 per pair in all-pairs mode
    issued = flop * (3 if precision == 'fp32' else 1)
    peak = peaks.get('bf16_tflops', 1590.0)
    ach = flop / (kms * 1e-3) / 1e12 if kms > 0 else 0.0
    roof = {'bound': 'tensor', 'kernel': f'allpairs_topk_kernel (K5, tcgen05 kind::f16, {"bf16 hi/lo split: 3 MMAs per k-step" if precision == "fp32" else "bf16"})',
            'achieved': round(ach, 1), 'peak': peak, 'unit': 'TFLOP/s', 'frac': round(ach / peak, 4),
            'issued_tflops': round(issued / (kms * 1e-3) / 1e12, 1) if kms > 0 else 0.0,
            'issued_frac': round(issued / (kms * 1e-3) / 1e12 / peak, 4) if kms > 0 else 0.0,
            'traffic': _traffic('allpairs'), 'peak_source': peaks['src'] + ' bf16_tflops (burst: kernel timed alone)', 'kernel_ms': round(kms, 4),
            'algorithmic_flops': int(flop),
            'op_ms_per_step': {f'{n}{list(m)}': round(v[0] * v[1], 4) for (n, m), v in sorted(ops_ms.items(), key=lambda kv: -kv[1][0] * kv[1][1])}}
    return dict(ms=ms, launches=launches, e2e_ms=e2e_ms, h2d=AP_USERS * F * 4, d2h=AP_USERS * AP_K * 12, roofline=roof, pairs=pairs, dump=dump)


def cpu_allpairs(w, n_users=16, n_items=2000):
    """reference forward on every pair of a sub-grid (oracle port), host cores"""
    from oracle import restatement as R
    torch.set_num_threads(os.cpu_count() or 1)
    xu, xi = w['users_host'][0][:n_users].clone(), w['items'][:n_items].cpu()
    with torch.no_grad():
        R.basic_ncf_all_pairs(w['sd'], xu[:2], xi)
        t0 = time.perf_counter()
        sc = R.basic_ncf_all_pairs(w['sd'], xu, xi)
        R.topk_stable(sc, AP_K)
        dt = time.perf_counter() - t0
    # the CUDA path on the same sub-grid: scores of the fp32-tolerance mode and of the bf16 mode, top-k against a stable sort of its own scores
    parity = {}
    try:
        dev = w['items'].device
        for precision, tol in (('fp32', 1e-5), ('bf16', 1e-2)):
            val, idx, scores = w['model'].recommend(xu.to(dev), w['items'][:n_items], k=AP_K, precision=precision, return_scores=True)
            pr = _parity(scores, sc, f'oracle/restatement.py::basic_ncf_all_pairs on a {n_users} x {n_items} sub-grid of the benchmarked inputs', tol)
            sv, si = R.topk_stable(scores.cpu(), AP_K)
            pr['topk_equals_stable_sort_of_own_scores'] = bool(torch.equal(idx.cpu(), si))
            parity[precision] = pr
    except Exception as e:
        parity = {'error': repr(e)[:300]}
    return n_users * n_items / dt, torch.get_num_threads(), \
        f'{n_users} users x {n_items} items sub-grid of the same inputs (reference forward per pair + stable top-{AP_K}), oracle/restatement.py', parity


# ----------------------------------------------------------------------------------------------------------------------
def reference_arm(args):
    """--impl reference: the reference's own CPU algorithm (the reference is pure Python/PyTorch and absent on the GPU box,
    so the oracle port — the same torch op sequence — stands in), all host threads, bounded samples of the same configs."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cpu = torch.device('cpu')

    class _NoPin:
        pass
    # build the same inputs without touching CUDA
    orig = torch.Tensor.pin_memory
    torch.Tensor.pin_memory = lambda self, *a, **k: self
    try:
        w = build_attention(cpu, 0, n_batches=max(1, min(args.steps + args.warmup, 8)))
    finally:
        torch.Tensor.pin_memory = orig
    from oracle import restatement as R
    sample = int(os.environ.get("B200REC_REF_SAMPLE", "512"))
    times = []
    with torch.no_grad():
        for i in range(args.warmup + args.steps):
            cand, rated, um = w['host'][i % len(w['host'])]
            t0 = time.perf_counter()
            R.attention_ncf_forward(w['sd'], cand[:sample], rated, um[:sample])
            if i >= args.warmup:
                times.append(time.perf_counter() - t0)
    total = float(np.sum(times))
    value = sample * args.steps / total
    line = {'impl': 'reference', 'metric': 'scored user-item pairs/sec (NCF fwd)', 'value': value, 'unit': 'pairs/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': total / args.steps * 1e3, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': attention_config(args.gpus, args.gemm),
            'run_info': {'note': (f'each reference step = one whole batch of {BATCH} pairs' if sample >= BATCH else f'each reference step = the first {sample} pairs of a batch of {BATCH}') +
                         f' (a bounded sample of the B200 arm\'s step of {N_ROTATING} batches; the reference materialises two (B*I,128) fp32 tensors, '
                         'attention_ncf.py:154-155: ~12 GB of host memory per batch)'},
            'cpu_baseline': {'value': value, 'unit': 'pairs/s', 'cores': torch.get_num_threads(), 'kind': 'port',
                             'sample': f'{sample} pairs per step x {args.steps} steps, oracle/restatement.py::attention_ncf_forward'},
            'e2e': {'value': value, 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


N_ROTATING = 8


def attention_config(world, gemm):
    """`config` of the headline line — the SAME dict in the B200 arm and in the reference arm (run-specific figures live in `run_info`)"""
    return {'workload': ATT_WORKLOAD, 'batch': BATCH, 'batches_per_step': N_ROTATING,
            'parallelism': f'dp{world} (pairs sharded, no collective)',
            'l2': f'one step = {N_ROTATING} rotating batches (~105 MB of inputs each, resident in HBM): working set of a step >> 126 MB L2',
            'gemm_engine': gemm}


# ----------------------------------------------------------------------------------------------------------------------
# workload E — GraphNCF 3 layers on 10M users x 1M items x 1B edges, BASELINE configs[4]: built AND run partitioned
# ----------------------------------------------------------------------------------------------------------------------
G5_USERS, G5_ITEMS, G5_EDGES, G5_D, G5_LAYERS, G5_VSHARDS = 10_000_000, 1_000_000, 1_000_000_000, 64, 3, 8


def g5_shard_edges(v, n_users_v, n_items, n_edges_v, dev, a_user=0.5, a_item=0.9, active_items=0.95):
    """interactions of VIRTUAL shard v (its own users x all items), unique pairs, Zipf-like degrees on both sides.  The graph is the union of
    G5_VSHARDS such shards whatever the number of ranks, so every --gpus N runs the SAME graph (a rank owns G5_VSHARDS / N of them)."""
    g = torch.Generator(device=dev).manual_seed(1000 + v)
    gi = torch.Generator(device=dev).manual_seed(999)                      # the item popularity order is shared by all shards
    n_act = max(1, int(round(n_items * active_items)))
    ip = torch.randperm(n_items, device=dev, generator=gi)[:n_act]
    cu = torch.cumsum(1.0 / torch.arange(1, n_users_v + 1, device=dev, dtype=torch.float64) ** a_user, 0)
    ci = torch.cumsum(1.0 / torch.arange(1, n_act + 1, device=dev, dtype=torch.float64) ** a_item, 0)
    cu, ci = cu / cu[-1], ci / ci[-1]
    up = torch.randperm(n_users_v, device=dev, generator=g)
    keys = torch.empty(0, dtype=torch.int64, device=dev)
    while keys.numel() < n_edges_v:
        m = int((n_edges_v - keys.numel()) * 1.25) + 1024
        u = torch.searchsorted(cu, torch.rand(m, device=dev, dtype=torch.float64, generator=g)).clamp_(max=n_users_v - 1)
        i = torch.searchsorted(ci, torch.rand(m, device=dev, dtype=torch.float64, generator=g)).clamp_(max=n_act - 1)
        new = up[u] * n_items + ip[i]
        del u, i
        keys = torch.unique(torch.cat((keys, new)))
        del new
    keys = keys[torch.randperm(keys.numel(), device=dev, generator=g)[:n_edges_v]]
    ratings = torch.randint(1, 11, (n_edges_v,), device=dev, generator=g).double() * 0.5
    return keys // n_items, keys % n_items, ratings


def run_graph5(args, dev, rank, world, dist, peaks, scale=1.0):
    """configs[4]: every rank generates and indexes ONLY its own users' interactions (deeprecommendation_b200/sharded.py), the propagation
    runs over peer memory (peer.py).  Parity at full size: with identity transforms and rank-one features x0[n] = s0[n]·v every layer stays
    rank-one, x_l[n] = s_l[n]·v with s_{l+1} = D^-1/2 A_w D^-1/2 s_l — a float64 torch SpMV recurrence (+ NCCL sums at check time) that the
    CUDA path must reproduce on EVERY owned row."""
    import torch.distributed as tdist
    from deeprecommendation_b200 import synth
    from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF
    from deeprecommendation_b200.peer import forward_peer
    from deeprecommendation_b200.sharded import build_shard
    V = G5_VSHARDS
    if world > V or V % world:
        raise ValueError(f'graph5 runs on 1, 2, 4 or 8 GPUs (the graph is the union of {V} virtual shards)')
    nU, nI, E, d, L_ = int(G5_USERS * scale), int(G5_ITEMS * scale), int(G5_EDGES * scale), G5_D, G5_LAYERS
    nU_v, E_v = nU // V, E // V
    nU, E = nU_v * V, E_v * V
    mine = list(range(rank * (V // world), (rank + 1) * (V // world)))
    t0 = time.perf_counter()
    us, its, rs = [], [], []
    for k, v in enumerate(mine):
        u, i, r = g5_shard_edges(v, nU_v, nI, E_v, dev)
        us.append(u + k * nU_v)
        its.append(i)
        rs.append(r)
    u_local, items, ratings = torch.cat(us), torch.cat(its), torch.cat(rs)
    del us, its, rs
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0
    n_local = nU_v * len(mine)
    users_r0 = mine[0] * nU_v
    gf = torch.Generator(device=dev).manual_seed(77)
    item_features = torch.randn(nI, d, device=dev, generator=gf)                        # pre-embedded (N, 64) node features
    user_features = torch.cat([torch.randn(nU_v, d, device=dev, generator=torch.Generator(device=dev).manual_seed(500 + v)) for v in mine])
    t0 = time.perf_counter()
    if dist is None:
        tdist.init_process_group('gloo', init_method='tcp://127.0.0.1:29597', rank=0, world_size=1) if not tdist.is_initialized() else None
    sh = build_shard(u_local, items, ratings, nI=nI, nU=nU, users_r0=users_r0, n_local_users=n_local, item_features=item_features,
                     user_features_local=user_features, d_max=d, batch_max=BATCH, edges_total=2 * E)
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    kw = dict(item_dim=d, user_dim=d, num_gnn_layers=L_, hetero=True, node_emb=d, mlp_dense_layers=[128], dropout_rate=0.2)
    model = GraphNCF(**kw).to(dev).eval()
    model.load_state_dict(synth.to_torch(synth.graph_ncf_weights(seed=2, **kw)))
    gb = torch.Generator(device=dev).manual_seed(5)                                    # the same batch on every rank
    pick = torch.randint(0, E_v, (BATCH,), device=dev, generator=gb)
    v0 = g5_batch_pairs(nU_v, nI, E_v, pick, dev)
    uid, iid = (v0[0] + nI).contiguous(), v0[1].contiguous()

    def step(i):
        with torch.no_grad():
            return forward_peer(model, sh, uid, iid)

    steps = max(3, min(args.steps, 10))
    ms, launches = timed_steps(step, steps, 3, dist, dev)
    torch.cuda.synchronize()
    sh.check()
    ops_ms = op_breakdown(step, 2, 0)
    spmm = sorted([(k, v) for k, v in ops_ms.items() if k[0] == 'spmm'], key=lambda kv: -kv[1][0])
    # ---- parity at full size: rank-one features through identity transforms vs a float64 SpMV recurrence ----
    parity = g5_rank_one_check(model, sh, dist, dev, nI, d, L_, uid, iid)
    sd0 = synth.to_torch(synth.graph_ncf_weights(seed=2, **kw))
    model.load_state_dict(sd0)
    msgs = 2.0 * E * L_ * steps
    kms = float(np.mean([v[0] for _, v in spmm])) if spmm else 0.0
    e_own = sh.edges_own / 2.0                                                          # directed entries of ONE of this rank's two SpMMs per layer
    alg = e_own * 8 + e_own * d * 4 + (sh.nI + sh.users_rows) / 2.0 * d * 4             # SURVEY.md §8d K3, features larger than L2
    roof = {'bound': 'hbm', 'kernel': 'spmm_chunk_kernel + spmm_fixup_kernel (K3; mean of the rank\'s two SpMMs per layer: partial item rows with the push '
                                      'epilogue, own user rows)', 'achieved': round(alg / (kms * 1e-3) / 1e9, 1) if kms else 0.0, 'peak': peaks['hbm_gbs'],
            'unit': 'GB/s', 'frac': round(alg / (kms * 1e-3) / 1e9 / peaks['hbm_gbs'], 4) if kms else 0.0, 'traffic': None, 'peak_source': peaks['src'],
            'kernel_ms': round(kms, 4), 'algorithmic_bytes': int(alg),
            'op_ms_per_step': {f'{n}{list(m)}': round(v[0] * v[1], 4) for (n, m), v in sorted(ops_ms.items(), key=lambda kv: -kv[1][0] * kv[1][1])}}
    exch = (world - 1) / world * nI * d * 4
    return {'metric': 'GNN propagation directed-edge messages/sec (GraphNCF fwd, configs[4])', 'value': msgs / (ms * 1e-3), 'unit': 'edges/s',
            'ms_per_step': ms / steps, 'steps': steps, 'n_gpus': world, 'scaling': 'strong', 'dtype': 'f32',
            'parallelism': PARALLELISM['peer'].format(P=world) + '; the graph is generated and indexed per rank (sharded.py): item means / degrees by one all-reduce at build time',
            'config': {'workload': f'configs[4]: GraphNCF L={L_} d={d} hetero mlp=[128] (train_model.py:166-174), synthetic nU={nU}, nI={nI}, E={E} '
                                   f'({2 * E} directed), pre-embedded (N,{d}) features, whole-graph propagation + MLP on a batch of {BATCH} per step',
                       'l2': f'per rank: CSR {sh.edges_own * 8 / 1e9:.1f} GB, features {(n_local + nI) * d * 4 / 1e9:.2f} GB >> L2',
                       'generate_s': round(gen_s, 2), 'index_build_s': round(build_s, 2), 'launch_mode': 'eager', 'scale': scale},
            'exchange_bytes_per_layer_per_rank': {'partials_pushed': int(exch), 'transformed_rows_received': int(exch),
                                                  'note': 'fp32; SURVEY.md §8d counted 2.46 GB for an all-gather of ALL N rows — only the item side crosses NVLink here'},
            'roofline': roof, 'parity': parity, 'gpu_launches': launches,
            'e2e': {'value': msgs / (ms * 1e-3), 'unit': 'edges/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0,
                    'note': 'the batch ids are resident; configs[2] carries the host-fed leg'}}


def g5_batch_pairs(nU_v, nI, E_v, pick, dev):
    """(user index, item index) of `pick` interactions of virtual shard 0 — regenerated, so that every rank knows the same batch"""
    u, i, _ = g5_shard_edges(0, nU_v, nI, E_v, dev)
    return u[pick], i[pick]


def g5_rank_one_check(model, sh, dist, dev, nI, d, L_, uid, iid):
    from deeprecommendation_b200.peer import forward_peer
    import torch.distributed as tdist
    eye = torch.eye(d, device=dev)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    for k in sd:
        if k.startswith(('item_embeddings', 'user_embeddings', 'gnn_convs')):
            sd[k] = eye.clone() if k.endswith('weight') else torch.zeros_like(sd[k])
    model.load_state_dict(sd)
    g = torch.Generator(device=dev).manual_seed(31)
    v = torch.randn(d, device=dev, generator=g)
    s_items = torch.rand(nI, device=dev, generator=g, dtype=torch.float64) + 0.5            # same on every rank
    s_users = torch.rand(sh.users_rows, device=dev, dtype=torch.float64, generator=torch.Generator(device=dev).manual_seed(900 + sh.rank)) + 0.5
    keep_feat = (sh.item_features_own, sh.user_features_own)
    sh.item_features_own = (s_items[sh.it_r0: sh.it_r0 + sh.it_rows, None] * v.double()).float()
    sh.user_features_own = (s_users[:, None] * v.double()).float()
    keep = {}
    try:
        with torch.no_grad():
            forward_peer(model, sh, uid, iid, keep)
        torch.cuda.synchronize()
        sh.check()
    finally:
        sh.item_features_own, sh.user_features_own = keep_feat
    # float64 recurrence with torch ops: s' = dinv ∘ (A_w (dinv ∘ s)) per node type; item rows are sums over ALL ranks' users
    iu, ii = sh.index_users, sh.index_items
    rows_u = torch.repeat_interleave(torch.arange(sh.users_rows, device=dev), (iu.row_ptr[1:] - iu.row_ptr[:-1]).long())
    rows_i = torch.repeat_interleave(torch.arange(nI, device=dev), (ii.row_ptr[1:] - ii.row_ptr[:-1]).long())
    du, di = sh.dinv_users.double(), sh.dinv_items_all.double()
    acc_u, acc_i = s_users.clone(), s_items.clone()
    su, si = s_users, s_items
    for _ in range(L_):
        nu = torch.zeros(sh.users_rows, dtype=torch.float64, device=dev).index_add_(0, rows_u, iu.w.double() * (di * si)[iu.col.long()]) * du
        part = torch.zeros(nI, dtype=torch.float64, device=dev).index_add_(0, rows_i, ii.w.double() * (du * su)[ii.col.long()])
        if dist is not None:
            tdist.all_reduce(part)
        su, si = nu, part * di
        acc_u, acc_i = acc_u + su, acc_i + si
    acc_u, acc_i = acc_u / (L_ + 1), acc_i / (L_ + 1)
    want_u = acc_u[:, None] * v.double()
    want_i = acc_i[sh.it_r0: sh.it_r0 + sh.it_rows, None] * v.double()
    den = max(float(want_u.abs().max()), float(want_i.abs().max()))
    err = max(float((keep['users'].double() - want_u).abs().max()), float((keep['items'].double() - want_i).abs().max()) if sh.it_rows else 0.0) / den
    err = _max_over_ranks(dist, err, dev)
    return {'max_rel': err, 'tolerance': 1e-5, 'ok': bool(err <= 1e-5), 'rows_checked': 'every owned user and item row of every rank (max over ranks)',
            'vs': 'float64 torch SpMV recurrence s_{l+1} = D^-1/2 A_w D^-1/2 s_l on rank-one features with identity transforms (size-independent linearity property)'}


# ----------------------------------------------------------------------------------------------------------------------
# workload F — configs[3] IN FULL: every (user, item) pair of 10^6 users x 10^5 items scored, top-10 per user, users sharded over the ranks
# ----------------------------------------------------------------------------------------------------------------------
APF_USERS, APF_ITEMS = 1_000_000, 100_000


def run_allpairs_full(args, dev, rank, world, dist, peaks, n_users_total=APF_USERS):
    """The serving pattern of src/webapp/backend.py:96-99,113-121 for the whole user base: per rank its share of the users (125 k at 8 GPUs)
    against the whole catalogue, both MLP variants ([256,128] and [256]), fp32-tolerance and bf16 operands.  Timed per variant, wall clock on the
    device, max over ranks: user + item projections (K1a), all-pairs MLP + top-k (K5), top-k lists copied to the host.  Nothing is extrapolated."""
    from deeprecommendation_b200 import synth
    from deeprecommendation_b200.neural_collaborative_filtering.models import BasicNCF
    from oracle import restatement as R
    n_users = n_users_total // world
    g = torch.Generator(device=dev).manual_seed(4000 + rank)

    def profiles(n, gen):
        x = torch.rand(n, F, device=dev, generator=gen)
        x[:, :966] = (x[:, :966] < 0.01).float()
        return x
    items = profiles(APF_ITEMS, torch.Generator(device=dev).manual_seed(4999))          # the catalogue is the same on every rank
    users = (profiles(n_users, g) - 0.3) * 0.1
    out = {'metric': f'scored user-item pairs/sec (BasicNCF all-pairs + top-{AP_K}, configs[3] in full)', 'unit': 'pairs/s', 'n_gpus': world, 'scaling': 'strong',
           'config': {'workload': f'configs[3]: {n_users_total} users x {APF_ITEMS} items = {n_users_total * APF_ITEMS:.3g} pairs, top-{AP_K} per user, '
                                  f'F={F} dense profiles on both sides; {n_users} users per GPU, catalogue replicated, no collective',
                      'l2': 'user profiles 1 GB, item profiles 0.84 GB, item tables 102 MB per GPU'},
           'variants': {}}
    pairs_total = float(n_users) * APF_ITEMS * world
    for mlp in ([256, 128], [256]):
        kw = dict(item_dim=F, user_dim=F, item_emb=128, user_emb=128, mlp_dense_layers=mlp, dropout_rate=0.2)
        sd = synth.to_torch(synth.basic_ncf_weights(seed=1, **kw))
        model = BasicNCF(**kw).to(dev).eval()
        model.load_state_dict(sd)
        for precision, tol in (('fp32', 1e-5), ('bf16', 1e-2)):
            model.recommend(users[:4736], items, k=AP_K, precision=precision)              # warm-up: packs, caches, lazy inits
            _barrier(dist)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            a.record()
            val, idx = model.recommend(users, items, k=AP_K, precision=precision)
            val_h, idx_h = val.cpu(), idx.cpu()                                            # the top-k lists leave the device inside the timed region
            b.record()
            torch.cuda.synchronize()
            wall_ms = (time.perf_counter() - t0) * 1e3
            ms = _max_over_ranks(dist, a.elapsed_time(b), dev)
            wall_ms = _max_over_ranks(dist, wall_ms, dev)
            ent = {'ms_total': round(ms, 2), 'wall_ms_total': round(wall_ms, 2), 'value': pairs_total / (ms * 1e-3),
                   'd2h_bytes': int(val_h.numel() * 4 + idx_h.numel() * 8)}
            if rank == 0:
                # sampled users against the oracle on a sub-grid + the selection against a stable sort of the kernel's own scores over ALL items
                su = torch.arange(0, n_users, max(1, n_users // 16), device=dev)[:16]
                v2, i2, sc = model.recommend(users[su], items, k=AP_K, precision=precision, return_scores=True)
                ref = R.basic_ncf_all_pairs(sd, users[su].cpu(), items[:2000].cpu())
                ent['parity'] = _parity(sc[:, :2000], ref, 'oracle/restatement.py::basic_ncf_all_pairs, 16 sampled users x 2000 items', tol)
                # selection of the FULL run for these users against the scores of this (separately launched) call: the picked items must carry
                # the k largest scores (near-ties may swap: the two launches project the users with different GEMM tilings, ~1e-7 apart)
                scc, pick_i = sc.cpu(), idx_h[su.cpu()]
                sv, si = R.topk_stable(scc, AP_K)
                picked = torch.gather(scc, 1, pick_i)
                span = float(scc.abs().max())
                ent['parity']['topk_of_the_full_run'] = {
                    'identical_to_stable_sort': bool(torch.equal(pick_i, si)),
                    'picked_scores_vs_k_best_max_rel': float((picked - sv).abs().max() / span),
                    'values_vs_rescored_max_rel': float((val_h[su.cpu()] - picked).abs().max() / span)}
                # full-catalogue error figure of this arithmetic mode: the same 16 users x ALL items in float64 on the device
                w64 = {k: v.to(dev).double() for k, v in sd.items()}
                ue = users[su].double() @ w64['user_embeddings.0.weight'].T + w64['user_embeddings.0.bias']
                ie = items.double() @ w64['item_embeddings.0.weight'].T + w64['item_embeddings.0.bias']
                keys = sorted({int(k.split('.')[1]) for k in w64 if k.startswith('MLP.')})
                worst = 0.0
                for r0 in range(0, su.numel(), 4):                                         # 4 users x 100 k items x 256 doubles = 0.8 GB at a time
                    h = torch.cat((ue[r0:r0 + 4, None, :].expand(-1, APF_ITEMS, -1), ie[None].expand(min(4, su.numel() - r0), -1, -1)), 2)
                    for q, kk in enumerate(keys):
                        h = h @ w64[f'MLP.{kk}.weight'].T + w64[f'MLP.{kk}.bias']
                        if q < len(keys) - 1:
                            h = h.relu()
                    worst = max(worst, float((sc[r0:r0 + 4].double() - h[..., 0]).abs().max() / h.abs().max()))
                    del h
                ent['full_catalogue_error'] = {'max_rel': worst, 'tolerance': tol, 'ok': bool(worst <= tol),
                                               'vs': 'float64 torch evaluation of the same forward on the device, 16 users x all 100k items'}
                del sc, ue, ie, w64
            out['variants'][f'mlp{mlp}_{precision}'] = ent
            del val, idx
        del model
    head = out['variants']['mlp[256, 128]_fp32']
    out.update({'value': head['value'], 'ms_total': head['ms_total'], 'dtype': 'f32',
                'note': 'headline = MLP [256,128], fp32-tolerance operands; `variants` carries [256] and the bf16 modes; every figure is a full run'})
    del users, items
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------------------------------------------------
# workload G — K1s: projection of one-hot / multi-hot profile rows (north_star (1), SURVEY.md §8d row 2)
# ----------------------------------------------------------------------------------------------------------------------
def run_sparse(args, dev, rank, world, dist, peaks):
    """(a) BasicNCF on the reference's item-profile structure — 966 multi-hot columns (~1 %) as index lists + 1,128 dense columns
    (content_providers.MixedRows) against the same rows streamed dense; (b) the one-hot variant (one_hot_provider.py:17-21) at a catalogue
    whose embedding table (4 M x 128 fp32 = 2 GB) does not fit L2: a pure gather, HBM roofline (E_emb*s + 8) bytes per non-zero."""
    from deeprecommendation_b200 import ops, synth
    from deeprecommendation_b200.content_providers import MixedRows, OneHotRows
    from deeprecommendation_b200.neural_collaborative_filtering.models import BasicNCF
    from oracle import restatement as R
    kw = dict(item_dim=F, user_dim=F, item_emb=128, user_emb=128, mlp_dense_layers=[256], dropout_rate=0.2)
    sd = synth.to_torch(synth.basic_ncf_weights(seed=1, **kw))
    model = BasicNCF(**kw).to(dev).eval()
    model.load_state_dict(sd)
    nb = 16
    xi = [synth.item_profiles(BATCH, seed=50 + b) for b in range(nb)]
    xu = [((synth.item_profiles(BATCH, seed=90 + b) - 0.3) * 0.1).astype(np.float32) for b in range(nb)]
    dense = [(torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev)) for u, i in zip(xu, xi)]
    mixed = [(torch.from_numpy(u).to(dev), MixedRows.from_dense(i, 966).to(dev)) for u, i in zip(xu, xi)]
    nnz = float(np.mean([m[1].col.numel() for m in mixed]))

    def step_dense(i):
        with torch.no_grad():
            out = None
            for b in range(nb):
                out = model(*dense[b])
            return out

    def step_mixed(i):
        with torch.no_grad():
            out = None
            for b in range(nb):
                out = model(*mixed[b])
            return out

    ms_d, _ = timed_steps(step_dense, args.steps, 3, dist, dev)
    ms_m, launches = timed_steps(step_mixed, args.steps, 3, dist, dev)
    with torch.no_grad():
        par = _parity(model(*mixed[0]), R.basic_ncf_forward(sd, torch.from_numpy(xu[0]), torch.from_numpy(xi[0])),
                      'oracle/restatement.py::basic_ncf_forward on the dense form of batch 0')
    # (b) one-hot lookups out of a table far larger than L2
    n_classes, E, M = 4_000_000, 128, 1 << 20
    g = torch.Generator(device=dev).manual_seed(3)
    wt = torch.randn(n_classes, E, device=dev, generator=g)           # W^T of the (E, n_classes) Linear = the embedding table (ops._transposed_weight caches it)
    bias = torch.randn(E, device=dev, generator=g)
    ids = torch.randint(0, n_classes, (M,), device=dev, generator=g)
    out = torch.empty((M, E), device=dev)
    from deeprecommendation_b200 import _lib as L
    import ctypes as C

    def lookup():
        L.check(L.lib().b200rec_linear_sparse(None, None, None, C.c_void_p(ids.data_ptr()), M, C.c_void_p(wt.data_ptr()), n_classes, E, E, L.F32,
                                              C.c_void_p(bias.data_ptr()), C.c_void_p(out.data_ptr()), E, 0,
                                              C.c_void_p(torch.cuda.current_stream().cuda_stream)), 'linear_sparse')
    ts = []
    for r in range(7):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        lookup()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    kms = float(np.median(ts[2:]))
    exact = bool(torch.equal(out[:4096], wt[ids[:4096]] + bias))
    alg = M * (E * 4 + 8) + M * E * 4                                  # table row + id per non-zero, + the output row
    roof = {'bound': 'hbm', 'kernel': 'gather_sum_kernel (K1s, one-hot ids -> rows of W^T, 4 M x 128 fp32 table = 2 GB)', 'achieved': round(alg / (kms * 1e-3) / 1e9, 1),
            'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': round(alg / (kms * 1e-3) / 1e9 / peaks['hbm_gbs'], 4), 'traffic': None,
            'peak_source': peaks['src'], 'kernel_ms': round(kms, 4), 'algorithmic_bytes': int(alg), 'lookup_equals_table_rows_plus_bias': exact}
    pairs = BATCH * nb * args.steps * world
    del wt, out, ids
    torch.cuda.empty_cache()
    return {'metric': 'scored user-item pairs/sec (BasicNCF fwd, multi-hot item columns as index lists)', 'value': pairs / (ms_m * 1e-3), 'unit': 'pairs/s',
            'ms_per_step': ms_m / args.steps, 'scaling': 'weak', 'dtype': 'f32',
            'config': {'workload': f'configs[0] shape with the item profiles handed over as MixedRows: 966 multi-hot columns as index lists (mean {nnz / BATCH:.1f} non-zeros '
                                   f'per row) + 1,128 dense columns; {nb} batches of {BATCH} per step, eager launches', 'l2': 'inputs 69 MB per step'},
            'dense_form_same_batches': {'value': pairs / (ms_d * 1e-3), 'ms_per_step': ms_d / args.steps},
            'roofline': roof, 'parity': par, 'gpu_launches': launches,
            'e2e': {'value': pairs / (ms_m * 1e-3), 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0, 'note': 'inputs resident; configs[0] carries the host-fed leg'}}


PARALLELISM = {
    'peer': 'users 1-D nnz-partitioned over {P} GPUs, item rows in {P} equal ranges; no library collective on the data path: K3 pushes partial item rows '
            'into the owner\'s receive slot over NVLink (reduce-scatter fused into the SpMM epilogue), slots summed in rank order, K1c writes the '
            'transformed item rows into every rank\'s table (all-gather fused into the GEMM epilogue), epoch flags in peer memory order the '
            'ranks, batch rows pushed by their owners (deeprecommendation_b200/peer.py, csrc/peer.cu)',
    'reduce': 'users 1-D nnz-partitioned over {P} GPUs, items replicated; one NCCL all-reduce of the (nI, d) item partials per non-final layer, hidden '
              'behind the user-row SpMM; batch rows by all-reduce',
    'gather': 'item and user rows each 1-D nnz-partitioned over {P} GPUs; two NCCL all-gathers per layer, the larger one hidden behind the first '
              'SpMM; batch rows by all-reduce'}


def graph_leg(args, dev, rank, world, dist, peaks):
    """GraphNCF propagation, BASELINE configs[2] (strong scaling).  Returns (entry, compact scaling summary, {name: outputs of the
    last timed step} for --dump-outputs)."""
    w = build_graph(dev, args.graph_scale, 1, args.graph_scheme)
    w['eager'] = args.eager
    w['dump'] = bool(args.dump_outputs)
    single_ms = None
    if world > 1:
        # the 1-GPU step of the SAME graph in the SAME job, BEFORE the graph is partitioned: every rank holds the whole graph and times the
        # unpartitioned forward on its own GPU (no collective in it); the slowest rank's figure is the denominator of `speedup_vs_1gpu`
        w['train_leg'] = False
        n1 = max(3, args.steps // 2)
        r1 = run_graph(w, n1, 3, None, dev, peaks)
        single_ms = _max_over_ranks(dist, r1['ms'] / n1, dev)
        from deeprecommendation_b200.parallel import partition_graph
        partition_graph(w['graph'], scheme=args.graph_scheme, d_max=w['d'], batch_max=BATCH)
    w['train_leg'] = world == 1 and not args.no_train_step
    r = run_graph(w, args.steps, args.warmup, dist, dev, peaks)
    msgs = 2.0 * w['E'] * w['L'] * args.steps          # the graph is fixed: strong scaling
    entry = {'metric': 'GNN propagation directed-edge messages/sec (GraphNCF fwd)', 'value': msgs / (r['ms'] * 1e-3),
             'unit': 'edges/s', 'ms_per_step': r['ms'] / args.steps, 'n_gpus': world,
             'scaling': 'strong', 'parallelism': PARALLELISM[args.graph_scheme].format(P=world) if world > 1 else 'single GPU',
             'dtype': 'f32',
             'config': {'workload': f'configs[2]: GraphNCF L=2 d=128 hetero, synthetic MovieLens-25M shape (nU={w["nU"]}, nI={w["nI"]}, '
                        f'E={w["E"]}), pre-embedded (N,128) node features, whole-graph propagation + MLP on a batch of 512 per step',
                        'l2': 'CSR (400 MB) + features (115 MB) > L2', 'index_build_s': round(w['build_s'], 3),
                        'launch_mode': r['launch_mode'], 'scheme': args.graph_scheme if world > 1 else 'single'},
             'roofline': r['roofline'],
             'e2e': {'value': msgs / (r['e2e_ms'] * 1e-3), 'unit': 'edges/s', 'h2d_bytes_per_step': r['h2d'], 'd2h_bytes_per_step': r['d2h']},
             'gpu_launches': r['launches']}
    outputs = {'graph_scores': r['dump'][0]} if r['dump'] else {}
    if r.get('trace'):
        traces = [None] * world
        if dist is not None:
            dist.all_gather_object(traces, r['trace'])
        else:
            traces = [r['trace']]
        entry['device_trace_us'] = {f'rank{q}': t for q, t in enumerate(traces)}
    if r.get('train'):
        t = r['train']
        entry['train_step'] = ({'value': 2.0 * w['E'] * w['L'] / (t['ms'] * 1e-3), 'unit': 'edges/s', 'ms_per_step': t['ms'], 'steps': t['steps'],
                                'launch_mode': 'eager',
                                'what': 'whole-graph forward in train mode with the 512 target edges masked out (pair hash + skip bitmap), conv and '
                                        'MLP dropout, sum-MSE backward (K3 on the reverse-edge weights, gradient GEMMs on K1a) and Adam; value counts '
                                        'the forward messages only (2E*L per step), like the inference line'} if 'ms' in t else t)
    w['train_leg'] = False
    bf16_ms = None
    if world == 1 or args.graph_scheme == 'peer':
        # bf16 message mode (north_star: rel <= 1e-2): the transform GEMM rounds t once to bf16, K3 gathers 2-byte features
        w['model'].message_dtype = 'bf16'
        try:
            n_steps = max(3, args.steps // 2)
            rb = run_graph(w, n_steps, 3, dist, dev, peaks)
            bf16_ms = rb['ms'] / n_steps
            if rb['dump']:
                outputs['graph_bf16_scores'] = rb['dump'][0]
            entry['bf16_mode'] = {'value': 2.0 * w['E'] * w['L'] * n_steps / (rb['ms'] * 1e-3), 'ms_per_step': rb['ms'] / n_steps, 'steps': n_steps,
                                  'dtype': 'bf16 messages, fp32 accumulate', 'roofline': rb['roofline'],
                                  'e2e': {'value': 2.0 * w['E'] * w['L'] * n_steps / (rb['e2e_ms'] * 1e-3), 'unit': 'edges/s',
                                          'h2d_bytes_per_step': rb['h2d'], 'd2h_bytes_per_step': rb['d2h']}}
        except Exception as e:
            entry['bf16_mode'] = {'error': repr(e)[:300]}
        w['model'].message_dtype = 'fp32'
    if single_ms is None:
        single_ms = r['ms'] / args.steps
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, cores, sample, cpu_out, gpu_out = cpu_graph(w)
        entry['cpu_baseline'] = {'value': v, 'unit': 'edges/s', 'cores': cores, 'kind': 'port', 'sample': sample}
        entry['parity'] = (_parity(gpu_out, cpu_out, 'oracle/restatement.py::graph_ncf_forward on the 4 % edge sample of the benchmarked graph '
                                                     '(the CUDA path rebuilt its index for the same sample)') if torch.is_tensor(gpu_out) else {'error': gpu_out})
    ms = r['ms'] / args.steps
    scaling = {'metric': entry['metric'], 'config': 'configs[2] MovieLens-25M shape, L=2, d=128, fp32', 'n_gpus': world, 'scheme': entry['config']['scheme'],
               'value': entry['value'], 'unit': 'edges/s', 'ms_per_step': round(ms, 4),
               'single_gpu_ms_per_step_same_job': round(single_ms, 4), 'speedup_vs_1gpu': round(single_ms / ms, 3), 'target_at_8': 7.0}
    if bf16_ms:
        scaling['bf16_messages'] = {'ms_per_step': round(bf16_ms, 4), 'value': 2.0 * w['E'] * w['L'] / (bf16_ms * 1e-3)}
    entry['speedup_vs_1gpu'] = scaling['speedup_vs_1gpu']
    return entry, scaling, outputs


ATT_WORKLOAD = ('configs[1]: AttentionNCF scoring, synthetic MovieLens-latest-small shape (610 users, 9724 items, 100836 ratings, '
                'F=2094 profiles, 128/128/128 + MLP [256,128]), batches of 512 pairs through forward(candidate_items, rated_items, '
                'user_matrix)')

DUMP_LIMIT = 64 << 20


def write_outputs(path, outputs):
    """--dump-outputs: one DIR/<name>.npy per array; float32 (float64 where the source is float64 or an integer array, which
    float64 holds exactly below 2^53)"""
    arrays = {k: (v.float() if v.is_floating_point() and v.element_size() <= 4 else v.double()).numpy() for k, v in outputs.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f'--dump-outputs: {total} bytes of outputs, more than the {DUMP_LIMIT} allowed')
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + '.npy'), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20,
                    help='timed steps K of the headline (attention), basic, graph and sparse legs; the other timed legs run a count derived from '
                         'K: allpairs max(3, K/4), graph bf16 mode max(3, K/2), attention '
                         'train max(3, K/2), graph train max(3, K/4), basic train 4K single batches, graph5 max(3, min(K, 10))')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='all', choices=['all', 'attention', 'graph', 'basic', 'allpairs', 'k3hbm', 'k2hbm', 'graph5', 'allpairs_full', 'sparse'])
    ap.add_argument('--allpairs-users', type=int, default=APF_USERS, help='total users of the configs[3] full run (default 10^6)')
    ap.add_argument('--graph5-scale', type=float, default=1.0, help='configs[4] at a fraction of its size (users, items and edges scaled together)')
    ap.add_argument('--graph-scale', type=float, default=1.0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--gemm', default='bf16x3', choices=['simt', 'tf32x3', 'bf16', 'bf16x3'],
                    help='K1a engine for large-M linears: fp32 FFMA, tcgen05 3xTF32 (fp32 parity), the same with the wide form on a bf16 hi/lo split (fp32 parity, default) or plain tcgen05 bf16')
    ap.add_argument('--skip-hbm-regime', action='store_true')
    ap.add_argument('--no-train-step', action='store_true', help='skip the eager train-step legs (AttentionNCF, GraphNCF)')
    ap.add_argument('--graph-scheme', default='peer', choices=['peer', 'reduce', 'gather'],
                    help="multi-GPU GraphNCF: 'peer' = users partitioned, the exchange fused into this library's kernels over peer-mapped "
                         "memory (deeprecommendation_b200/peer.py); 'reduce' / 'gather' = the same partitions with NCCL collectives issued "
                         "from Python (deeprecommendation_b200/parallel.py), kept as the comparison baseline")
    ap.add_argument('--eager', action='store_true', help='do not capture the steps into CUDA graphs')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the attention, basic, allpairs and graph legs returned in their last timed step '
                         'as DIR/<name>.npy (float32, integer arrays as float64): all batches of an attention step, the last batch of a basic '
                         'step (its captured forward reuses one output buffer per batch), the top-k of an allpairs step, the scores of a graph '
                         'step; the inputs are seeded, so two builds can be compared')
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != 'b200' or args.workload not in ('all', 'attention', 'basic', 'allpairs', 'graph')):
        ap.error('--dump-outputs covers the attention, basic, allpairs and graph legs of --impl b200')
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup

    if args.impl == 'reference':
        reference_arm(args)
        return

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    numa = bind_to_gpu_numa(local) if world > 1 else None
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')      # stdout carries exactly one JSON line, whatever NCCL_DEBUG says
        dist_mod.init_process_group('nccl', device_id=dev)
        dist = dist_mod
    peaks = _peaks()
    result, also, outputs = None, [], {}
    from deeprecommendation_b200 import ops as _ops
    _ops.set_gemm_engine(args.gemm)

    with ClockSampler(local) as clocks:
        if args.workload in ('all', 'attention'):
            w = build_attention(dev, rank)
            w['gemm'] = args.gemm
            w['no_train'] = world > 1 or args.no_train_step              # the train-step leg is single-GPU (no gradient all-reduce: out of scope, SURVEY.md §8e)
            w['eager'] = args.eager
            w['dump'] = bool(args.dump_outputs)
            r = run_attention(w, args.steps, args.warmup, dist, dev, peaks)
            if r['dump']:
                outputs['attention_scores'] = torch.stack(r['dump'])        # (batches per step, 512, 1)
            pairs = BATCH * r['nb'] * args.steps * world
            result = {'metric': 'scored user-item pairs/sec (NCF fwd)', 'value': pairs / (r['ms'] * 1e-3), 'unit': 'pairs/s',
                      'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': r['ms'] / args.steps,
                      'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                      'config': attention_config(world, args.gemm),
                      'run_info': {'mean_rated_union_I': r['I_mean'], 'mean_nnz_per_batch': r['nnz_mean'], 'launch_mode': r['launch_mode'],
                                   'pairs_per_step_per_gpu': BATCH * r['nb']},
                      'roofline': r['roofline'],
                      'e2e': {'value': pairs / (r['e2e_ms'] * 1e-3), 'unit': 'pairs/s', 'h2d_bytes_per_step': r['h2d'],
                              'd2h_bytes_per_step': r['d2h'], 'ms_per_step': r['e2e_ms'] / args.steps},
                      'gpu_launches': r['launches']}
            if r.get('e2e_res'):
                result['e2e_resident'] = {'value': pairs / (r['e2e_res']['ms'] * 1e-3), 'unit': 'pairs/s', 'h2d_bytes_per_step': r['e2e_res']['h2d'],
                                          'd2h_bytes_per_step': r['d2h'], 'ms_per_step': r['e2e_res']['ms'] / args.steps,
                                          'note': 'same batches through content_providers.ResidentDynamicProvider + AttentionNCF.forward_resident: '
                                                  'profile table resident in HBM, per step only row numbers + the CSR of user_matrix are copied '
                                                  '(pinned host -> device) and the scores read back; `e2e` above is the dense 6-tuple contract'}
            if r.get('e2e_ids'):
                t = r['e2e_ids']
                result['e2e_device_collate'] = ({'value': pairs / (t['ms'] * 1e-3), 'unit': 'pairs/s', 'h2d_bytes_per_step': t['h2d'],
                                                 'd2h_bytes_per_step': r['d2h'] + t['d2h_extra'], 'ms_per_step': t['ms'] / args.steps,
                                                 'bit_equal_to_dense_contract': t['bit_equal_to_dense_contract'],
                                                 'host_collate_ms_per_batch': t['host_collate_ms_per_batch'],
                                                 'note': 'from (user, item) samples: DeviceCollateProvider.collate_device (K6: rated-item union + CSR of user_matrix built '
                                                         'on the device from the resident rating lists, dynamic_profiles_provider.py:30-73) + AttentionNCF.forward_resident; '
                                                         'the collate is INSIDE the timed region (`e2e` and `e2e_resident` start from batches collated beforehand on the '
                                                         'host: `host_collate_ms_per_batch` is what that numpy collate costs per batch)'} if 'ms' in t else t)
            if r.get('serving'):
                result['serving'] = r['serving']
            if r.get('train'):
                t = r['train']
                result['train_step'] = ({'value': BATCH * world / (t['ms'] * 1e-3), 'unit': 'pairs/s', 'ms_per_step': t['ms'], 'steps': t['steps'],
                                         'launch_mode': t.get('launch_mode', 'eager'), 'op_ms_per_step': t['op_ms_per_step'],
                                         'what': 'forward in train mode (MLP dropout 0.2, AttentionNet inner dropout 0.2 as a Philox mask inside K2, isclose target mask) '
                                                 '+ sum-MSE backward + Adam on the same batches: K2 backward = attention_pool_bwd_kernel, forward and gradient '
                                                 'GEMMs on K1a, torch elementwise ops for the MLP dropout masks / bias sums / the optimizer'} if 'ms' in t else t)
            if rank == 0 and world == 1 and not args.no_cpu_baseline:
                v, cores, sample, cpu_out = cpu_attention(w)
                result['cpu_baseline'] = {'value': v, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port', 'sample': sample}
                result['parity'] = _parity(r['out0'], cpu_out, 'oracle/restatement.py::attention_ncf_forward on batch 0 of the benchmarked config')
                if r.get('serving') and 'ms_per_request' in r['serving']:
                    try:
                        result['serving']['cpu_ms_per_request'] = cpu_serving(w)
                    except Exception as e:
                        result['serving']['cpu_error'] = repr(e)[:200]
                if r.get('train') and 'ms' in r['train']:
                    try:
                        tv, tsample = cpu_attention_train(w)
                        result['cpu_baseline']['train_step_value'] = tv
                        result['cpu_baseline']['train_step_sample'] = tsample
                    except Exception as e:
                        result['cpu_baseline']['train_step_error'] = repr(e)[:200]
            del w
            torch.cuda.empty_cache()
        if args.workload in ('all', 'basic'):
            w = build_basic(dev, rank)
            w['eager'] = args.eager
            w['dump'] = bool(args.dump_outputs)
            r = run_basic(w, args.steps, args.warmup, dist, dev, peaks)
            if r['dump']:
                outputs['basic_scores'] = r['dump'][0]
            pairs = BATCH * r['nb'] * args.steps * world
            entry = {'metric': 'scored user-item pairs/sec (BasicNCF fwd)', 'value': pairs / (r['ms'] * 1e-3), 'unit': 'pairs/s',
                     'ms_per_step': r['ms'] / args.steps, 'scaling': 'weak', 'dtype': 'f32',
                     'config': {'workload': 'configs[0] shape: BasicNCF(2094, 2094, 128, 128, [256]) forward, batches of 512 (user, item) '
                                'profile pairs', 'batches_per_step': r['nb'], 'l2': f'one step = {len(w["host"])} rotating batches (275 MB of inputs) > L2',
                                'launch_mode': r.get('launch_mode')},
                     'roofline': r['roofline'],
                     'e2e': {'value': pairs / (r['e2e_ms'] * 1e-3), 'unit': 'pairs/s', 'h2d_bytes_per_step': r['h2d'], 'd2h_bytes_per_step': r['d2h']},
                     'gpu_launches': r['launches']}
            for name, t in (r.get('res_legs') or {}).items():
                entry[name] = ({'value': pairs / (t['ms'] * 1e-3), 'unit': 'pairs/s', 'h2d_bytes_per_step': t['h2d'], 'd2h_bytes_per_step': r['d2h'],
                                'ms_per_step': t['ms'] / args.steps, 'max_rel_vs_dense_contract': t['max_rel_vs_dense_contract'],
                                'bit_equal_to_dense_contract': t['bit_equal_to_dense_contract'],
                                'note': ('content_providers.ResidentProfilesProvider + BasicNCF.forward_resident: both profile tables resident in HBM, a batch is '
                                         '2 x 512 row numbers; ' + ('every table row projected ONCE per weight version (cache_eval_embeddings, inference only), a batch '
                                                                    'is one MLP-tower launch over gathered embedding rows — not the per-batch projection `value` times'
                                                                    if name.endswith('cached') else 'rows gathered on the device, then the kernels of the dense contract'))}
                               if 'ms' in t else t)
            if r.get('train_ms'):
                entry['train_step'] = {'value': BATCH * args.steps * world / (r['train_ms'] * 1e-3), 'unit': 'pairs/s', 'ms_per_step': r['train_ms'] / args.steps,
                                       'launch_mode': r.get('train_mode'),
                                       'what': 'forward (dropout 0.2) + sum-MSE backward + Adam on the same batches; forward and gradient GEMMs on K1a, '
                                               'torch elementwise ops for masks / bias sums / the optimizer'}
            if rank == 0 and world == 1 and not args.no_cpu_baseline:
                v, cores, sample, cpu_out = cpu_basic(w)
                entry['cpu_baseline'] = {'value': v, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port', 'sample': sample}
                entry['parity'] = _parity(r['out0'], cpu_out, 'oracle/restatement.py::basic_ncf_forward on batch 0 of the benchmarked config')
                entry['cpu_baseline']['train_step_value'] = cpu_basic_train(w)
            if result is None:
                result = entry
            else:
                also.append(entry)
            del w
            torch.cuda.empty_cache()
        if args.workload in ('all', 'allpairs'):
            w = build_allpairs(dev, rank)
            w['dump'] = bool(args.dump_outputs)
            entry = None
            for precision in ('fp32', 'bf16'):
                r = run_allpairs(w, max(3, args.steps // 4), 3, dist, dev, peaks, precision)
                if r['dump']:
                    outputs[f'allpairs_{precision}_topk_scores'], outputs[f'allpairs_{precision}_topk_items'] = r['dump']
                n_steps = max(3, args.steps // 4)
                e = {'metric': f'scored user-item pairs/sec (BasicNCF all-pairs + top-{AP_K})', 'value': r['pairs'] * n_steps * world / (r['ms'] * 1e-3),
                     'unit': 'pairs/s', 'ms_per_step': r['ms'] / n_steps, 'steps': n_steps, 'scaling': 'weak',
                     'parallelism': f'dp{world}: users sharded, catalogue replicated, no collective', 'dtype': 'f32' if precision == 'fp32' else 'bf16',
                     'config': {'workload': f'configs[3] slab: BasicNCF(2094, 2094, 128, 128, [256,128]).recommend — {AP_USERS} users x {AP_ITEMS} items '
                                            f'per GPU and step (configs[3] = 211 such slabs per 10^6 users), F=2094 profiles in, top-{AP_K} per user out; '
                                            'embeddings + layer-1 halves by K1a, the rest fused in K5',
                                'precision': 'fp32 tolerance (bf16 hi/lo split operands, rel <= 1e-5)' if precision == 'fp32' else 'bf16 operands (rel <= 1e-2)',
                                'l2': 'item tables 100k x 1 KB = 102 MB streamed once per 32 users; profiles 838 MB > L2'},
                     'roofline': r['roofline'],
                     'e2e': {'value': r['pairs'] * n_steps * world / (r['e2e_ms'] * 1e-3), 'unit': 'pairs/s', 'h2d_bytes_per_step': r['h2d'], 'd2h_bytes_per_step': r['d2h']},
                     'gpu_launches': r['launches']}
                if entry is None:
                    entry = e
                else:
                    entry['bf16_mode'] = {k: e[k] for k in ('value', 'ms_per_step', 'roofline', 'e2e', 'dtype')}
            if rank == 0 and world == 1 and not args.no_cpu_baseline:
                v, cores, sample, par = cpu_allpairs(w)
                entry['cpu_baseline'] = {'value': v, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port', 'sample': sample}
                entry['parity'] = par
            if result is None:
                result = entry
            else:
                also.append(entry)
            del w
            torch.cuda.empty_cache()
    if args.workload in ('all', 'k3hbm') and world == 1 and not args.skip_hbm_regime:
        try:
            also.append(run_k3_hbm_regime(dev, peaks))
        except Exception as e:
            also.append({'metric': 'K3 HBM regime', 'error': repr(e)[:300]})
    if args.workload in ('all', 'k2hbm') and world == 1 and not args.skip_hbm_regime:
        try:
            also.append(run_k2_hbm_regime(dev, peaks))
        except Exception as e:
            also.append({'metric': 'K2 HBM regime', 'error': repr(e)[:300]})
    if args.workload in ('all', 'sparse') and world == 1:
        try:
            also.append(run_sparse(args, dev, rank, world, dist, peaks))
        except Exception as e:
            also.append({'metric': 'K1s sparse projection', 'error': repr(e)[:400]})
        torch.cuda.empty_cache()
    if args.workload == 'allpairs_full' or (args.workload == 'all' and world == 8):  # configs[3] names 8 GPUs; other sizes on request
        try:
            also.append(run_allpairs_full(args, dev, rank, world, dist, peaks, args.allpairs_users))
        except Exception as e:
            also.append({'metric': 'scored user-item pairs/sec (BasicNCF all-pairs, configs[3] in full)', 'error': repr(e)[:400]})
        torch.cuda.empty_cache()
    if args.workload == 'graph5' or (args.workload == 'all' and world == 8):       # configs[4] names 8 GPUs; other sizes on request
        try:
            also.append(run_graph5(args, dev, rank, world, dist, peaks, args.graph5_scale))
        except Exception as e:
            also.append({'metric': 'GNN propagation directed-edge messages/sec (GraphNCF fwd, configs[4])', 'error': repr(e)[:400]})
        torch.cuda.empty_cache()
    graph_scaling = None
    if args.workload in ('all', 'graph'):                  # LAST, so that the tail of the line carries the strong-scaling leg
        with ClockSampler(local) as gclocks:
            entry, graph_scaling, graph_outputs = graph_leg(args, dev, rank, world, dist, peaks)
        outputs.update(graph_outputs)
        if args.workload == 'graph':
            clocks = gclocks
        else:
            entry['clocks'] = gclocks.summary()
        also.append(entry)
    if result is None:
        result, also = also[0], also[1:]
    result.setdefault('config', {}).setdefault('gemm_engine', args.gemm)
    for k, v in (('n_gpus', world), ('steps', args.steps), ('warmup', args.warmup), ('higher_is_better', True), ('vs_baseline', None),
                 ('data', 'synthetic')):
        result.setdefault(k, v)
    result['clocks'] = clocks.summary()
    if numa is not None:
        result['host_binding'] = numa
    for e in [result] + also:                               # every roofline object says where its `traffic` figure comes from
        for ro in (e.get('roofline'), (e.get('bf16_mode') or {}).get('roofline')):
            if isinstance(ro, dict) and 'traffic' in ro:
                ro.setdefault('traffic_source', 'profiles/traffic.json (static: one `ncu --set full` capture of this kernel per round, not measured in this run)')
    if also:
        result['also'] = also
    if graph_scaling is not None:
        result['graph_scaling'] = graph_scaling            # compact copy of the strong-scaling leg at the very end of the line
    if rank == 0 and args.dump_outputs:
        write_outputs(args.dump_outputs, outputs)
    if rank == 0:
        print(json.dumps(result), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
