"""AttentionNCF.recommend (K8) and AttentionNCF.explain (K9) at config 2 and on a catalogue larger than L2, against the per-user
`recommend_for_user` loop (which ranks and explains) in the same run.

    python tools/attention_recommend_bench.py [--out FILE.json] [--large-users N] [--large-items N]

Config 2 = the inputs of bench.py's build_attention (synth.interactions_small(610, 9724, 100_836, seed=42), item profiles seed 43, weights
seed 1, item_emb = user_emb = att_dense = 128, MLP [256, 128]): all 610 users x the catalogue, top-10.  Call times are host clocks around
calls bracketed by a device synchronise; per-op times come from CUDA events of one extra call (ops.OpTimer).  The operation-count model
is computed from the shapes and printed as an estimate, never as a measurement."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deeprecommendation_b200 import ops, synth                                          # noqa: E402
from deeprecommendation_b200.content_providers import DeviceCollateProvider             # noqa: E402
from deeprecommendation_b200.neural_collaborative_filtering.models import AttentionNCF  # noqa: E402

KW = dict(item_emb=128, user_emb=128, att_dense=128, mlp_dense_layers=[256, 128], dropout_rate=0.2)


def gpu_info():
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True,
                           timeout=30)
        name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(',')]
        return {'name': name, 'power_limit': power, 'max_sm_clock': clock}
    except Exception as e:                                                     # the device name from torch is still recorded
        return {'name': torch.cuda.get_device_name(0), 'nvidia_smi_error': repr(e)[:200]}


def setup(n_users, n_items, n_ratings, seed, profile_seed, dev, whole_catalogue=False):
    users_raw, items_raw, ratings = synth.interactions_small(n_users, n_items, n_ratings, seed=seed)
    _, u = synth.dense_ids(users_raw)
    if whole_catalogue:                  # every one of the n_items items is a candidate, rated or not (movieId = 7 k + 1)
        it, nI = (items_raw - 1) // 7, n_items
    else:                                # bench.py's build_attention: the catalogue is the set of rated items
        item_ids, it = synth.dense_ids(items_raw)
        nI = len(item_ids)
    profiles = synth.item_profiles(nI, seed=profile_seed)
    row_ptr, idx, rr, _ = synth.user_rating_lists(u, it, ratings, n_users)
    prov = DeviceCollateProvider(np.arange(nI), profiles, np.arange(n_users), row_ptr, idx, rr, device=dev)
    model = AttentionNCF(item_dim=profiles.shape[1], **KW).to(dev).eval()
    model.load_state_dict(synth.to_torch(synth.attention_ncf_weights(item_dim=profiles.shape[1], seed=1, **KW)))
    return model, prov, row_ptr, idx, rr


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def op_model(list_lens, nI, H, H1, clock_ghz, sms=148):
    inter = float(np.sum(list_lens)) * nI
    lane = inter * (3 * H + H1)
    return {'what': 'ESTIMATE from shapes, not a measurement: (candidate, list entry) interactions = sum of list lengths x catalogue; '
                    'lane-instructions ~ 3·H per interaction for the scores (FADD, FMNMX, FFMA) + H1 for the pooling (FFMA)',
            'interactions': inter, 'lane_instructions': lane, 'clock_ghz': clock_ghz,
            'fp32_bound_ms': lane / (sms * 128 * clock_ghz * 1e9) * 1e3}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--large-users', type=int, default=1000)
    ap.add_argument('--large-items', type=int, default=100_000)
    ap.add_argument('--reps', type=int, default=7)
    a = ap.parse_args()
    dev = torch.device('cuda:0')
    res = {'device': gpu_info()}
    H, H1 = KW['att_dense'], KW['mlp_dense_layers'][0]

    # ---------------- config 2 ----------------
    model, prov, row_ptr, idx, rr = setup(610, 9724, 100_836, 42, 43, dev)
    lists = (prov.table, prov.d_list_ptr, prov.d_list_item, prov.d_list_val)
    nI, nU = prov.table.shape[0], 610
    first_ms, _ = timed(lambda: model.recommend(*lists, k=10))
    model.invalidate_caches()
    cold_ms, _ = timed(lambda: model.recommend(*lists, k=10))
    for _ in range(2):
        model.recommend(*lists, k=10)
    warm = [timed(lambda: model.recommend(*lists, k=10))[0] for _ in range(a.reps)]
    model.invalidate_caches()
    tables_ms, _ = timed(lambda: model._recommend_tables(prov.table))
    timer = ops.OpTimer()
    prev = ops.set_timer(timer)
    model.recommend(*lists, k=10)
    torch.cuda.synchronize()
    ops.set_timer(prev)
    per_op = {}
    for (name, meta), v in timer.summary().items():
        per_op.setdefault(name, 0.0)
        per_op[name] += sum(v)
    val, items, scores = model.recommend(*lists, k=10, return_scores=True)

    # explanations of the same top-10 (K9), on the tables recommend() cached
    for _ in range(2):
        model.explain(*lists, items)
    explain_warm = [timed(lambda: model.explain(*lists, items))[0] for _ in range(a.reps)]
    timer = ops.OpTimer()
    prev = ops.set_timer(timer)
    for _ in range(a.reps):
        expl = model.explain(*lists, items)
    torch.cuda.synchronize()
    ops.set_timer(prev)
    explain_ops = {name: statistics.median(v) for (name, _), v in timer.summary().items()}

    # the per-user loop of the existing serving call, same users, end to end
    pos = [torch.from_numpy(idx[row_ptr[u]:row_ptr[u + 1]].astype(np.int64)).to(dev) for u in range(nU)]
    rat = [torch.from_numpy(rr[row_ptr[u]:row_ptr[u + 1]].astype(np.float64)).to(dev) for u in range(nU)]
    for u in range(20):
        model.recommend_for_user(prov.table, pos[u], rat[u], k=10)
    loop_ms, recs = timed(lambda: [model.recommend_for_user(prov.table, pos[u], rat[u], k=10) for u in range(nU)])
    same_items = sum(int(torch.equal(items[u], recs[u]['items'])) for u in range(nU))
    top_rel = max(float((val[u] - recs[u]['scores']).abs().max() / recs[u]['scores'].abs().max()) for u in range(nU))
    e_ptr, e_because = expl[0].tolist(), expl[1]
    same_because = sum(int(torch.equal(e_because[e_ptr[u * 10 + j]:e_ptr[u * 10 + j + 1]], recs[u]['because'][j]))
                       for u in range(nU) for j in range(10) if torch.equal(items[u], recs[u]['items']))
    loop_entries = sum(int(b.numel()) for r in recs for b in r['because'])

    # parity on sampled users against forward (K2 path) over the same (user, unseen item) pairs
    sample = np.random.default_rng(0).choice(nU, 16, replace=False)
    par = []
    with torch.no_grad():
        for u in sample:
            r = pos[u]
            keep = torch.ones(nI, dtype=torch.bool, device=dev)
            keep[r] = False
            cand = keep.nonzero().view(-1)
            um = prov.d_list_val[row_ptr[u]:row_ptr[u + 1]].view(1, -1).expand(cand.numel(), -1).contiguous()
            y = model(prov.table[cand], prov.table[r], um).view(-1).double()
            par.append(float((scores[u, cand].double() - y).abs().max() / y.abs().max()))
    lens = np.diff(row_ptr)
    clock = res['device'].get('max_sm_clock', '')
    try:
        clock_ghz = float(clock.split()[0]) / 1e3
    except (ValueError, IndexError):
        clock_ghz = 1.36
    med = statistics.median(warm)
    res['config2'] = {
        'users': nU, 'items': nI, 'k': 10, 'pairs': nU * nI, 'list_entries': int(lens.sum()), 'longest_list': int(lens.max()),
        'recommend_ms_median': med, 'recommend_ms_all': warm, 'pairs_per_s': nU * nI / (med * 1e-3),
        'first_call_in_process_ms': first_ms, 'cold_call_ms_incl_tables': cold_ms, 'tables_ms': tables_ms,
        'per_op_ms_one_warm_call (CUDA events)': per_op,
        'baseline_recommend_for_user_loop_ms': loop_ms, 'speedup_vs_loop': loop_ms / med,
        'top10_items_identical_to_loop_users': same_items, 'top10_scores_max_rel_vs_loop': top_rel,
        'parity_vs_forward_sampled_users': len(sample), 'parity_max_rel': max(par),
        'op_model': op_model(lens, nI, H, H1, clock_ghz),
        'explain': {
            'explain_ms_median': statistics.median(explain_warm), 'explain_ms_all': explain_warm,
            'explain_over_recommend': statistics.median(explain_warm) / med,
            'kernel_ms_median (CUDA events)': explain_ops,
            'explanations': int(e_ptr[-1]), 'explanations_in_loop': loop_entries,
            'rows_with_because_identical_to_loop': same_because, 'rows': nU * 10,
            'op_model': {'what': 'ESTIMATE from shapes, not a measurement: 3 passes over each user list for each of its k candidates, ~3·H '
                                 'lane-instructions per (candidate, entry) score',
                         'lane_instructions': 3.0 * 10 * float(lens.sum()) * 3 * H,
                         'longest_list_chunks_per_pass': int((lens.max() + 31) // 32)},
        },
    }
    del model, prov, scores
    torch.cuda.empty_cache()

    # ---------------- a catalogue larger than L2 ----------------
    nUl, nIl = a.large_users, a.large_items
    model, prov, row_ptr, _, _ = setup(nUl, nIl, int(round(100_836 / 610 * nUl)), 7, 44, dev, whole_catalogue=True)
    lists = (prov.table, prov.d_list_ptr, prov.d_list_item, prov.d_list_val)
    nIl = prov.table.shape[0]
    _, top = model.recommend(*lists, k=10)
    times = [timed(lambda: model.recommend(*lists, k=10))[0] for _ in range(3)]
    model.explain(*lists, top)
    explain_times = [timed(lambda: model.explain(*lists, top))[0] for _ in range(3)]
    tables = model._recommend_tables(prov.table)
    table_bytes = tables[0].shape[0] * tables[0].stride(0) * 4          # the four tables are views of one (nI, N) GEMM output
    lens = np.diff(row_ptr)
    res['large_catalogue'] = {'users': nUl, 'items': nIl, 'list_entries': int(lens.sum()), 'tables_bytes': table_bytes,
                              'recommend_ms_median': statistics.median(times), 'recommend_ms_all': times,
                              'pairs_per_s': nUl * nIl / (statistics.median(times) * 1e-3), 'op_model': op_model(lens, nIl, H, H1, clock_ghz),
                              'explain_top10_ms_median': statistics.median(explain_times), 'explain_top10_ms_all': explain_times}
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(txt + '\n')


if __name__ == '__main__':
    main()
