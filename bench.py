#!/usr/bin/env python
"""bench.py -- predict_rank throughput of the B200-native hot path (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload (BASELINE.json north_star / SURVEY.md 8d, "C5 at 1M x 1M"): predict_rank top-10 over 1M users x 1M items,
n_components = 128, indicator-regime sparse features (identity + 3 random tags per row, F = 1.2 R, ~4 nnz/row),
LinearRepresentationGraph x DotProductPredictionGraph, biased, n_tastes = 1.  Synthetic, seeded.

One step = one full pass of the hot path over the batch:
    K1 users -> split operand,  K1 items -> split operand,  2 x project_biases,  pack item meta,
    K2+K3 fused tcgen05 score + top-k,  merge           [N > 1: item axis sharded, + 1 NCCL all-gather, merge]
value  = U * I / step time with the CSR inputs and the weights already resident in HBM (CUDA events, max over ranks);
e2e    = the same metric through TensorRec.predict_rank(user_features, item_features, k) with HOST scipy matrices
         (pinned): host->device copy of the CSR arrays and device->host read of the top-k inside the timed region;
roofline: the fused kernel's algorithmic flops (2*U*I*d) / its CUDA-event time against the measured bf16 peak;
cpu_baseline: the oracle (numpy/scipy restatement of the reference's TF-CPU ops) on this box's host cores, on a
         bounded user sample of the same workload.
`--impl reference` times that oracle alone (TensorFlow, the reference's only back-end, cannot be installed)."""
import argparse
import concurrent.futures
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'predict_rank_pairs_per_s'
UNIT = 'pairs/s'


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------------------------------- inputs
def indicator_csr(rows, seed):
    """tensorrec/util.py:88-108 (indicator regime), vectorised and seeded; float32 CSR with sorted rows."""
    rng = np.random.default_rng(seed)
    n_features = int(rows * 1.2)
    n_tags = rows * 3
    r = np.concatenate([np.arange(rows, dtype=np.int64), rng.integers(0, rows, n_tags)])
    c = np.concatenate([np.arange(rows, dtype=np.int64), rng.integers(rows, n_features, n_tags)])
    m = sp.csr_matrix((np.ones(r.shape[0], dtype=np.float32), (r, c)), shape=(rows, n_features))
    m.sum_duplicates()
    m.data[:] = 1.0
    return m


def make_weights(n_features, d, seed):
    """representation_graphs.py:35-36: normal rows, L2-normalised (float32)."""
    rng = np.random.default_rng(seed)
    w = rng.standard_normal((n_features, d), dtype=np.float32)
    w /= np.sqrt(np.einsum('ij,ij->i', w, w, dtype=np.float32))[:, None]
    return w


def movielens_shaped(users, items, seed):
    """SURVEY C3 (examples/getting_started.py:57-58, 164): identity user features; item features = identity + 18 binary
    genre columns, 1-3 genres per item."""
    rng = np.random.default_rng(seed)
    uf = sp.identity(users, dtype=np.float32, format='csr')
    n_genres = rng.integers(1, 4, items)
    r = np.repeat(np.arange(items, dtype=np.int64), n_genres)
    c = items + rng.integers(0, 18, r.shape[0])
    itf = sp.csr_matrix((np.ones(items + r.shape[0], dtype=np.float32),
                         (np.concatenate([np.arange(items, dtype=np.int64), r]),
                          np.concatenate([np.arange(items, dtype=np.int64), c]))), shape=(items, items + 18))
    itf.sum_duplicates()
    itf.data[:] = 1.0
    return uf, itf


def make_problem(args):
    """--scores iid: the headline inputs (normal weights: continuous scores, ties have probability zero);
    ties: integer-valued weights and biases on the same features (massive exact ties: the reference's normal case before
    training -- indicator features, integer ratings); c3: MovieLens-shaped features, cosine prediction."""
    t0 = time.time()
    scores = getattr(args, 'scores', 'iid')
    if scores == 'c3':
        uf, itf = movielens_shaped(args.users, args.items, seed=0)
    else:
        uf = indicator_csr(args.users, seed=0)
        itf = indicator_csr(args.items, seed=1)
    rng = np.random.default_rng(4)
    if scores == 'const':
        wu = np.zeros((uf.shape[1], args.d), dtype=np.float32)
        wi = np.zeros((itf.shape[1], args.d), dtype=np.float32)
        bu = np.zeros(uf.shape[1], dtype=np.float32)
        bi = np.zeros(itf.shape[1], dtype=np.float32)
    elif scores == 'ties':
        wu = rng.integers(-2, 3, size=(uf.shape[1], args.d)).astype(np.float32)
        wi = rng.integers(-2, 3, size=(itf.shape[1], args.d)).astype(np.float32)
        bu = rng.integers(-3, 4, size=uf.shape[1]).astype(np.float32)
        bi = rng.integers(-3, 4, size=itf.shape[1]).astype(np.float32)
    else:
        wu = make_weights(uf.shape[1], args.d, seed=2)
        wi = make_weights(itf.shape[1], args.d, seed=3)
        bu = (0.1 * rng.standard_normal(uf.shape[1])).astype(np.float32)
        bi = (0.1 * rng.standard_normal(itf.shape[1])).astype(np.float32)
    log('[bench] synthetic problem built in %.1fs: users %s nnz %d, items %s nnz %d, d=%d'
        % (time.time() - t0, uf.shape, uf.nnz, itf.shape, itf.nnz, args.d))
    return uf, itf, wu, wi, bu, bi


# ----------------------------------------------------------------------------------------------------- CPU oracle leg
def cpu_oracle_leg(uf, itf, wu, wi, bu, bi, k, budget_s, threads, cosine=False):
    """Times the oracle (reference semantics: SpMM, fp32 GEMM, bias adds, the literal double full sort per user,
    then the rank <= k entries) on a bounded sample of users against ALL items.  Returns (pairs_per_s, description).

    The item-side work (item representation + item biases) is done once per predict_rank call by the reference; it is
    timed once and charged to the sample in proportion sample_users / total_users."""
    from oracle import reference_ops as R
    n_users, n_items = uf.shape[0], itf.shape[0]
    t0 = time.perf_counter()
    item_repr = R.sparse_dense_matmul_fast(itf, wi)
    if cosine:
        item_repr = R.l2_normalize(item_repr)
    item_bias = np.asarray(itf @ bi, dtype=np.float32)
    t_items = time.perf_counter() - t0

    def rank_rows(block):
        order = np.argsort(-block, axis=1, kind='stable').astype(np.int32)           # recommendation_graphs.py:81
        ranks = np.argsort(order, axis=1, kind='stable').astype(np.int32) + 1         # :82
        rows, cols = np.nonzero(ranks <= k)                                           # eval.py:23,49 read only these
        top = np.empty((block.shape[0], min(k, block.shape[1])), dtype=np.int32)
        top[rows, ranks[rows, cols] - 1] = cols
        return top

    def run(u0, u1):
        sub = uf[u0:u1]
        user_repr = R.sparse_dense_matmul_fast(sub, wu)
        if cosine:
            user_repr = R.l2_normalize(user_repr)
        user_bias = np.asarray(sub @ bu, dtype=np.float32)
        scores = R.bias_prediction_dense(R.dot_product_dense(user_repr, item_repr), user_bias, item_bias)
        rows_per = max(1, (u1 - u0 + threads - 1) // threads)
        blocks = [scores[i:i + rows_per] for i in range(0, u1 - u0, rows_per)]
        with concurrent.futures.ThreadPoolExecutor(max_workers=threads) as pool:
            return np.concatenate(list(pool.map(rank_rows, blocks)))

    chunk = max(threads, 8)
    chunk = min(chunk, n_users)
    t0 = time.perf_counter()
    first_top = run(0, chunk)       # kept: the GPU result of the same users is checked against it (full item axis)
    t_chunk = time.perf_counter() - t0
    n_chunks = int(max(1, min(budget_s / max(t_chunk, 1e-3), n_users // chunk)))
    t0 = time.perf_counter()
    done = 0
    for c in range(n_chunks):
        run(c * chunk, (c + 1) * chunk)
        done += chunk
        if time.perf_counter() - t0 > budget_s:
            break
    t_users = time.perf_counter() - t0
    total = t_users + t_items * done / float(n_users)
    desc = ('%d of %d users x all %d items, d=%d: scipy CSR SpMM + numpy fp32 GEMM + per-user double stable argsort '
            '(rank_predictions) + rank<=%d selection, %d threads; item-side time charged pro rata'
            % (done, n_users, n_items, wu.shape[1], k, threads))
    return done * float(n_items) / total, desc, total, first_top


# ----------------------------------------------------------------------------------------------------- clocks
class ClockSampler(object):
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '--query-gpu=' + self.QUERY, '--format=csv,noheader,nounits',
                                          '-lms', '100', '-i', str(self.gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.lines:
            f = [x.strip() for x in line.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, flag in zip(names, f[5:9]):
                if flag.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        busy = [s for s, p in zip(sm, power) if p >= 0.5 * max(power)] or sm
        return {'sm_mhz': float(np.median(busy)), 'sm_max_mhz': float(max(smax)), 'reasons': sorted(reasons),
                'power_w_max': float(max(power)), 'samples': len(sm)}


def ncu_traffic(kernel_key):
    """DRAM bytes (read + write) of one launch of the dominant kernel at the bench workload, from the committed ncu
    capture (profiles/ncu_traffic.json, written by scripts/ncu_summary.py runs); None if not captured."""
    path = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if os.path.exists(path):
        return json.load(open(path)).get(kernel_key)
    return None


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return {'hbm_gbs': p['hbm_gbs'], 'tflops_burst': p['bf16_tflops'],
                'tflops_sustained': p.get('bf16_tflops_sustained', p['bf16_tflops']), 'source': 'measured'}
    return {'hbm_gbs': 6650.0, 'tflops_burst': 1590.0, 'tflops_sustained': 1400.0, 'source': 'fallback'}


# ----------------------------------------------------------------------------------------------------- GPU arm
def workload_config(args):
    """`config` of the JSON line: IDENTICAL in both arms (the driver compares them); arm-specific facts go to `details`."""
    d_pad = ((args.d + 63) // 64) * 64
    f_users, f_items = int(args.users * 1.2), int(args.items * 1.2)
    operands_mb = (args.users + args.items) * 2 * d_pad * 2 / 1e6
    tables_mb = (f_users + f_items) * args.d * 4 / 1e6
    return {'workload': workload_string(args),
            'l2': 'split operands %.0f MB, weight tables %.0f MB against 126 MB of L2: %s'
                  % (operands_mb, tables_mb, 'inputs exceed L2, no flush between steps needed'
                     if min(operands_mb, tables_mb) > 126 else 'inputs FIT in L2 - a test size, not a bench line')}


def workload_string(args):
    """config.workload: the same string in both arms (the driver compares them)."""
    scores = getattr(args, 'scores', 'iid')
    if scores == 'c3':
        return ('predict_rank top-%d, %d users x %d items, d=%d, MovieLens-shaped features (identity users; identity + 18 '
                'genre columns items), LinearRepr x CosineSimilarity, biased (BASELINE configs[2] structure, SURVEY C3, '
                'scaled up)' % (args.k, args.users, args.items, args.d))
    return ('predict_rank top-%d, %d users x %d items, d=%d, indicator-regime features, LinearRepr x DotProduct, biased '
            '(BASELINE configs[4] shape at the size the metric is quoted on; SURVEY C5)%s'
            % (args.k, args.users, args.items, args.d,
               {'iid': '', 'ties': '; INTEGER-valued weights and biases: massive exact ties',
                'const': '; ALL weights and biases zero: every score equal, every row rejected by the certificate'}[scores]))


PHASES = ['k1_users', 'items_prep', 'filter', 'rescore', 'fallback', 'exchange', 'merge']


def oracle_topk_rows(uf, itf, wu, wi, bu, bi, rows, k, item_repr=None, item_bias=None, cosine=False):
    """Reference-semantics top-k (oracle) of the given user rows against ALL items (CPU)."""
    from oracle import reference_ops as R
    if item_repr is None:
        item_repr = R.sparse_dense_matmul_fast(itf, wi)
        if cosine:
            item_repr = R.l2_normalize(item_repr)
        item_bias = np.asarray(itf @ bi, dtype=np.float32)
    out = np.empty((len(rows), k), dtype=np.int32)
    for c0 in range(0, len(rows), 512):
        sub = uf[rows[c0:c0 + 512]]
        user_repr = R.sparse_dense_matmul_fast(sub, wu)
        if cosine:
            user_repr = R.l2_normalize(user_repr)
        user_bias = np.asarray(sub @ bu, dtype=np.float32)
        scores = R.bias_prediction_dense(R.dot_product_dense(user_repr, item_repr), user_bias, item_bias)
        out[c0:c0 + 512] = R.top_k_from_scores_fast(scores, k)[0]
    return out, item_repr, item_bias


DUMP_BYTES = 48 << 20      # --dump-outputs budget: a seeded row sample keeps larger results under 64 MB


def dump_topk(out_dir, top, first_user):
    """Writes the top-k a caller of the timed path receives (item ids, scores) for a fixed, seeded sample of its user
    rows (all rows when they fit DUMP_BYTES), with the global user id of every row.  Ids are stored as float64 (exact
    for any int32), scores as float32."""
    import torch
    n_users, k = top.items.shape
    n_rows = min(n_users, DUMP_BYTES // (8 + k * (8 + 4)))
    rows = np.arange(n_users) if n_rows == n_users else \
        np.sort(np.random.default_rng(0).choice(n_users, n_rows, replace=False))
    idx = torch.from_numpy(rows).to(top.items.device)
    os.makedirs(out_dir, exist_ok=True)
    arrays = {'user_ids': (rows + first_user).astype(np.float64),
              'topk_items': top.items[idx].cpu().numpy().astype(np.float64),
              'topk_scores': top.scores[idx].cpu().numpy().astype(np.float32)}
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), arr)
    log('[bench] wrote %s (%d of %d user rows, top-%d)' % (', '.join(n + '.npy' for n in arrays), n_rows, n_users, k))


def run_b200(args):
    import torch
    import torch.distributed as dist
    import tensorrec_b200
    from tensorrec_b200 import kernels
    from tensorrec_b200.distributed import shard_bounds, exchange_rows

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus:
        log('[bench] note: --gpus %d but WORLD_SIZE=%d; using WORLD_SIZE' % (args.gpus, world))
    kernels.require_cuda()
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)

    uf, itf, wu, wi, bu, bi = make_problem(args)
    n_users, n_items, d, k = args.users, args.items, args.d, args.k
    d_pad = kernels.d_pad_for(d)
    # item axis sharded over ranks (SURVEY 8e); --emulate-shards N times ONE shard of N on one GPU (development aid)
    # Layout of the ranks: item_shards ranks form one ITEM GROUP (they split the item axis and exchange their per-shard
    # top-k); world / item_shards such groups split the users.  Default item_shards = world: the item axis sharded over all
    # GPUs (BASELINE north_star); --item-shards S < world is the grid form (users are independent: no collective
    # between groups).
    item_shards = world if args.item_shards in (None, 0) else int(args.item_shards)
    if world % item_shards != 0:
        raise SystemExit('--item-shards %d does not divide the %d ranks' % (item_shards, world))
    n_groups = world // item_shards
    user_group, item_rank = rank // item_shards, rank % item_shards
    item_group = None
    if world > 1:
        for g in range(n_groups):
            grp = dist.new_group(list(range(g * item_shards, (g + 1) * item_shards)))
            if g == user_group:
                item_group = grp
    n_shards = args.emulate_shards if (world == 1 and args.emulate_shards > 1) else item_shards
    lo, hi = shard_bounds(n_items, n_shards, item_rank if world > 1 else 0)
    itf_local = itf[lo:hi]
    n_local = hi - lo
    g_lo, g_hi = shard_bounds(n_users, n_groups, user_group)       # the users of this rank's group
    uf_all, n_users_all = uf, n_users
    uf, n_users = uf[g_lo:g_hi], g_hi - g_lo                       # from here on: the group's users
    s_lo, s_hi = shard_bounds(n_users, item_shards, item_rank)     # ... of which this rank forms the final answer for
    u_lo, u_hi = g_lo + s_lo, g_lo + s_hi                          # (global user ids)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident inputs for `value` ------------------------------------------------------------------
    ucsr = kernels.DeviceCSR.from_scipy(uf, device=dev)
    icsr = kernels.DeviceCSR.from_scipy(itf_local, device=dev)
    wu_d, wi_d = torch.from_numpy(wu).to(dev), torch.from_numpy(wi).to(dev)
    bu_d, bi_d = torch.from_numpy(bu).to(dev), torch.from_numpy(bi).to(dev)
    phase_events = []

    use_filter = args.topk_path == 'filter' and k <= kernels.filter_max_k()
    last = {}
    cosine = args.scores == 'c3'
    n_norm = 1 if cosine else 0          # CosineSimilarityPredictionGraph: both representations L2-normalised in K1

    def step(record=False):
        marks = []

        def mark():
            if record:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                marks.append(e)

        mark()
        out = kernels.gather_reduce(ucsr, wu_d, n_normalize=n_norm, want_f32=False, split_d_pad=d_pad,
                                    want_norm=use_filter)
        us, usc = out[1], out[2]
        user_norm = out[3] if use_filter else None
        ub = kernels.project_biases(ucsr, bu_d)
        users = kernels.SideOperands(None, us, usc, ub, n_users, d, d_pad, norm=user_norm)
        mark()
        stats = torch.empty((3,), dtype=torch.float32, device=dev) if use_filter else None
        _, its, isc = kernels.gather_reduce(icsr, wi_d, n_normalize=n_norm, want_f32=False, split_d_pad=d_pad,
                                            stats=stats)
        ib = kernels.project_biases(icsr, bi_d)
        items = kernels.SideOperands(None, its, isc, ib, n_local, d, d_pad, stats=stats)
        if use_filter:
            fitems = kernels.FilterItems(items)      # bias-sorted processing order, global-scale hi, bias blocks
            mark()
            _, ci, theta = kernels.score_filter(us, usc, ub, user_norm, fitems.hi, fitems.stats, fitems.bias_pad,
                                                fitems.block_max, fitems.perm, n_users, n_local, d_pad, k,
                                                item_id_offset=lo, block_bias_min=fitems.block_min)
            mark()
            top, bad = kernels.rescore_topk(users, items, ci, theta, user_norm, fitems.stats, k, item_id_offset=lo)
            mark()
            # rows whose bound could not be certified go through the exact kernel, routed on the device
            counters, cap = kernels.rerun_uncertified(users, items, bad, top, k, item_id_offset=lo)
            last['counters'], last['cap'], last['bad'] = counters, cap, bad
            if args.scores != 'iid' and int(counters[0]) > cap:
                # more rejected rows than the device-side fallback holds (tie-heavy scores): what the API does at its
                # final synchronisation -- the whole batch through the exact kernel (this check synchronises)
                top = kernels.topk_exact(users, items, k, item_id_offset=lo)
                last['overflow'] = True
        else:
            meta = kernels.pack_item_meta(isc, ib, n_local)
            mark()
            cs, ci = kernels.score_topk(us, usc, ub, its, meta, n_users, n_local, d_pad, k, item_id_offset=lo)
            mark()
            top = kernels.topk_merge(cs, ci, k)
            mark()
        mark()
        if item_shards > 1:
            recv, _ = exchange_rows(top.buf, item_group)
            mark()
            top = kernels.topk_merge_received(recv, u_hi - u_lo, item_shards, k)
        else:
            mark()
        mark()
        if record:
            phase_events.append(marks)
        return top

    n_splits = kernels.default_splits(n_users, n_local)

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0 and not args.no_clocks:
        sampler.start()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches_before = tensorrec_b200._lib.launch_count
    start.record()
    for _ in range(args.steps):
        out = step(record=True)
    end.record()
    barrier()
    gpu_launches = tensorrec_b200._lib.launch_count - launches_before   # kernel-launching C-ABI calls, counted
    ms_total = start.elapsed_time(end)
    clocks = (sampler.stop() if not args.no_clocks else {'sm_mhz': None, 'reasons': ['sampling disabled']}) \
        if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_topk(args.dump_outputs, out, u_lo)
    t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    # whole job: all users x all items; --emulate-shards times ONE shard's pairs (development aid, not a bench value)
    pairs = n_users_all * float(n_local if (world == 1 and n_shards > 1) else n_items)
    value = pairs / (ms_step * 1e-3)
    # per-phase device time of this rank (means over the timed steps)
    phase_ms = np.zeros(len(PHASES))
    for marks in phase_events:
        for j in range(len(PHASES)):
            phase_ms[j] += marks[j].elapsed_time(marks[j + 1])
    phase_ms /= max(1, len(phase_events))
    fused_ms = float(phase_ms[PHASES.index('filter')])
    k1u_ms = float(phase_ms[PHASES.index('k1_users')])
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, phase_ms.tolist())
        all_phase = np.asarray(gathered)
    else:
        all_phase = phase_ms[None, :]
    n_check = min(args.parity_users, u_hi - u_lo)
    top_items_check = out.items[:n_check].cpu().numpy()      # compared with the CPU oracle's ranking below (rank 0)
    top_items_value = out.items[:4].cpu().numpy()
    fallback_rows, fallback_ids, fallback_items = 0, np.zeros(0, np.int64), None
    if use_filter:
        fallback_rows = int(last['counters'][0])
        bad_ids = torch.nonzero(last['bad'], as_tuple=True)[0]
        bad_ids = bad_ids[(bad_ids >= s_lo) & (bad_ids < s_hi)][:args.parity_fallback_rows]      # rows within the group
        fallback_ids = bad_ids.cpu().numpy() + g_lo                                               # global user ids
        fallback_items = out.items[bad_ids - s_lo].cpu().numpy()

    # ---- e2e: the public API with host buffers ----------------------------------------------------------
    def pinned_csr(m):
        arrs = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in (m.data, m.indices, m.indptr)]
        return sp.csr_matrix((arrs[0].numpy(), arrs[1].numpy(), arrs[2].numpy()), shape=m.shape), arrs

    del ucsr, icsr, out
    last_overflow = last.get('overflow', False)
    last.clear()
    tensorrec_b200.tensorrec.TOPK_PATH = 'auto' if use_filter else 'exact'
    model = tensorrec_b200.TensorRec(
        n_components=d, prediction_graph=(tensorrec_b200.prediction_graphs.CosineSimilarityPredictionGraph() if cosine
                                          else tensorrec_b200.prediction_graphs.DotProductPredictionGraph()))
    model.set_weights({'linear_weights_user_0': wu, 'linear_weights_item': wi, 'feature_biases_user': bu[:, None],
                       'feature_biases_item': bi[:, None]})
    uf_host, _keep_u = pinned_csr(uf)
    itf_host, _keep_i = pinned_csr(itf_local)
    group = item_group if item_shards > 1 else None

    def e2e_step():
        return model.predict_top_k(uf_host, itf_host, k, item_id_offset=lo, gather_group=group, gather='slice',
                                   user_batch_size=args.user_batch)

    held = []
    for _ in range(max(3, args.warmup)):      # results are held like in the timed loop: the page-locked pool warms up
        held.append(e2e_step())
    del held
    barrier()
    t0 = time.perf_counter()
    s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s2.record()
    for _ in range(args.steps):
        top = e2e_step()
    e2.record()
    barrier()
    wall = (time.perf_counter() - t0) * 1e3
    # host conversion and the blocking D2H sit between kernels: use the larger of the event and wall times
    e2e_ms = max(s2.elapsed_time(e2), wall)
    t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms_step = float(t.item()) / args.steps
    e2e_value = pairs / (e2e_ms_step * 1e-3)
    h2d = 4 * (uf.nnz * 2 + uf.shape[0] + 1 + itf_local.nnz * 2 + itf_local.shape[0] + 1)
    d2h = n_users_all * k * 8  # whole job: every rank reads back the top-k of ITS user slice
    same = bool(np.array_equal(top.items[:4], top_items_value))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    flops = 2.0 * n_users * n_local * d                        # algorithmic flops of one fused launch (this rank)
    achieved = flops / (fused_ms * 1e-3) / 1e12
    peak = peaks['tflops_sustained']
    # K1 (users) algorithmic bytes, SURVEY 8(d): nnz*8 + (R+1)*4 + D*d*4 (each DISTINCT weight row once) + R*d*4 (the
    # output: here the split operand, hi + lo fp16 = 4 bytes per component, + 8 bytes of scale and norm per row)
    distinct = int(np.unique(uf.indices).shape[0])
    k1_bytes = uf.nnz * 8 + (n_users + 1) * 4 + distinct * d * 4 + n_users * (2 * d_pad * 2 + 8)
    k1_survey_bytes = uf.nnz * 8 + (n_users + 1) * 4 + distinct * d * 4 + n_users * d * 4
    # the k1_users phase also holds project_biases (one more pass over the CSR arrays): charge the phase, report both
    k1_gbs = k1_survey_bytes / (k1u_ms * 1e-3) / 1e9

    cores = os.cpu_count() or 1
    cpu_value, cpu_desc, cpu_s, cpu_top = cpu_oracle_leg(uf_all, itf, wu, wi, bu, bi, k, args.cpu_budget, cores,
                                                         cosine=cosine)
    # parity at the full item count: the reference-semantics ranking (oracle, CPU) of the first users of this rank's
    # slice AND of the rows the certificate rejected in the last step, against the GPU top-k of the same users; only
    # sub-tolerance near-ties may order differently (fp32 rounding of the two GEMMs)
    t0 = time.perf_counter()
    rows = np.concatenate([np.arange(u_lo, u_lo + n_check), fallback_ids]).astype(np.int64)
    emulating = world == 1 and n_shards > 1
    exp, _, _ = oracle_topk_rows(uf_all, itf_local if emulating else itf, wu, wi, bu, bi, rows, k, cosine=cosine)
    exp = exp + (lo if emulating else 0)
    got = np.concatenate([top_items_check, fallback_items]) if len(fallback_ids) else top_items_check
    agree = float((exp == got).mean()) if len(rows) else None
    same_sets = float(np.mean([set(exp[i]) == set(got[i]) for i in range(len(rows))])) if len(rows) else None
    fb_agree = float((exp[n_check:] == got[n_check:]).mean()) if len(fallback_ids) else None
    # the double-argsort oracle of the cpu_baseline leg ranks the same first users: its top-k must equal the fast oracle's
    n_dbl = min(cpu_top.shape[0], n_check)
    oracle_self = bool(np.array_equal(cpu_top[:n_dbl], exp[:n_dbl])) if (n_dbl and u_lo == 0 and not emulating) else None
    log('[bench] parity check on %d users in %.1fs' % (len(rows), time.perf_counter() - t0))

    def phase_table(col):
        return {name: round(float(col[j]), 4) for j, name in enumerate(PHASES)}

    rest_ms = ms_step - fused_ms
    result = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
        'dtype': ('f32 (1 fp16 tcgen05 filter pass with a certified bound + re-scoring of the survivors from the 22-bit '
                  'split operands, fp32 accumulate)'
                  if use_filter else 'f32 (3 x fp16 split-product tcgen05 passes, fp32 accumulate)'),
        'data': 'synthetic',
        'config': workload_config(args),
        'details': {'parallelism': ('item axis sharded x%d%s: 1 NCCL all-to-all of the per-shard top-k per item group, '
                                    'each rank merges its user slice'
                                    % (item_shards, '' if n_groups == 1 else ' x %d user groups' % n_groups))
                    if world > 1 else 'single GPU',
                    'n_splits': n_splits, 'topk_path': 'filter+rescore' if use_filter else 'exact3',
                    'fallback_rows_last_step': fallback_rows, 'scores': args.scores,
                    'fallback_overflow_whole_batch_exact': bool(last_overflow)},
        'clocks': clocks,
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                'ms_per_step': e2e_ms_step, 'api': 'TensorRec.predict_rank(user_features, item_features, k) on pinned '
                'host CSR' + ('; every rank reads back its user slice' if world > 1 else ''),
                'matches_value_arm': same},
        'gpu_launches': int(gpu_launches),
        'roofline': {'kernel': ('score_filter_kernel (trk_score_filter_f16)' if use_filter
                                else 'score_tc_kernel<topk> (trk_score_topk_f16x3)'), 'bound': 'tensor',
                     'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s', 'frac': achieved / peak,
                     'traffic': ncu_traffic('score_filter_kernel@%dx%dx%d' % (n_users, n_local, d)) if use_filter
                     else ncu_traffic('score_tc_kernel@%dx%dx%d' % (n_users, n_local, d)),
                     'peak_source': peaks['source'] + ' bf16_tflops_sustained', 'ms_per_launch': fused_ms,
                     'issued_tflops': (1 if use_filter else 3) * achieved,
                     'issued_frac': (1 if use_filter else 3) * achieved / peak, 'share_of_step': fused_ms / ms_step},
        'roofline_k1': {'kernel': 'csr_gather_reduce_kernel (users) + csr_project_biases_kernel', 'bound': 'hbm',
                        'achieved': k1_gbs, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': k1_gbs / peaks['hbm_gbs'],
                        'ms_per_launch': k1u_ms, 'algorithmic_bytes': int(k1_survey_bytes),
                        'bytes_with_scale_and_norm': int(k1_bytes),
                        'traffic': ncu_traffic('csr_gather_reduce_kernel@%dx%d' % (n_users, d))},
        'phases_ms': {'rank0': phase_table(phase_ms), 'max_over_ranks': phase_table(all_phase.max(axis=0)),
                      'mean_over_ranks': phase_table(all_phase.mean(axis=0)),
                      'unsharded_share_of_step': rest_ms / ms_step if world > 1 or n_shards > 1 else None},
        'cpu_baseline': {'value': cpu_value, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': cpu_desc,
                         'seconds': cpu_s},
        'parity': {'users_checked': int(n_check), 'fallback_rows_checked': int(len(fallback_ids)),
                   'items': int(n_items), 'rank_positions_equal': agree, 'topk_sets_equal': same_sets,
                   'fallback_rank_positions_equal': fb_agree, 'double_argsort_oracle_agrees': oracle_self,
                   'against': 'oracle (numpy restatement of the reference: fp32 GEMM + bias adds + rank<=k in '
                              'tf.nn.top_k order)'},
    }
    if world == 1 and n_shards > 1:
        result['emulated_shard'] = '1 of %d (development aid: one shard timed alone, no exchange)' % n_shards
    if world == 1 and n_shards == 1 and not args.no_extra:
        del model, uf_host, itf_host, _keep_u, _keep_i, wu_d, wi_d
        torch.cuda.empty_cache()
        result['extra'] = run_extras(args)
    print(json.dumps(result), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_extras(args):
    """Secondary workloads measured in the same default run (N = 1) so that they are driver-run too: each entry is the
    JSON object the corresponding --workload prints."""
    import copy
    extras = {}
    for name, fn, over in (('dense', run_dense, {'users': 65536, 'items': 100000, 'd': 64}),
                           ('ranks', run_full_ranks, {'users': 8192, 'items': 131072, 'd': 128}),
                           ('train', run_train, {'users': 1000000, 'items': 1000000, 'd': 128})):
        a = copy.copy(args)
        for key, val in over.items():
            setattr(a, key, val)
        try:
            extras[name] = fn(a, emit=False)
        except Exception as exc:      # a secondary line must not take the headline down
            extras[name] = {'error': repr(exc)}
    return extras


# ----------------------------------------------------------------------------------------------------- reference arm
def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    uf, itf, wu, wi, bu, bi = make_problem(args)
    cores = os.cpu_count() or 1
    per_step_budget = max(2.0, min(args.cpu_budget, 90.0 / max(1, args.steps + args.warmup)))
    cosine = args.scores == 'c3'
    for _ in range(args.warmup):
        cpu_oracle_leg(uf, itf, wu, wi, bu, bi, args.k, per_step_budget, cores, cosine=cosine)
    values, secs, desc = [], 0.0, ''
    for _ in range(args.steps):
        v, desc, s, _ = cpu_oracle_leg(uf, itf, wu, wi, bu, bi, args.k, per_step_budget, cores, cosine=cosine)
        values.append(v)
        secs += s
    value = float(np.mean(values))
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': secs / args.steps * 1e3, 'higher_is_better': True, 'scaling': 'strong',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                         'sample': desc + ' -- numpy/scipy restatement of the reference TF-CPU semantics (TensorFlow is '
                         'not installable here); each step is a bounded user sample of the workload, ms_per_step is the '
                         'time of that sample'},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }), flush=True)


def run_dense(args, emit=True):
    """Secondary measurement (BASELINE configs[1], 1M users x 100K items d=64 predict(); the 400 GB result exceeds HBM, so
    the API streams user blocks -- TensorRec.predict_batches).  Two numbers:
      value: the dense tensor-core kernel alone on a resident block (bound: HBM write, U*I*4 bytes);
      e2e:   TensorRec.predict_batches over `--users` users with HOST inputs, every block copied to page-locked host
             memory inside the timed region (bound: the device->host link)."""
    import torch
    import tensorrec_b200
    from tensorrec_b200 import kernels
    kernels.require_cuda()
    torch.cuda.set_device(0)
    dev = torch.device('cuda', 0)
    uf, itf, wu, wi, bu, bi = make_problem(args)
    d_pad = kernels.d_pad_for(args.d)
    n_res = min(args.users, 65536)                      # resident block of the kernel-only number
    ucsr = kernels.DeviceCSR.from_scipy(uf[:n_res], device=dev)
    icsr = kernels.DeviceCSR.from_scipy(itf, device=dev)
    wu_d, wi_d = torch.from_numpy(wu).to(dev), torch.from_numpy(wi).to(dev)
    bu_d, bi_d = torch.from_numpy(bu).to(dev), torch.from_numpy(bi).to(dev)
    out = torch.empty((n_res, args.items), dtype=torch.float32, device=dev)
    ev = []

    def step():
        _, us, usc = kernels.gather_reduce(ucsr, wu_d, want_f32=False, split_d_pad=d_pad)
        _, its, isc = kernels.gather_reduce(icsr, wi_d, want_f32=False, split_d_pad=d_pad)
        ub, ib = kernels.project_biases(ucsr, bu_d), kernels.project_biases(icsr, bi_d)
        meta = kernels.pack_item_meta(isc, ib, args.items)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        kernels.score_dense_tc(us, usc, ub, its, meta, n_res, args.items, d_pad, out=out)
        b.record()
        ev.append((a, b))

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    del ev[:]
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(args.steps):
        step()
    s1.record()
    torch.cuda.synchronize()
    ms = s0.elapsed_time(s1) / args.steps
    kms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    peaks = measured_peaks()
    gbs = n_res * float(args.items) * 4 / (kms * 1e-3) / 1e9
    del out, ucsr, icsr
    torch.cuda.empty_cache()

    # e2e through the API: host CSR in, every score block out to page-locked host memory
    model = tensorrec_b200.TensorRec(n_components=args.d)
    model.set_weights({'linear_weights_user_0': wu, 'linear_weights_item': wi, 'feature_biases_user': bu[:, None],
                       'feature_biases_item': bi[:, None]})

    def sweep():
        n_rows, checksum = 0, 0.0
        for u0, u1, block in model.predict_batches(uf, itf, user_batch_size=args.user_batch):
            n_rows += u1 - u0
            checksum += float(block[0, 0])           # touch the page-locked result
        assert n_rows == args.users
        return checksum

    sweep()                                           # warm-up: also page-locks the two staging buffers
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sweep()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    pairs = args.users * float(args.items)
    result = {'metric': 'predict_pairs_per_s', 'value': n_res * float(args.items) / (ms * 1e-3),
              'unit': UNIT, 'n_gpus': 1, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms,
              'config': {'workload': 'predict() dense fp32 scores, %d users x %d items, d=%d (BASELINE configs[1] shape; '
                                     'value = one resident block of %d users, e2e = all users streamed through '
                                     'TensorRec.predict_batches)' % (args.users, args.items, args.d, n_res)},
              'roofline': {'kernel': 'score_tc_kernel<dense>', 'bound': 'hbm', 'achieved': gbs,
                           'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': gbs / peaks['hbm_gbs'],
                           'ms_per_launch': kms},
              'e2e': {'value': pairs / (e2e_ms * 1e-3), 'unit': UNIT, 'ms_per_step': e2e_ms,
                      'h2d_bytes_per_step': int(4 * (uf.nnz * 2 + uf.shape[0] + 1 + itf.nnz * 2 + itf.shape[0] + 1)),
                      'd2h_bytes_per_step': int(pairs * 4), 'd2h_gbs': pairs * 4 / (e2e_ms * 1e-3) / 1e9,
                      'api': 'TensorRec.predict_batches(user_features, item_features): user blocks, double-buffered '
                             'page-locked device->host copies overlapped with the next block\'s kernels',
                      'bound': 'device->host link (PCIe Gen5 x16: 64 GB/s nominal)'}}
    del model
    torch.cuda.empty_cache()
    if emit:
        print(json.dumps(result), flush=True)
    return result


def run_full_ranks(args, emit=True):
    """Secondary measurement: predict_rank() in the reference's full mode -- dense scores, then the exact int32 rank of
    every (user, item) pair (rank_predictions, tensorrec/recommendation_graphs.py:73-82) -- at a shape whose [U, I]
    matrices fit HBM.  Bound: HBM (the score matrix is written once, read by the chunk sort, the sorted keys are
    written and re-read by log2(#chunks) merge passes, the ranks are written once)."""
    import torch
    from tensorrec_b200 import kernels
    kernels.require_cuda()
    torch.cuda.set_device(0)
    dev = torch.device('cuda', 0)
    uf, itf, wu, wi, bu, bi = make_problem(args)
    d_pad = kernels.d_pad_for(args.d)
    ucsr, icsr = kernels.DeviceCSR.from_scipy(uf, device=dev), kernels.DeviceCSR.from_scipy(itf, device=dev)
    wu_d, wi_d = torch.from_numpy(wu).to(dev), torch.from_numpy(wi).to(dev)
    bu_d, bi_d = torch.from_numpy(bu).to(dev), torch.from_numpy(bi).to(dev)
    out = torch.empty((args.users, args.items), dtype=torch.float32, device=dev)
    ev = []

    def step():
        _, us, usc = kernels.gather_reduce(ucsr, wu_d, want_f32=False, split_d_pad=d_pad)
        _, its, isc = kernels.gather_reduce(icsr, wi_d, want_f32=False, split_d_pad=d_pad)
        ub, ib = kernels.project_biases(ucsr, bu_d), kernels.project_biases(icsr, bi_d)
        meta = kernels.pack_item_meta(isc, ib, args.items)
        kernels.score_dense_tc(us, usc, ub, its, meta, args.users, args.items, d_pad, out=out)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ranks = kernels.rank_full(out)
        b.record()
        ev.append((a, b))
        return ranks

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    del ev[:]
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(args.steps):
        ranks = step()
    s1.record()
    torch.cuda.synchronize()
    ms = s0.elapsed_time(s1) / args.steps
    kms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    # spot check against the closed form on a few rows: rank = 1 + #greater + #equal with a lower index
    rows = np.linspace(0, args.users - 1, 4).astype(np.int64)
    sc, rk = out[rows].cpu().numpy(), ranks[rows].cpu().numpy()
    for r in range(len(rows)):
        order = np.lexsort((np.arange(args.items), -sc[r].astype(np.float64)))
        expect = np.empty(args.items, dtype=np.int64)
        expect[order] = np.arange(1, args.items + 1)
        assert np.array_equal(expect, rk[r]), 'rank_full disagrees with the closed form on row %d' % rows[r]
    peaks = measured_peaks()
    pairs = args.users * float(args.items)
    alg_bytes = pairs * (4 + 4)        # scores read once, ranks written once
    gbs = alg_bytes / (kms * 1e-3) / 1e9
    result = {'metric': 'predict_rank_full_ranks_per_s', 'value': pairs / (ms * 1e-3), 'unit': 'ranks/s',
              'n_gpus': 1, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms,
              'config': {'workload': 'predict_rank() full int32 ranks, %d users x %d items, d=%d (reference '
                                     'semantics: every pair ranked)' % (args.users, args.items, args.d)},
              'roofline': {'kernel': 'trk_rank_full', 'bound': 'hbm', 'achieved': gbs, 'peak': peaks['hbm_gbs'],
                           'unit': 'GB/s', 'frac': gbs / peaks['hbm_gbs'], 'ms_per_launch': kms,
                           'ranks_per_s_kernel': pairs / (kms * 1e-3)}}
    del out, ranks
    torch.cuda.empty_cache()
    if emit:
        print(json.dumps(result), flush=True)
    return result


def run_train(args, emit=True):
    """Secondary measurement (BASELINE configs[3]: WMRBLossGraph sampled-rank training step, d=128, bf16): one Adam step of
    LinearRepr x DotProduct x WMRB over `--users` users x `--items` items on the kernels of tensorrec_b200/train_kernels.py --
    K1 forward, device sampler, fused serial-prediction + WMRB forward / backward, K1^T backward, fused L2 + Adam.
    metric: (user, item) pairs scored AND back-propagated per second = users x (n_sampled + interactions per user) / step.
    Bound: HBM (one item-row gather per pair + the sparse products + the optimiser's pass over every weight)."""
    import torch
    import tensorrec_b200
    from tensorrec_b200 import kernels, train_kernels
    from tensorrec_b200.input_utils import SparseInput
    kernels.require_cuda()
    torch.cuda.set_device(0)
    dev = torch.device('cuda', 0)
    uf, itf, wu, wi, bu, bi = make_problem(args)
    n_users, n_items, d, n_s = args.users, args.items, args.d, args.n_sampled
    rng = np.random.default_rng(5)
    per_user = 4                                            # positive interactions per user, + 1 negative in 4 users
    rows = np.repeat(np.arange(n_users, dtype=np.int64), per_user)
    cols = rng.integers(0, n_items, rows.shape[0])
    vals = np.ones(rows.shape[0], dtype=np.float32)
    neg_rows = np.arange(0, n_users, 4, dtype=np.int64)
    interactions = sp.csr_matrix((np.concatenate([vals, -np.ones(neg_rows.shape[0], np.float32)]),
                                  (np.concatenate([rows, neg_rows]),
                                   np.concatenate([cols, rng.integers(0, n_items, neg_rows.shape[0])]))),
                                 shape=(n_users, n_items))
    bf16 = args.train_dtype == 'bf16'

    def new_model(users=None):
        model = tensorrec_b200.TensorRec(n_components=d, loss_graph=tensorrec_b200.loss_graphs.WMRBLossGraph())
        model.set_weights({'linear_weights_user_0': wu, 'linear_weights_item': wi, 'feature_biases_user': bu[:, None],
                           'feature_biases_item': bi[:, None]})
        return model, train_kernels.WmrbStep(model, dev, seed=0, bf16=bf16)

    model, stepper = new_model()
    int_in, uf_in, if_in = SparseInput(interactions), SparseInput(uf), SparseInput(itf)
    n_pos = int_in.n_positive
    lr, l2 = 0.01, n_pos * 1e-5

    def step():
        return stepper.step(int_in, uf_in, if_in, n_s, lr, l2)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    stepper.marks = []
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(args.steps):
        loss, _ = step()
    s1.record()
    torch.cuda.synchronize()
    ms = s0.elapsed_time(s1) / args.steps
    names = ['representations', 'sampler', 'wmrb_step', 'weight_gradients', 'adam']
    phase = {n: 0.0 for n in names}
    marks = stepper.marks
    per = len(names) + 1
    for s in range(args.steps):
        for j, n in enumerate(names):
            phase[n] += marks[s * per + j][1].elapsed_time(marks[s * per + j + 1][1]) / args.steps
    stepper.marks = None
    loss_sum = float(loss.sum())
    pairs = float(n_users) * n_s + interactions.nnz
    esz = 2 if bf16 else 4
    n_w = (uf.shape[1] + itf.shape[1]) * (d + 1)
    k1 = lambda m, r: m.nnz * 8 + (r + 1) * 4 + m.shape[1] * d * 4 + r * d * 4        # noqa: E731  (SURVEY 8d per side)
    alg_bytes = (k1(uf, n_users) + k1(itf, n_items)                        # representations
                 + ((n_users + n_items) * d * (4 + 2) if bf16 else 0)      # rounding pass
                 + n_users * n_s * 4                                       # sampler
                 + pairs * d * esz + n_users * d * (esz + 4) + n_users * n_s * 4 + interactions.nnz * 24
                 + 2 * n_items * d * 4                                     # wmrb: item rows, user rows, dU, zero + write dI
                 + (uf.nnz + itf.nnz) * (8 + d * 4) + n_w * 4              # K1^T: gathered gradient rows, weight gradients
                 + n_w * 4 * 7)                                            # Adam: read w, g, m, v; write w, m, v
    peaks = measured_peaks()

    # CPU oracle beside it: the same step (forward + backward) on a bounded user sample, item side complete
    from oracle import loss_ops
    n_cpu = min(n_users, args.train_cpu_users)
    sub_int, sub_uf = interactions[:n_cpu], uf[:n_cpu]
    m2, st2 = new_model()
    st2.t = stepper.t - 1                                   # same sampler step as the last timed step
    samples = train_kernels.sample_items_device(n_items, n_cpu, n_s, False, 0, st2.t, dev)
    loss2, _ = st2.step(SparseInput(sub_int), SparseInput(sub_uf), if_in, n_s, lr, l2, samples=samples)
    t0 = time.perf_counter()
    ref = loss_ops.wmrb_step_reference(sub_uf, itf, sub_int, wu, wi, bu, bi, samples.cpu().numpy(),
                                       round_repr=loss_ops.round_to_bfloat16 if bf16 else None)
    cpu_s = time.perf_counter() - t0
    cpu_pairs = float(n_cpu) * n_s + sub_int.nnz
    g_gpu = st2.last['grads']['linear_weights_item'].cpu().numpy()
    scale = max(1.0, float(np.abs(ref['d_w_item']).max()))
    parity = {'users_checked': int(n_cpu),
              'loss_sum_rel_err': abs(float(loss2.sum()) - float(ref['loss'].sum())) / max(1e-30, abs(float(ref['loss'].sum()))),
              'item_weight_grad_max_abs_err_over_scale': float(np.abs(g_gpu - ref['d_w_item']).max() / scale),
              'against': 'oracle/loss_ops.wmrb_step_reference (numpy forward + analytic backward, same samples)'}
    result = {'metric': 'wmrb_train_pairs_per_s', 'value': pairs / (ms * 1e-3), 'unit': 'pairs/s', 'n_gpus': 1,
              'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms, 'dtype': args.train_dtype + ' representations, '
              'f32 weights / accumulation / Adam',
              'config': {'workload': 'WMRB sampled-rank training step, %d users x %d items, d=%d, n_sampled_items=%d, '
                                     '%d interactions (BASELINE configs[3] shape: the slice of 10M x 1M run per step)'
                                     % (n_users, n_items, d, n_s, interactions.nnz),
                         'loss_sum_last_step': loss_sum},
              'phases_ms': {k: round(v, 4) for k, v in phase.items()},
              'roofline': {'kernel': 'whole step (K1 x2, sampler, wmrb_step_kernel, K1^T x2, adam_step_kernel x4)',
                           'bound': 'hbm', 'achieved': alg_bytes / (ms * 1e-3) / 1e9, 'peak': peaks['hbm_gbs'],
                           'unit': 'GB/s', 'frac': alg_bytes / (ms * 1e-3) / 1e9 / peaks['hbm_gbs'],
                           'algorithmic_bytes': int(alg_bytes),
                           'wmrb_kernel_gather_gbs': pairs * d * esz / (phase['wmrb_step'] * 1e-3) / 1e9},
              'cpu_baseline': {'value': cpu_pairs / cpu_s, 'unit': 'pairs/s', 'cores': os.cpu_count() or 1, 'kind': 'port',
                               'sample': '%d of %d users (all items): numpy forward + backward of the same step, %.1f s'
                                         % (n_cpu, n_users, cpu_s)},
              'parity': parity}
    del model, stepper, m2, st2
    torch.cuda.empty_cache()
    if emit:
        print(json.dumps(result), flush=True)
    return result


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--users', type=int, default=1000000)
    ap.add_argument('--items', type=int, default=1000000)
    ap.add_argument('--d', type=int, default=128)
    ap.add_argument('--k', type=int, default=10)
    ap.add_argument('--workload', default='topk', choices=['topk', 'dense', 'ranks', 'train'])
    ap.add_argument('--topk-path', default='filter', choices=['filter', 'exact'])
    ap.add_argument('--scores', default='iid', choices=['iid', 'ties', 'c3', 'const'],
                    help='score distribution of the top-k workload: continuous (headline), integer-valued (massive ties), '
                         'or MovieLens-shaped features with cosine prediction')
    ap.add_argument('--cpu-budget', type=float, default=15.0, help='seconds of CPU work for the cpu_baseline sample')
    ap.add_argument('--parity-users', type=int, default=4096, help='users checked against the oracle at full size')
    ap.add_argument('--parity-fallback-rows', type=int, default=1024,
                    help='rows rejected by the certificate (last step) that are also checked against the oracle')
    ap.add_argument('--user-batch', type=int, default=None, help='user_batch_size of the API (e2e) arm')
    ap.add_argument('--emulate-shards', type=int, default=1,
                    help='development aid (1 GPU): time the work of ONE item shard out of this many, no exchange')
    ap.add_argument('--no-clocks', action='store_true', help='do not sample nvidia-smi during the timed region')
    ap.add_argument('--item-shards', type=int, default=None,
                    help='ranks per item group (default: all ranks = the item axis sharded over every GPU); a divisor of the '
                         'rank count gives the grid form: item_shards x (ranks / item_shards) user groups')
    ap.add_argument('--no-extra', action='store_true', help='skip the secondary workloads of the default run')
    ap.add_argument('--n-sampled', type=int, default=64, help='--workload train: n_sampled_items')
    ap.add_argument('--train-dtype', default='bf16', choices=['bf16', 'f32'], help='--workload train: representations')
    ap.add_argument('--train-cpu-users', type=int, default=20000, help='--workload train: users of the CPU oracle sample')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write the top-k of the last step (a seeded sample of its user rows) '
                         'as DIR/<name>.npy, for output-for-output comparison of two builds')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    if args.dump_outputs and (args.workload != 'topk' or args.impl != 'b200'):
        ap.error('--dump-outputs writes the top-k of --workload topk --impl b200')
    if args.workload == 'dense':
        run_dense(args)
    elif args.workload == 'ranks':
        run_full_ranks(args)
    elif args.workload == 'train':
        run_train(args)
    elif args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
