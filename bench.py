#!/usr/bin/env python
"""bench.py -- the OCR forward hot path on B200, one JSON line per run (rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

Workloads (BASELINE.json `configs`; the default is the one the headline metric is quoted on):

  omni      config 2: OmniParser Swin-B text spotting, 1024x1024 synthetic pages, batch 16 per GPU, N = 64 text
            instances per page pinned (pt_seq_length 128, 32 polygon + 25 recognition tokens each; SURVEY.md 8d)
  mgpstr    config 3: MGP-STR ViT-Base, 512 32x128 crops per GPU per step, bf16 (single-pass; --nsplit 3 = parity mode)
  table     config 5: OmniParser at 1920x1920, 8 pages per GPU, one 512-token point-decoder sequence per page
            (the table head itself is not released, SURVEY F4: the generic pt decoder is what is timed)
  platypus  config 4: Platypus ships no code (SURVEY F3): the OmniParser encoder + decoder at 896x896, 8 pages per GPU
            (32 over 4 GPUs), throughput only, NO parity oracle

A step = one batch through the whole path.  `value`: inputs resident in HBM; `e2e`: the same metric through the adapter
with pinned HOST inputs, H2D and D2H inside the timed region.  With N > 1 GPUs every step ends with ONE all-gather of the
decoded sequences (alm_gather_sequences, the library's own NCCL communicator; the contexts' host threads take turns in
batch order, dist.CollectiveOrder) inside the timed region, and the weights reach the ranks by ONE NCCL broadcast of the
converted planes (alm_broadcast_weights).

`--impl reference` times the reference algorithm (the CPU oracle port: fp32, no KV cache, memory repeated per instance,
transformer.py:74-100) on the host cores on the SAME workload: one page (omni / table / platypus) or 32 crops (mgpstr)
per step.  A full config-2 page costs the no-cache loops ~1.5-3 minutes of CPU, so the arm runs at most 3 timed steps
(and reports the steps it actually ran); the oracle is the checker everywhere else, this leg only times it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

REC_LEN = 25
N_INST = 64
ENC_GFLOP = {1024: 682.1, 896: 493.8, 1920: 2335.7}   # SURVEY.md 8d: algorithmic 2*M*N*K of the Swin-B encoder per image
MGP_GFLOP_PER_CROP = 49.75

WORKLOADS = {
    'omni': dict(kind='omni', page=1024, batch=16, n_inst=N_INST, pt_len=2 * N_INST, points_only=False, inflight=5,
                 workspace_mb=20480, gemm=(65536, 2048, 512), gemm_name='Swin stage-2 fc1', gemm_ncu='r02f_prof_gemm_fc1_metrics.csv',
                 text=f'OmniParser Swin-B text spotting, 1024x1024 synthetic pages, batch 16 per GPU, N={N_INST} '
                      f'instances/page pinned (pt 128 + poly 32 + rec {REC_LEN} tokens)'),
    'platypus': dict(kind='omni', page=896, batch=8, n_inst=N_INST, pt_len=2 * N_INST, points_only=False, inflight=5,
                     workspace_mb=16384, gemm=(25088, 2048, 512), gemm_name='Swin stage-2 fc1',
                     text=f'Platypus stand-in (no reference code, SURVEY F3): OmniParser encoder + decoder, 896x896 synthetic '
                          f'pages, batch 8 per GPU, N={N_INST} instances/page; throughput only, no parity oracle'),
    'table': dict(kind='omni', page=1920, batch=8, n_inst=0, pt_len=512, points_only=True, inflight=2,
                  workspace_mb=40960, gemm=(115200, 2048, 512), gemm_name='Swin stage-2 fc1',
                  text='OmniParser 1920x1920 synthetic pages, batch 8 per GPU, one 512-token point-decoder sequence per page '
                       '(table head not released, SURVEY F4: generic pt decoder)'),
    'mgpstr': dict(kind='mgp', batch=512, inflight=2, gemm=(131584, 3072, 768), gemm_name='ViT fc1', gemm_ncu='r02f_prof_gemm_vit_fc1_metrics.csv',
                   text='MGP-STR ViT-Base, 512 synthetic 32x128 crops per GPU per step, ids + probabilities of the three heads'),
}


# ---------------------------------------------------------------------------------------------------- utilities
def peaks():
    p = os.path.join(REPO, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d['bf16_tflops'], d['bf16_tflops_sustained'], d['hbm_gbs'], 'measured (MEASURED_PEAKS.json)'
    return 1590.0, 1400.0, 6650.0, 'fallback (B200_PROFILING.md)'


def ncu_traffic_bytes(name):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant GEMM launch from a committed ncu capture."""
    p = os.path.join(REPO, 'profiles', name)
    try:
        tot = 0.0
        for line in open(p):
            k, v, u = line.rstrip('\n').rsplit(',', 2)
            if k in ('dram__bytes_read.sum', 'dram__bytes_write.sum'):
                tot += float(v) * {'Mbyte': 1e6, 'Gbyte': 1e9, 'Kbyte': 1e3, 'byte': 1.0}[u]
        return tot or None
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader,nounits', '-lms', '100',
                                          '-i', str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = max([int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()] or [0])
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i] == 'Active' for r in self.rows)]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx or None, 'reasons': reasons,
                'samples': len(sm)}


def effective_cpus():
    """Host threads the process may really use: min(affinity mask, cgroup CPU quota), capped at 64."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    quota = None
    try:
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            quota = max(1, int(float(q) / float(per)))
    except Exception:
        try:
            q = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())
            per = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if q > 0:
                quota = max(1, q // per)
        except Exception:
            pass
    if quota:
        n = min(n, quota)
    return max(1, min(n, 64)), {'affinity': len(os.sched_getaffinity(0)), 'cgroup_quota': quota, 'cpu_count': os.cpu_count()}


def page_tensor(side, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    return torch.randn(1, 3, side, side, generator=g)


def workload_config(name, world, nsplit):
    """The `config` object: identical for the GPU arm and the reference arm of a workload."""
    w = WORKLOADS[name]
    return {'workload': w['text'], 'global_batch': world * w['batch'], 'parallelism': f'dp{world}',
            'inputs': 'synthetic, seeded per page / crop (page p of the job: seed 1000 + p)',
            'weights': 'synthetic seed 0 (advancedliteratemachinery_b200/synthetic.py)' +
                       (', pt_eos suppressed so that every page decodes the pinned length' if w['kind'] == 'omni' else ''),
            'l2': 'no explicit flush: per-step inputs and activations exceed the 126 MB L2'}


# ---------------------------------------------------------------------------------------------------- CPU reference
def _cpu_child(name, n_inst, pt_len):
    """Subprocess body: ONE unit of the reference algorithm on the host cores (oracle port); prints seconds."""
    import torch
    from advancedliteratemachinery_b200 import synthetic as W
    torch.set_grad_enabled(False)
    threads, _ = effective_cpus()
    torch.set_num_threads(threads)
    w = WORKLOADS[name]
    if w['kind'] == 'mgp':
        from oracle import mgpstr_ref as M
        sd = W.mgpstr_state_dict(seed=0)
        g = torch.Generator().manual_seed(1000)
        img = torch.rand(n_inst, 3, 32, 128, generator=g)   # n_inst = crops in this sample
        M.forward(img[:2], sd)                              # thread pool / allocator warm-up
        t = time.time()
        M.forward(img, sd)
        print(json.dumps({'sec': time.time() - t, 'threads': torch.get_num_threads()}), flush=True)
        return
    from oracle import omniparser_ref as O
    sd = W.omniparser_state_dict(seed=0, pt_eos_bias=-30.0)
    img = page_tensor(w['page'], 1000)
    mask = torch.zeros(1, w['page'], w['page'], dtype=torch.bool)
    t = time.time()
    if w['points_only']:
        mem, pos, kpm, _ = O.encode(img, mask, sd)
        t_enc = time.time() - t
        seq = O.default_prompts(True)[0]
        t1 = time.time()
        for _ in range(pt_len):  # decode_pt_seq, no cache (transformer.py:102-141): whole prefix + memory K/V per token
            lg = O.decode_logits(seq, mem[0], kpm[0], pos[0], sd, 'pt')[:, -1, :]
            seq = torch.cat([seq, lg[:, :1000].argmax(-1, keepdim=True)], 1)
        print(json.dumps({'sec': time.time() - t, 'enc_sec': t_enc, 'step_sec': (time.time() - t1) / pt_len,
                          'threads': torch.get_num_threads()}), flush=True)
        return
    O.forward(img, mask, sd, pt_seq_length=pt_len, rec_length=REC_LEN)
    print(json.dumps({'sec': time.time() - t, 'threads': torch.get_num_threads()}), flush=True)


def cpu_sample(name, n_inst, pt_len, timeout):
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), '--cpu-child', name, str(n_inst), str(pt_len)],
                           capture_output=True, text=True, timeout=timeout, cwd=REPO)
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:
        return {'error': type(e).__name__}


def cpu_baseline_bounded(name):
    """The bounded (10-30 s) CPU sample printed next to the GPU number: a REDUCED unit of the workload, stated as such.
    The like-for-like CPU number is the `--impl reference` arm."""
    threads, info = effective_cpus()
    w = WORKLOADS[name]
    if w['kind'] == 'mgp':
        d = cpu_sample(name, 32, 0, 200)
        val = 32 / d['sec'] if 'sec' in d else None
        return {'value': val, 'unit': 'images/s', 'cores': d.get('threads', threads), 'kind': 'port',
                'sample': f'32 crops, one forward of the reference algorithm (fp32): {d.get("sec", float("nan")):.1f} s', 'host': info}
    if w['points_only']:
        d = cpu_sample(name, 0, 4, 300)
        val = None
        if 'sec' in d:
            val = 1.0 / (d['enc_sec'] + d['step_sec'] * w['pt_len'])
        return {'value': val, 'unit': 'images/s', 'cores': d.get('threads', threads), 'kind': 'port',
                'sample': f'1 page {w["page"]}x{w["page"]}: encoder {d.get("enc_sec", float("nan")):.1f} s + 4 no-cache point-decoder '
                          f'tokens at {d.get("step_sec", float("nan")):.2f} s each; value = 1 / (encoder + {w["pt_len"]} x token time), i.e. '
                          'EXTRAPOLATED from the first 4 tokens (later tokens are slower: the prefix grows)', 'host': info}
    d = cpu_sample(name, 8, 16, 400)
    return {'value': (1.0 / d['sec']) if 'sec' in d else None, 'unit': 'images/s', 'cores': d.get('threads', threads), 'kind': 'port',
            'sample': f'1 page {w["page"]}x{w["page"]} at N=8 instances (pt 16 + poly 32 + rec {REC_LEN} tokens each; the GPU arm '
                      f'decodes N={w["n_inst"]}): {d.get("sec", float("nan")):.1f} s of the no-cache reference algorithm; the same-workload '
                      'number is the --impl reference arm', 'host': info}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    name = args.workload
    w = WORKLOADS[name]
    threads, info = effective_cpus()
    t0 = time.time()
    budget = args.ref_budget_s
    if w['kind'] == 'mgp':
        unit_n, n_inst, pt_len, unit_desc = 32, 32, 0, '32 crops per step (1/16 of a 512-crop batch)'
        max_steps = args.steps
    else:
        unit_n, n_inst, pt_len = 1, w['n_inst'], w['pt_len']
        unit_desc = (f'1 page per step (the reference is batch-1, engine/val.py:22): full workload, N={n_inst} instances, '
                     f'pt {pt_len} + poly 32 + rec {REC_LEN} tokens, no KV cache') if not w['points_only'] else \
                    f'1 page per step: encoder + {pt_len} no-cache point-decoder tokens'
        max_steps = min(args.steps, 3)
    # warm-up: one reduced unit (pays library loading, thread-pool start, allocator growth)
    warm = cpu_sample(name, 2 if w['kind'] != 'mgp' else 4, 4 if w['kind'] != 'mgp' else 0, 600)
    secs = []
    for _ in range(max_steps):
        if secs and (time.time() - t0) + secs[-1] > budget:
            break
        d = cpu_sample(name, n_inst, pt_len, 3600)
        if 'sec' not in d:
            break
        secs.append(d['sec'])
        threads = d.get('threads', threads)
    world = args.gpus
    if not secs:
        print(json.dumps({'impl': 'reference', 'unavailable': 'the CPU reference sample did not finish'}), flush=True)
        return
    med = sorted(secs)[len(secs) // 2]
    ips = unit_n / med
    cb = {'value': ips, 'unit': 'images/s', 'cores': threads, 'kind': 'port',
          'sample': f'{unit_desc}; {len(secs)} timed step(s) after 1 reduced warm-up unit ({warm.get("sec", float("nan")):.1f} s); '
                    f'seconds per step: {[round(s, 1) for s in secs]}; value = median', 'host': info}
    line = {
        'impl': 'reference', 'metric': 'doc_images_per_sec', 'value': ips, 'unit': 'images/s', 'n_gpus': world,
        'steps': len(secs), 'warmup': 1, 'requested_steps': args.steps, 'requested_warmup': args.warmup,
        'ms_per_step': med * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic', 'config': workload_config(name, world, args.nsplit), 'cpu_baseline': cb,
        'e2e': {'value': ips, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'note': 'CPU arm: rank 0 only, host cores only; it does not scale with --gpus (one process, one page at a time)',
        'wall_s': time.time() - t0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------- GPU arm
def mgp_decoded_chars(ids):
    """char-head tokens before '[s]' (id 1), position 0 dropped (demo.py:39-60): what `decoded-chars/s` counts."""
    c = ids[0][:, 1:]
    eos = (c == 1)
    first = (eos.float().cumsum(1) == 0).sum(1)   # tokens before the first [s] (all 26 when there is none)
    return int(first.sum())


def dump_outputs(out, w, outdir):
    """Write what one batch of the timed path returned to its caller as `outdir/<name>.npy`: token ids as float64 (exact),
    probabilities as float32.  Per-page sequences are padded with -1 to the workload's maximum length, so every run of a
    workload writes the same shapes and two builds can be compared array for array (well under 64 MB for every workload)."""
    import numpy as np
    B = out[0].shape[1] if w['kind'] == 'mgp' else len(out)
    if w['kind'] == 'mgp':
        ids, prob = out
        arrays = {'ids': ids.numpy().astype(np.float64), 'probs': prob.numpy().astype(np.float32)}
    elif w['points_only']:
        P = w['pt_len']
        n = np.zeros(B)
        tok, pr = np.full((B, P), -1.0), np.full((B, P), -1.0, dtype=np.float32)
        for b, (t, p) in enumerate(out):
            n[b] = t.numel()
            tok[b, :t.numel()], pr[b, :p.numel()] = t.numpy(), p.numpy()
        arrays = {'n_tokens': n, 'pt': tok, 'pt_probs': pr}
    else:
        maxi = w['pt_len'] // 2
        n = np.zeros(B)
        pt, poly, rec = np.full((B, maxi, 2), -1.0), np.full((B, maxi, 32), -1.0), np.full((B, maxi, REC_LEN), -1.0)
        prob = np.full((B, maxi, REC_LEN), -1.0, dtype=np.float32)
        for b, o in enumerate(out):
            if o is None:          # no point decoded on this page
                continue
            (p, q, r), (pr,) = o
            k = p.numel() // 2
            n[b] = k
            pt[b, :k], poly[b, :k] = p.numpy().reshape(k, 2), q.numpy().reshape(k, 32)
            rec[b, :k], prob[b, :k] = r.numpy()[0], pr.numpy()
        arrays = {'n_instances': n, 'pt': pt, 'poly': poly, 'rec': rec, 'rec_probs': prob}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    os.makedirs(outdir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(outdir, k + '.npy'), a)


def self_check_omni(out0):
    """Page 0 of rank 0 (page seed 1000) against the reference's own output (tests/golden/omni_config2_page0.npz,
    written by oracle/gen_golden.py config2 from the unmodified reference).  Sequences that leave the reference are
    counted; tests/test_gpu_omniparser.py judges every such flip against the reference top-1/top-2 gap."""
    import numpy as np
    p = os.path.join(REPO, 'tests', 'golden', 'omni_config2_page0.npz')
    if out0 is None or not os.path.exists(p):
        return {'checked': False}
    gold = np.load(p)
    (pt, poly, rec), _ = out0
    n = gold['pt'].size // 2
    same_pt = bool(np.array_equal(pt.numpy(), gold['pt']))
    bad_poly = int((poly.numpy().reshape(n, 32) != gold['poly'].reshape(n, 32)).any(1).sum()) if same_pt else None
    bad_rec = int((rec.numpy()[0] != gold['rec'][0]).any(1).sum()) if same_pt else None
    ok = same_pt and bad_poly + bad_rec <= 3
    return {'checked': True, 'against': 'reference output on page seed 1000 (tests/golden/omni_config2_page0.npz)',
            'pt_ids_equal': same_pt, 'poly_sequences_differing': bad_poly, 'rec_sequences_differing': bad_rec,
            'sequences': 2 * n + 1, 'ok': bool(ok)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='omni', choices=sorted(WORKLOADS))
    ap.add_argument('--nsplit', type=int, default=0, help='3 = fp32-class split operands (parity mode), 1 = single-pass bf16; '
                    'default: 3 for the OmniParser workloads, 1 for mgpstr (config 3 is stated in bf16)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--inflight', type=int, default=0, help='execution contexts in flight per GPU (one stream + host thread '
                    'each, ONE shared set of weights): the per-token decode loops are latency-bound, concurrent batches fill '
                    'their launch gaps.  0 = the workload default')
    ap.add_argument('--opt', action='append', default=[], metavar='NAME=VALUE', help='extra alm_set_option (A/B runs)')
    ap.add_argument('--ref-budget-s', type=float, default=330.0, help='reference arm: stop adding timed steps past this')
    ap.add_argument('--collectives', default='order', choices=['order', 'lane'], help='N > 1: who issues the per-batch gathers. '
                    'order = every compute thread gathers on its own context\'s communicator, taking turns in batch order '
                    '(dist.CollectiveOrder) [default]; lane = one host thread per rank on a dedicated context / communicator, '
                    'the compute threads do not wait (dist.CollectiveLane; measured: no gain at 2 GPUs, lower e2e)')
    ap.add_argument('--watchdog-s', type=float, default=600.0, help='a timed phase that takes longer dumps every host '
                    'thread\'s stack to stderr and exits non-zero (a hung collective must not burn the GPU box)')
    ap.add_argument('--dump-outputs', default=None, metavar='DIR', help='after the timed steps, write what the last timed '
                    'step returned (rank 0\'s batch) as DIR/<name>.npy, for output-for-output comparison of two builds')
    ap.add_argument('--cpu-child', nargs=3, default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of the GPU arm (--impl ours)')
    if args.cpu_child:
        return _cpu_child(args.cpu_child[0], int(args.cpu_child[1]), int(args.cpu_child[2]))
    if args.impl == 'reference':
        return run_reference(args)

    import faulthandler
    import numpy as np
    import torch
    import torch.distributed as dist
    from advancedliteratemachinery_b200 import MGPSTRB200, NestedTensor, OmniParserB200, OmniVocab, _lib
    from advancedliteratemachinery_b200.dist import CollectiveLane, CollectiveOrder, gather_sequences, init_comm, load_weights_broadcast
    from advancedliteratemachinery_b200 import synthetic as W  # synthetic checkpoint (data only)

    torch.set_grad_enabled(False)
    name = args.workload
    w = WORKLOADS[name]
    is_mgp = w['kind'] == 'mgp'
    nsplit = args.nsplit or (1 if is_mgp else 3)
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert world == args.gpus or world == 1, 'launch with torchrun --nproc-per-node N for --gpus N'
    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    # ---- contexts: ONE set of weights per GPU, C execution contexts over it
    C_ = args.inflight if args.inflight > 0 else w['inflight']
    C_ = max(1, min(C_, args.steps))
    streams = [torch.cuda.Stream() for _ in range(C_)]
    ctxs = []
    for j in range(C_):
        cx = _lib.Context(local, streams[j].cuda_stream)
        cx.set_option('nsplit', nsplit)
        if not is_mgp:
            cx.set_option('workspace_mb', w['workspace_mb'])
        for kv in args.opt:
            cx.set_option(kv.split('=')[0], int(kv.split('=')[1]))
        ctxs.append(cx)
    # weights: rank 0 builds the synthetic checkpoint; ONE NCCL broadcast of the converted planes (C ABI) to the others
    kind = _lib.MODEL_MGPSTR if is_mgp else _lib.MODEL_OMNI_SPOT
    sd = None
    if rank == 0:
        sd = W.mgpstr_state_dict(seed=0) if is_mgp else W.omniparser_state_dict(seed=0, pt_eos_bias=-30.0)
    t_w = time.time()
    gctx, gstream = None, None
    if world > 1:
        # two communicators per rank: context 0's for the weight broadcast, and one on a dedicated context + stream for the
        # per-batch gathers, which ONE host thread (the collective lane) issues in batch order
        if args.collectives == 'lane':
            init_comm(ctxs[0], device=dev)
            gstream = torch.cuda.Stream()
            gctx = _lib.Context(local, gstream.cuda_stream)
            init_comm(gctx, device=dev)
        else:
            for cx in ctxs:                  # one communicator per context, created in the same order on every rank
                init_comm(cx, device=dev)
        load_weights_broadcast(ctxs[0], kind, sd, src=0, device=dev)
    else:
        ctxs[0].load_state_dict(kind, sd)
    weights_s = time.time() - t_w
    del sd
    if is_mgp:
        models = [MGPSTRB200(None, ctx=ctxs[0])] + [None] * (C_ - 1)
        for j in range(1, C_):
            ctxs[j].share_weights(ctxs[0])
            models[j] = MGPSTRB200(None, ctx=ctxs[j])
        vocab = None
    else:
        vocab = OmniVocab(pt_seq_length=w['pt_len'], rec_length=REC_LEN)
        models = [OmniParserB200(None, vocab, ctx=ctxs[0])] + [None] * (C_ - 1)
        for j in range(1, C_):
            ctxs[j].share_weights(ctxs[0])
            models[j] = OmniParserB200(None, vocab, ctx=ctxs[j])
    ctx, model = ctxs[0], models[0]

    # ---- inputs: this rank's round-robin shard of the job's pages (page p -> rank p % world), seeded per page
    B = w['batch']
    pages = [rank + i * world for i in range(B)]
    if is_mgp:
        host_in = torch.cat([torch.rand(1, 3, 32, 128, generator=torch.Generator().manual_seed(1000 + p)) for p in pages])
    else:
        host_in = torch.cat([page_tensor(w['page'], 1000 + p) for p in pages])
    host_in = host_in.pin_memory()
    dev_in = host_in.cuda(non_blocking=False)
    h2d_bytes = host_in.numel() * 4

    def run_model(j, x):
        if is_mgp:
            return models[j].recognize(x)
        models[j].encode(x, None)
        return models[j].decode_points() if w['points_only'] else models[j].decode()

    lane = CollectiveLane(max_ahead=2 * C_) if world > 1 and args.collectives == 'lane' else None
    order = CollectiveOrder() if world > 1 and args.collectives == 'order' else None
    turn_results = {}

    def gather_now(out, gc):
        """ONE all-gather of the decoded sequences of a batch over context `gc`'s NCCL communicator."""
        if is_mgp:
            ids, prob = out
            buf = np.concatenate([ids.numpy().reshape(-1), prob.numpy().view(np.int32).reshape(-1)])
            return gc.gather(buf, world)
        if w['points_only']:
            buf = np.zeros((B, 1 + 2 * w['pt_len']), dtype=np.int32)
            for b, (tok, pr) in enumerate(out):
                buf[b, 0] = tok.numel()
                buf[b, 1:1 + tok.numel()] = tok.numpy()
                buf[b, 1 + w['pt_len']:1 + w['pt_len'] + tok.numel()] = pr.numpy().view(np.int32)
            return gc.gather(buf, world)
        return gather_sequences(out, vocab, n_pages=world * B, ctx=gc)

    def gather(j, out, s):
        if lane is not None:      # issued by the lane thread in batch order on the gather context; not waited for here
            lane.submit(s, lambda: gather_now(out, gctx))
        elif order is not None:   # this thread gathers on its own context, when it is batch s's turn
            turn_results[s] = order.run(s, lambda: gather_now(out, ctxs[j]))

    def step_resident(j, s):
        out = run_model(j, dev_in)
        gather(j, out, s)
        return out

    def step_e2e(j, s):
        out = run_model(j, host_in)
        gather(j, out, s)
        return out

    def run_steps(fn, steps):
        """`steps` batches; step s runs on context s % C.  One host thread per context (the C calls release the GIL, the
        per-context streams overlap on the device) + the collective lane.  Returns, per context, (last result, its gathered
        copy) once every gather of the run has completed."""
        outs = [None] * C_
        errors = []
        turn_results.clear()
        if lane is not None:
            lane.start(0)
        if order is not None:
            order.reset(0)

        def worker(j):
            try:
                for s in range(j, steps, C_):
                    outs[j] = fn(j, s)
            except BaseException as e:       # do not leave the other threads waiting on the lane
                errors.append(e)
                if lane is not None:
                    lane.fail(e)
                if order is not None:
                    order.fail(e)
        if C_ == 1:
            worker(0)
        else:
            ts = [threading.Thread(target=worker, args=(j,)) for j in range(C_)]
            for t in ts:
                t.start()
            for t in ts:
                t.join()
        if errors:
            raise errors[0]
        if lane is not None:
            lane.drain(steps)
        last_step = [j + C_ * ((steps - 1 - j) // C_) if j < steps else None for j in range(C_)]
        gathered = (lambda t: lane.result(t)) if lane is not None else (lambda t: turn_results.get(t))
        return [(outs[j], gathered(last_step[j]) if last_step[j] is not None else None) for j in range(C_)]

    def timed(fn, steps, warmup):
        faulthandler.dump_traceback_later(args.watchdog_s, exit=True)
        try:
            return timed_(fn, steps, warmup)
        finally:
            faulthandler.cancel_dump_traceback_later()

    def timed_(fn, steps, warmup):
        if lane is not None:
            lane.start(0)
        if order is not None:
            order.reset(0)
        for j in range(C_):          # every context runs once, one after the other (graph capture, descriptor caches) ...
            fn(j, j)
        if lane is not None:
            lane.drain(C_)
        run_steps(fn, warmup)        # ... then `warmup` untimed steps through the scheduler
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        for cx in ctxs:
            cx.launch_count(True)
        e0 = torch.cuda.Event(enable_timing=True)
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(C_)]
        e0.record(streams[0])
        for j in range(1, C_):
            streams[j].wait_event(e0)
        last = run_steps(fn, steps)   # returns after the last gather of the run has completed
        for j in range(C_):
            ends[j].record(streams[j])
        if gstream is not None:
            eg = torch.cuda.Event(enable_timing=True)
            eg.record(gstream)
            ends.append(eg)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = max(e0.elapsed_time(e) for e in ends)
        t = torch.tensor([ms], device='cuda', dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), sum(cx.launch_count(True) for cx in ctxs), last

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_total, launches, last = timed(step_resident, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(last[(args.steps - 1) % C_][0], w, args.dump_outputs)   # step s ran on context s % C
    ms_e2e, _, last_e2e = timed(step_e2e, args.steps, max(3, args.warmup // 2))

    out0, gathered0 = last[0]
    # ---- what was decoded, and what crossed PCIe per step
    if is_mgp:
        n_chars = mgp_decoded_chars(out0[0])
        d2h_bytes = out0[0].numel() * 4 + out0[1].numel() * 4
    elif w['points_only']:
        n_chars = sum(int(t.numel()) for t, _ in out0)
        d2h_bytes = sum(int(t.numel()) * 12 for t, _ in out0) + 4 * B
    else:
        n_chars = sum(0 if o is None else o[0][2].numel() for o in out0)
        d2h_bytes = sum(0 if o is None else sum(t.numel() * 8 for t in o[0]) + o[1][0].numel() * 4 for o in out0) + 4 * B

    # ---- self-check of the timed run: rank 0's first page (page seed 1000) against the reference's own output; with
    #      N > 1 also the all-gathered copy of that page and the global page count
    check = None
    if name == 'omni':
        check = self_check_omni(out0[0])
        if world > 1 and rank == 0:
            check['gathered_pages'] = len(gathered0)
            g0 = gathered0[0]
            check['gathered_page0_equals_local'] = bool(g0 is not None and all(
                torch.equal(a, b) for a, b in zip(g0[0], out0[0][0])))
            check['ok'] = bool(check.get('ok')) and check['gathered_page0_equals_local'] and len(gathered0) == world * B

    # ---- roofline of the dominant kernel (tcgen05 GEMM), measured live with CUDA events on the ctx stream
    M_, N_, K_ = w['gemm']
    gemm_ms, _ = ctx.bench_gemm_ex(M_, N_, K_, 1, 1, 1, iters=20)   # GELU + split-bf16 epilogue, as the model issues it
    burst, sustained, hbm, peak_src = peaks()
    achieved = 2.0 * M_ * N_ * K_ / (gemm_ms * 1e-3) / 1e12
    torch.cuda.synchronize()
    phase_ms, enc_ms = None, None
    def one_step():
        if lane is not None:
            lane.start(0)
        if order is not None:
            order.reset(0)
        step_resident(0, 0)
        if lane is not None:
            lane.drain(1)

    one_step()                             # one isolated step: device times without cross-batch contention
    if not is_mgp:
        phase_ms = ctx.omni_last_timing()
    ctx.set_option('profile_gemm', 1)
    one_step()
    g_ms, g_flops, g_n = ctx.profile_read()
    ctx.set_option('profile_gemm', 0)
    torch.cuda.synchronize()
    e_a, e_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_a.record(streams[0])
    if is_mgp:
        model.recognize(dev_in)
    else:
        model.encode(dev_in, None)
    e_b.record(streams[0])
    torch.cuda.synchronize()
    iso_ms = e_a.elapsed_time(e_b)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    ms_per_step = ms_total / args.steps
    ips = world * B / (ms_per_step * 1e-3)
    ips_e2e = world * B / (ms_e2e / args.steps * 1e-3)
    cfg = workload_config(name, world, nsplit)
    line = {
        'metric': 'doc_images_per_sec', 'value': ips, 'unit': 'images/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None,
        'dtype': 'bf16x3-split (fp32-class, fp32 accumulate)' if nsplit == 3 else 'bf16',
        'data': 'synthetic', 'config': cfg,
        'run': {'in_flight_contexts_per_gpu': C_, 'weights_shared_by_contexts': True,
                'weights_startup_s': weights_s, 'weights_path': 'alm_broadcast_weights (one NCCL broadcast of the converted '
                'planes)' if world > 1 else 'alm_load_weights', 'gather': f'alm_gather_sequences for every timed step ({args.collectives}), all complete inside the timed region'
                if world > 1 else 'n/a (1 GPU)', **({'options': args.opt} if args.opt else {})},
        'decoded_chars_per_sec': world * n_chars / (ms_per_step * 1e-3),
        'e2e': {'value': ips_e2e, 'unit': 'images/s', 'h2d_bytes_per_step': h2d_bytes, 'd2h_bytes_per_step': d2h_bytes},
        'gpu_launches': launches,
        'clocks': clocks,
        'self_check': check,
        'roofline': {'bound': 'tensor', 'kernel': f'gemm_tcgen05_kernel<256,{nsplit}>',
                     'launch': f'{w["gemm_name"]} (bias + GELU + split-bf16 output), timed alone with CUDA events',
                     'shape': {'M': M_, 'N': N_, 'K': K_}, 'achieved': achieved, 'peak': burst, 'unit': 'TFLOP/s',
                     'frac': achieved / burst,
                     'traffic': ncu_traffic_bytes(w.get('gemm_ncu', '')),
                     'algorithmic_bytes': float(M_ * K_ * 4 + N_ * K_ * 4 + M_ * N_ * 4) if nsplit == 3 else float(M_ * K_ * 2 + N_ * K_ * 2 + M_ * N_ * 4),
                     'peak_source': f'{peak_src}, bf16 burst (kernel timed alone)',
                     'mma_passes_per_flop': nsplit, 'tensor_pipe_frac': achieved * nsplit / burst,
                     'all_gemms_per_step': {'launches': g_n, 'ms': g_ms,
                                            'algorithmic_tflops': g_flops / (g_ms * 1e-3) / 1e12 if g_ms else None,
                                            'frac_of_sustained_peak': (g_flops / (g_ms * 1e-3) / 1e12 / sustained) if g_ms else None}},
    }
    if is_mgp:
        line['forward_ms_per_batch_isolated'] = iso_ms
        line['algorithmic_tflops'] = MGP_GFLOP_PER_CROP * B / iso_ms
        line['frac_of_sustained_peak'] = MGP_GFLOP_PER_CROP * B / iso_ms / sustained
    else:
        line['phase_ms'] = phase_ms
        line['encoder_ms_per_batch'] = iso_ms
        line['encoder_algorithmic_tflops'] = ENC_GFLOP[w['page']] * B / iso_ms
        line['encoder_frac_of_sustained_peak'] = ENC_GFLOP[w['page']] * B / iso_ms / sustained
    if not args.no_cpu_baseline:
        line['cpu_baseline'] = cpu_baseline_bounded(name)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
