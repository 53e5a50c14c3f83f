"""Window-prompted decoding at config 2: does tiling a page into R windows shorten the decode?

16 x 1024^2 synthetic pages (bench.py's config-2 pages, seed 1000 + p), synthetic weights with pt_eos_bias -30 (no
EOS is ever emitted, so the decode work is pinned by pt_seq_length), 64 points per page in every arm:

  A  the default prompt, 64 points per page            (pt_seq_length 128, S = 16 point sequences, skinny path)
  B  the 2x2 grid, R = 4, 16 points per window          (pt_seq_length 32,  S = 64, skinny 64-row path)
  C  the 3x3 grid, R = 9, 7 points per window (63/page) (pt_seq_length 14,  S = 144, tensor-core path)

The arms run alternated after a warm-up of each.  Per arm: point-loop ms and poly + rec ms (alm_omni_last_timing,
device events), decode ms (host clock around the synchronous decode call), pages/s of encode + decode, instances per
page.  Arm B's outputs are checked against four separate single-window decodes of the same pages.  The card name and
power limit are read in the same run.

    python tools/bench_prompted.py [--rounds 5] [--out profiles/r03_bench_prompted.json]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

B, PAGE, REC_LEN = 16, 1024, 25
ARMS = {'A': (1, 1, 64), 'B': (2, 2, 16), 'C': (3, 3, 7)}   # grid nx, ny, points per window


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(',')]
        return {'name': name, 'power_limit': power, 'max_sm_clock': clock}
    except Exception as e:  # the numbers are still device-event timings; say that the card was not read
        return {'error': repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--out', default=os.path.join(REPO, 'profiles', 'r03_bench_prompted.json'))
    a = ap.parse_args()
    import torch
    from advancedliteratemachinery_b200 import OmniParserB200, OmniVocab
    from advancedliteratemachinery_b200 import synthetic as W
    assert torch.cuda.is_available(), 'this measurement needs the GPU'
    info = card()
    m = OmniParserB200(W.omniparser_state_dict(seed=0, pt_eos_bias=-30.0), OmniVocab(rec_length=REC_LEN),
                       workspace_mb=20480)
    g = [torch.Generator().manual_seed(1000 + p) for p in range(B)]
    pages = torch.cat([torch.randn(1, 3, PAGE, PAGE, generator=x) for x in g]).cuda()
    torch.cuda.synchronize()

    def run(arm):
        nx, ny, npts = ARMS[arm]
        m.vocab.pt_seq_length = 2 * npts
        prompts = m.vocab.grid_prompts(nx, ny)
        t0 = time.perf_counter()
        m.encode(pages)
        m.ctx.synchronize()
        t1 = time.perf_counter()
        outs = m.decode_prompted(prompts, merge=True)
        t2 = time.perf_counter()
        tm = m.ctx.omni_last_timing()
        inst = [0 if o is None else o[0][0].numel() // 2 for o in outs]
        return dict(encode_ms=tm['encode_ms'], pt_loop_ms=tm['pt_loop_ms'], poly_rec_ms=tm['poly_rec_loops_ms'],
                    decode_ms=(t2 - t1) * 1e3, step_ms=(t2 - t0) * 1e3, inst=statistics.mean(inst))

    for arm in ARMS:
        for _ in range(a.warmup):
            run(arm)
    samples = {arm: [] for arm in ARMS}
    for _ in range(a.rounds):
        for arm in ARMS:
            samples[arm].append(run(arm))
    res = {}
    for arm, ss in samples.items():
        med = {k: statistics.median(s[k] for s in ss) for k in ss[0]}
        nx, ny, npts = ARMS[arm]
        res[arm] = {'windows': nx * ny, 'points_per_window': npts, 'point_sequences': B * nx * ny,
                    'pt_loop_ms': round(med['pt_loop_ms'], 2), 'poly_rec_ms': round(med['poly_rec_ms'], 2),
                    'decode_ms': round(med['decode_ms'], 2), 'encode_ms': round(med['encode_ms'], 2),
                    'pages_per_s': round(B / (med['step_ms'] / 1e3), 1), 'instances_per_page': med['inst'],
                    'decode_ms_all': [round(s['decode_ms'], 2) for s in ss]}

    # arm B against four separate single-window decodes of the same pages
    nx, ny, npts = ARMS['B']
    m.vocab.pt_seq_length = 2 * npts
    grid = m.vocab.grid_prompts(nx, ny)
    m.encode(pages)
    pts, outs = m.decode_points_prompted(grid), m.decode_prompted(grid)
    check = {'points_bit_identical': True, 'poly_rec_ids_equal': True, 'rec_prob_max_rel': 0.0}
    for r in range(nx * ny):
        sp, so = m.decode_points(grid[r][None]), m.decode(grid[r][None])
        for b in range(B):
            check['points_bit_identical'] &= bool(torch.equal(pts[b][r][0], sp[b][0]) and torch.equal(pts[b][r][1], sp[b][1]))
            (pt, poly, rec), (pr,) = outs[b][r]
            (pt1, poly1, rec1), (pr1,) = so[b]
            check['poly_rec_ids_equal'] &= bool(torch.equal(pt, pt1) and torch.equal(poly, poly1) and torch.equal(rec, rec1))
            rel = float(((pr - pr1).abs() / pr1.abs().clamp_min(1e-30)).max())
            check['rec_prob_max_rel'] = max(check['rec_prob_max_rel'], rel)
    out = {'workload': f'config 2: {B} x {PAGE}^2 synthetic pages (seed 1000 + p), synthetic weights seed 0 with '
                       f'pt_eos_bias -30 (no EOS: decode pinned by pt_seq_length), rec_length {REC_LEN}',
           'card': info, 'rounds': a.rounds, 'warmup_per_arm': a.warmup, 'statistic': 'median over rounds',
           'arms': res, 'arm_B_vs_single_window_decodes': check}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == '__main__':
    main()
