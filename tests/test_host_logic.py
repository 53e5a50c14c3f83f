"""CPU checks of host-side scheduling arithmetic (no GPU).

* `bench.py`: workload table / config object shared by both arms, decoded-character counting.
* the run / owner arithmetic of the persistent fused cross-attention (`csrc/xattn.cu`): restated here line for
  line (integer arithmetic only) and checked for the invariants the kernel's merge protocol relies on.
"""
import importlib.util
import os
import random

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location('bench_mod', os.path.join(REPO, 'bench.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_bench_workloads_and_reference_config_agree():
    """Every BASELINE config that bench.py measures is a named workload, and the GPU arm and the reference arm print
    the same `config` object for it (what the driver's same_config check compares)."""
    b = _bench()
    assert set(b.WORKLOADS) == {'omni', 'mgpstr', 'table', 'platypus'}
    for name, w in b.WORKLOADS.items():
        for world in (1, 2, 8):
            c1, c2 = b.workload_config(name, world, 3), b.workload_config(name, world, 1)
            assert c1 == c2 and c1['global_batch'] == world * w['batch'] and c1['parallelism'] == f'dp{world}'
    assert b.WORKLOADS['omni']['pt_len'] == 2 * b.N_INST == 128 and b.WORKLOADS['table']['pt_len'] == 512


def test_roofline_traffic_comes_from_the_committed_captures_of_the_same_launch():
    """`roofline.traffic` of the bench line is read from the ncu capture of the launch the line names (profiles/): the
    file every workload points at exists, parses, and its DRAM bytes are of the order of the launch's algorithmic bytes."""
    b = _bench()
    for name, w in b.WORKLOADS.items():
        f = w.get('gemm_ncu')
        if not f:
            continue
        t = b.ncu_traffic_bytes(f)
        assert t is not None and t > 0, (name, f)
        M, N, K = w['gemm']
        assert 0.3 < t / (M * K * 4 + N * K * 4 + M * N * 4) < 3.0, (name, t)


def test_mgp_decoded_chars_counts_tokens_before_eos():
    import torch
    b = _bench()
    ids = torch.zeros(3, 2, 27, dtype=torch.int32)
    ids[0, 0, 1:6] = torch.tensor([5, 6, 7, 1, 9])   # 3 chars then [s]
    ids[0, 1, 1:] = 4                                 # no [s]: all 26 positions count
    assert b.mgp_decoded_chars(ids) == 3 + 26


def test_dump_outputs_writes_fixed_shape_float_arrays(tmp_path):
    """bench.py --dump-outputs: per workload kind, what the timed path returns is written as float32 / float64 .npy files
    of fixed shape (ragged per-page sequences padded with -1), with the ids and probabilities unchanged."""
    import numpy as np
    import torch
    b = _bench()
    L, maxi = b.REC_LEN, b.WORKLOADS['omni']['pt_len'] // 2
    page = lambda n: ([torch.arange(2 * n).reshape(1, -1), torch.arange(32 * n).reshape(1, -1) + 7,
                       torch.arange(n * L).reshape(1, n, L) + 1000], [torch.rand(n, L)])
    omni = [page(3), None, page(maxi)]
    b.dump_outputs(omni, b.WORKLOADS['omni'], str(tmp_path / 'omni'))
    d = {k: np.load(tmp_path / 'omni' / f'{k}.npy') for k in ('n_instances', 'pt', 'poly', 'rec', 'rec_probs')}
    assert d['n_instances'].tolist() == [3, 0, maxi]
    assert d['pt'].shape == (3, maxi, 2) and d['poly'].shape == (3, maxi, 32) and d['rec'].shape == (3, maxi, L)
    assert d['rec_probs'].dtype == np.float32 and all(d[k].dtype == np.float64 for k in ('n_instances', 'pt', 'poly', 'rec'))
    assert np.array_equal(d['poly'][0, :3].reshape(-1), omni[0][0][1].numpy()[0]) and (d['poly'][0, 3:] == -1).all()
    assert (d['pt'][1] == -1).all() and np.array_equal(d['rec'][2], omni[2][0][2].numpy()[0])
    assert np.array_equal(d['rec_probs'][0, :3], omni[0][1][0].numpy())
    P = b.WORKLOADS['table']['pt_len']
    pts = [(torch.arange(5), torch.rand(5)), (torch.arange(P), torch.rand(P))]
    b.dump_outputs(pts, b.WORKLOADS['table'], str(tmp_path / 'table'))
    tok, pr = np.load(tmp_path / 'table' / 'pt.npy'), np.load(tmp_path / 'table' / 'pt_probs.npy')
    assert tok.shape == pr.shape == (2, P) and np.load(tmp_path / 'table' / 'n_tokens.npy').tolist() == [5, P]
    assert np.array_equal(tok[0, :5], np.arange(5)) and (tok[0, 5:] == -1).all() and np.array_equal(pr[1], pts[1][1].numpy())
    ids, prob = torch.randint(0, 50, (3, 4, 27), dtype=torch.int32), torch.rand(3, 4, 27)
    b.dump_outputs((ids, prob), b.WORKLOADS['mgpstr'], str(tmp_path / 'mgp'))
    assert np.array_equal(np.load(tmp_path / 'mgp' / 'ids.npy'), ids.numpy())
    assert np.array_equal(np.load(tmp_path / 'mgp' / 'probs.npy'), prob.numpy())


def _plan(npairs, nkb, num_sms, ctas_per_sm):
    """cross_attn_mq_plan (csrc/xattn.cu)."""
    nb = npairs * nkb
    g = min(nb, num_sms * max(1, ctas_per_sm))
    bpc = nb // g
    return g, (nkb + bpc - 1) // bpc + 1


def test_xattn_runs_partition_the_work_and_bound_the_partials():
    rnd = random.Random(0)
    cases = [(128, 64, 148, 2), (16, 4, 148, 2), (8, 1, 148, 2), (1, 1, 148, 3), (256, 64, 148, 2)]
    cases += [(rnd.randint(1, 300), rnd.randint(1, 70), rnd.choice([16, 132, 148]), rnd.randint(1, 3)) for _ in range(400)]
    for npairs, nkb, sms, cps in cases:
        nb = npairs * nkb
        g, max_parts = _plan(npairs, nkb, sms, cps)
        owner = lambda b: ((b + 1) * g - 1) // nb            # the kernel's `owner` lambda
        seen = [None] * nb
        for cta in range(g):
            lo, hi = cta * nb // g, (cta + 1) * nb // g     # the kernel's run [b, b_end)
            assert hi > lo                                  # no empty CTA: every counted CTA arrives at the merge
            for b in range(lo, hi):
                assert seen[b] is None
                seen[b] = cta
        assert all(x is not None for x in seen)
        for b in range(nb):
            assert owner(b) == seen[b]
        for p in range(npairs):
            first, last = owner(p * nkb), owner(p * nkb + nkb - 1)
            assert 1 <= last - first + 1 <= max_parts      # partial slots reserved per pair suffice
            for cta in range(first, last + 1):              # every CTA in first..last owns a block of this pair
                assert any(seen[b] == cta for b in range(p * nkb, (p + 1) * nkb))


def test_collective_order_runs_tickets_in_order_and_releases_waiters_on_failure():
    """dist.CollectiveOrder: the gathers of several contexts' host threads are issued in ticket (global step) order
    whatever order the threads arrive in; a failing ticket releases the later ones with an error instead of hanging."""
    import threading
    import time
    import pytest
    from advancedliteratemachinery_b200.dist import CollectiveOrder
    order, seen = CollectiveOrder(timeout_s=20.0), []

    def worker(t, delay):
        time.sleep(delay)
        order.run(t, lambda: seen.append(t))
    ts = [threading.Thread(target=worker, args=(t, d)) for t, d in ((3, 0.0), (1, 0.05), (0, 0.15), (2, 0.1))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert seen == [0, 1, 2, 3]

    order.reset(0)
    errs = []

    def waiter():
        try:
            order.run(1, lambda: None)
        except RuntimeError as e:
            errs.append(e)
    w = threading.Thread(target=waiter)
    w.start()
    with pytest.raises(ValueError):
        order.run(0, lambda: (_ for _ in ()).throw(ValueError('boom')))
    w.join(10)
    assert not w.is_alive() and len(errs) == 1


def test_collective_lane_runs_in_ticket_order_without_blocking_the_submitters():
    """dist.CollectiveLane: the compute threads submit their batch's gather and go on; ONE lane thread runs the gathers in
    ticket order; drain() waits for them, a failing gather surfaces in drain() / submit() instead of hanging anyone."""
    import threading
    import time
    import pytest
    from advancedliteratemachinery_b200.dist import CollectiveLane
    lane, seen = CollectiveLane(max_ahead=4, timeout_s=20.0), []
    lane.start(0)

    def worker(j):
        for s in range(j, 12, 3):
            time.sleep(0.01 * ((s * 7) % 3))
            lane.submit(s, lambda s=s: (time.sleep(0.005), seen.append(s), s * s)[-1])
    ts = [threading.Thread(target=worker, args=(j,)) for j in range(3)]
    t0 = time.time()
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    lane.drain(12)
    assert seen == list(range(12)) and lane.result(11) == 121 and time.time() - t0 < 10
    lane.start(0)
    lane.submit(0, lambda: (_ for _ in ()).throw(ValueError('boom')))
    with pytest.raises(RuntimeError):
        lane.drain(1)
    with pytest.raises(RuntimeError):
        lane.submit(1, lambda: None)
    lane.stop()


def test_epilogue_and_window_staging_layouts_are_bijective_and_conflict_free():
    """Integer restatement of the shared-memory addressing of the round-2 kernels (no GPU):
    * TMA-store GEMM epilogue (csrc/gemm.cu, PLAIN == 2): lane r writes 16-byte chunk k of its 64-byte row at
      r*64 + ((k ^ ((r >> 1) & 3)) << 4) -- the CU_TENSOR_MAP_SWIZZLE_64B pattern (address bits [4,5] ^= bits [7,8]); every
      quarter-warp store covers 32 distinct banks and the block is filled exactly once;
    * window_attention_ms (csrc/wattn_ms.cu): sw128(row, chunk) = row*128 + ((chunk ^ (row & 7)) << 4), the 128-byte swizzle
      (bits [4,6] ^= bits [7,9]): the 8 rows of an ldmatrix 8x8 tile hit 8 distinct 16-byte bank groups; the bias pitch of 56
      floats makes the float2 reads of a half-warp (4 rows x 4 column pairs) conflict-free."""
    # --- 64-byte swizzle of the epilogue staging block (32 rows x 64 bytes)
    seen = set()
    for k in range(4):
        for q in range(4):                                    # a 16-byte store is issued per quarter-warp (8 lanes)
            banks = set()
            for r in range(8 * q, 8 * q + 8):
                a = r * 64 + ((k ^ ((r >> 1) & 3)) << 4)
                assert a ^ (((a >> 7) & 3) << 4) == r * 64 + k * 16      # == hardware pattern applied to the linear address
                seen.add(a)
                banks.update(range((a // 4) % 32, (a // 4) % 32 + 4))
            assert len(banks) == 32
    assert seen == set(range(0, 2048, 16))
    # --- 128-byte swizzle of the window tiles (64 rows x 128 bytes), ldmatrix row groups
    sw128 = lambda row, chunk: row * 128 + ((chunk ^ (row & 7)) << 4)
    for chunk in range(8):
        for r0 in range(0, 64, 8):
            groups = {(sw128(r0 + i, chunk) // 16) % 8 for i in range(8)}
            assert len(groups) == 8
            for i in range(8):
                a = sw128(r0 + i, chunk)
                assert a ^ (((a >> 7) & 7) << 4) == (r0 + i) * 128 + chunk * 16
    # --- bias pitch: lanes (g, t) of a half-warp read float2 at row g (4 consecutive rows), columns 8j + 2t
    pitch = 56
    for j in range(7):
        for half in range(2):
            banks = []
            for g in range(4 * half, 4 * half + 4):
                for t in range(4):
                    w0 = (16 + g) * pitch + 8 * j + 2 * t       # any band: the row offset only adds a multiple of the pitch
                    banks += [w0 % 32, (w0 + 1) % 32]
            assert len(set(banks)) == 32
