"""Window-prompted OmniParser decoding: R spatial / character window prompts per page over one encode
(alm_omni_decode_prompted / alm_omni_decode_points_prompted, OmniVocab.window_prompt / grid_prompts).

CPU: the restated oracle reproduces the prompted reference fixture (oracle/gen_golden_prompts.py), the prompt builders
reproduce the windows of dataset/collate_fn.py, and the merged per-page packing.
GPU: fixture parity in one call, per-page prompt sets, R = 1 == the classic entry points, window independence at
benchmark scale, per-sequence EOS, error paths.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle.gen_golden import config2_page, omni_inputs
from oracle.gen_golden_prompts import PROMPT_PAGES, PROMPT_PT_SEQ_LENGTH, PROMPT_REC_LENGTH, PROMPT_WEIGHTS

torch.set_grad_enabled(False)


def _fixture(golden_dir):
    return np.load(os.path.join(golden_dir, 'omni_prompts.npz'))


def _page(gold, i):
    return omni_inputs(dict(PROMPT_PAGES[i], seed=int(gold['page_seeds'][i])))


# ------------------------------------------------------------------------------------------------------- CPU
def test_prompt_fixture_is_well_formed(golden_dir):
    gold = _fixture(golden_dir)
    assert int(gold['wseed'][0]) == PROMPT_WEIGHTS['wseed'] and float(gold['pt_eos_bias'][0]) == PROMPT_WEIGHTS['pt_eos_bias']
    assert tuple(gold['lengths']) == (PROMPT_PT_SEQ_LENGTH, PROMPT_REC_LENGTH)
    R = gold['prompts'].shape[0]
    assert R >= 4
    for i in range(len(PROMPT_PAGES)):
        n = [0 if gold[f'p{i}_r{j}_none'][0] else gold[f'p{i}_r{j}_pt'].size // 2 for j in range(R)]
        assert len(set(n)) > 1 and 0 in n, n   # different lengths and a None on every page
        for j in range(R):
            assert float(gold[f'p{i}_r{j}_min_gap'].min()) >= 1e-4


def test_oracle_matches_prompted_reference_fixture(golden_dir):
    from oracle import omniparser_ref as O
    from tests.conftest import omni_sd
    gold = _fixture(golden_dir)
    sd = omni_sd(PROMPT_WEIGHTS['wseed'], PROMPT_WEIGHTS['pt_eos_bias'])
    for i in range(len(PROMPT_PAGES)):
        img, mask = _page(gold, i)
        mem, pos, kpm, _ = O.encode(img, mask, sd)
        for j, window in enumerate(gold['prompts']):
            res = O.greedy_text_spotting(mem[0], kpm[0], pos[0], sd, torch.from_numpy(window)[None],
                                         PROMPT_PT_SEQ_LENGTH, PROMPT_REC_LENGTH)
            key = f'p{i}_r{j}_'
            if gold[key + 'none'][0]:
                assert res is None, (i, j)
                continue
            (pt, poly, rec), (probs,) = res
            assert np.array_equal(pt.numpy(), gold[key + 'pt']), (i, j)
            assert np.array_equal(poly.numpy(), gold[key + 'poly']), (i, j)
            assert np.array_equal(rec.numpy(), gold[key + 'rec']), (i, j)
            np.testing.assert_allclose(probs.numpy(), gold[key + 'probs'], atol=1e-5, rtol=0)


# (num_x, num_y) pairs of dataset/collate_fn.py:55-56 and their tiles written out by hand ([x0, y0, x1, y1], i over x
# outer, j over y inner)
GRIDS = {
    (3, 3): [[0, 0, 333, 333], [0, 333, 333, 666], [0, 666, 333, 999], [333, 0, 666, 333], [333, 333, 666, 666],
             [333, 666, 666, 999], [666, 0, 999, 333], [666, 333, 999, 666], [666, 666, 999, 999]],
    (3, 1): [[0, 0, 333, 999], [333, 0, 666, 999], [666, 0, 999, 999]],
    (1, 3): [[0, 0, 999, 333], [0, 333, 999, 666], [0, 666, 999, 999]],
    (3, 2): [[0, 0, 333, 500], [0, 500, 333, 999], [333, 0, 666, 500], [333, 500, 666, 999], [666, 0, 999, 500],
             [666, 500, 999, 999]],
    (2, 3): [[0, 0, 500, 333], [0, 333, 500, 666], [0, 666, 500, 999], [500, 0, 999, 333], [500, 333, 999, 666],
             [500, 666, 999, 999]],
    (2, 2): [[0, 0, 500, 500], [0, 500, 500, 999], [500, 0, 999, 500], [500, 500, 999, 999]],
    (2, 1): [[0, 0, 500, 999], [500, 0, 999, 999]],
    (1, 2): [[0, 0, 999, 500], [0, 500, 999, 999]],
}


@pytest.mark.parametrize('nx,ny', list(GRIDS))
def test_grid_prompts_are_the_training_tiles(nx, ny):
    from advancedliteratemachinery_b200 import OmniVocab
    v = OmniVocab()
    p = v.grid_prompts(nx, ny)
    want = [w + [1000, 1095, v.pt_sos_index] for w in GRIDS[(nx, ny)]]
    assert p.dtype == torch.long and p.tolist() == want
    p5 = OmniVocab(use_char_window_prompt=False).grid_prompts(nx, ny)
    assert p5.tolist() == [w + [v.pt_sos_index] for w in GRIDS[(nx, ny)]]
    pc = v.grid_prompts(nx, ny, char_window=(10, 40))
    assert pc[:, 4:6].tolist() == [[1010, 1040]] * (nx * ny)


def test_window_prompt_layout():
    from advancedliteratemachinery_b200 import OmniVocab
    v = OmniVocab()
    assert torch.equal(v.window_prompt(0, 0, 999, 999), v.pt_prompt())   # the default prompt is the whole-page window
    assert v.window_prompt(120, 250, 870, 999, 10, 40).tolist() == [[120, 250, 870, 999, 1010, 1040, 1100]]
    v5 = OmniVocab(use_char_window_prompt=False)
    assert torch.equal(v5.window_prompt(0, 0, 999, 999), v5.pt_prompt())
    assert v5.window_prompt(5, 6, 7, 8, 10, 40).tolist() == [[5, 6, 7, 8, 1100]]


def _out(n, seed, L=25):
    g = torch.Generator().manual_seed(seed)
    return ([torch.randint(0, 1000, (1, 2 * n), generator=g), torch.randint(0, 1000, (1, 32 * n), generator=g),
             torch.randint(1000, 1100, (1, n, L), generator=g)], [torch.rand(n, L, generator=g)])


def test_merge_packs_windows_in_prompt_order():
    from advancedliteratemachinery_b200.omniparser import merge_window_outputs
    a, b = _out(2, 1), _out(3, 2)
    m = merge_window_outputs([None, a, None, b])
    assert torch.equal(m[0][0], torch.cat([a[0][0], b[0][0]], 1)) and m[0][0].shape == (1, 10)
    assert torch.equal(m[0][1], torch.cat([a[0][1], b[0][1]], 1)) and m[0][1].shape == (1, 160)
    assert torch.equal(m[0][2], torch.cat([a[0][2], b[0][2]], 1)) and m[0][2].shape == (1, 5, 25)
    assert torch.equal(m[1][0], torch.cat([a[1][0], b[1][0]], 0)) and m[1][0].shape == (5, 25)
    assert merge_window_outputs([None, None]) is None
    assert merge_window_outputs([]) is None
    one = merge_window_outputs([a])
    assert all(torch.equal(x, y) for x, y in zip(one[0] + one[1], a[0] + a[1]))


# ------------------------------------------------------------------------------------------------------- GPU
_MODELS = {}


def _model(wseed, bias, vie=0):
    from advancedliteratemachinery_b200 import OmniParserB200, OmniVocab
    from tests.conftest import omni_sd
    key = (wseed, bias, vie)
    if key not in _MODELS:
        for k in list(_MODELS):
            _MODELS.pop(k).ctx.close()
        if vie:
            from advancedliteratemachinery_b200 import synthetic as W
            sd = W.omniparser_state_dict(seed=wseed, vie_categories=vie, pt_eos_bias=bias)
        else:
            sd = omni_sd(wseed, bias)
        _MODELS[key] = OmniParserB200(sd, OmniVocab(vie_categories=vie), workspace_mb=20480)
    m = _MODELS[key]
    m.ctx.set_option('use_graphs', 1)
    return m


def _fixture_model(gold):
    m = _model(PROMPT_WEIGHTS['wseed'], PROMPT_WEIGHTS['pt_eos_bias'])
    m.vocab.pt_seq_length, m.vocab.rec_length = PROMPT_PT_SEQ_LENGTH, PROMPT_REC_LENGTH
    imgs, masks = zip(*[_page(gold, i) for i in range(len(PROMPT_PAGES))])
    m.encode(torch.cat(imgs).cuda(), torch.cat(masks).cuda())
    return m


def _check_against_fixture(gold, i, j, out):
    key = f'p{i}_r{j}_'
    if gold[key + 'none'][0]:
        assert out is None, (i, j)
        return
    assert out is not None, (i, j)
    (pt, poly, rec), (probs,) = out
    assert np.array_equal(pt.numpy(), gold[key + 'pt']), (i, j, 'pt ids differ from the reference')
    assert np.array_equal(poly.numpy(), gold[key + 'poly']), (i, j, 'poly ids differ from the reference')
    assert np.array_equal(rec.numpy(), gold[key + 'rec']), (i, j, 'rec ids differ from the reference')
    np.testing.assert_allclose(probs.numpy(), gold[key + 'probs'], rtol=2e-3, atol=1e-7)


@pytest.mark.gpu
def test_prompted_fixture_parity_in_one_call(golden_dir):
    gold = _fixture(golden_dir)
    m = _fixture_model(gold)
    pages = m.decode_prompted(torch.from_numpy(gold['prompts']))
    for i, outs in enumerate(pages):
        assert len(outs) == gold['prompts'].shape[0]
        for j, out in enumerate(outs):
            _check_against_fixture(gold, i, j, out)


@pytest.mark.gpu
def test_per_page_prompt_sets(golden_dir):
    gold = _fixture(golden_dir)
    m = _fixture_model(gold)
    sets = [[0, 1, 2], [3, 4, 0]]
    P = torch.from_numpy(gold['prompts'])
    pages = m.decode_prompted(torch.stack([P[s] for s in sets]))
    for i, outs in enumerate(pages):
        for r, out in enumerate(outs):
            _check_against_fixture(gold, i, sets[i][r], out)
    merged = m.decode_prompted(torch.stack([P[s] for s in sets]), merge=True)
    from advancedliteratemachinery_b200.omniparser import merge_window_outputs
    for i in range(2):
        want = merge_window_outputs(pages[i])
        assert (merged[i] is None) == (want is None)
        if want is not None:
            assert all(torch.equal(x, y) for x, y in zip(merged[i][0] + merged[i][1], want[0] + want[1]))


def _raw_decode(m, prompts, R, maxi=None):
    """alm_omni_decode_prompted on [B][R][L] prompts: the raw output arrays."""
    v = m.vocab
    B = m.memory_shape()[0]
    maxi = maxi or max(1, v.pt_seq_length // 2)
    p = prompts.to(torch.long).contiguous()
    o = dict(n=np.zeros((B, R), np.int32), pt=np.zeros((B, R, maxi, 2), np.int64), poly=np.zeros((B, R, maxi, 32), np.int64),
             rec=np.zeros((B, R, maxi, v.rec_length), np.int64), prob=np.zeros((B, R, maxi, v.rec_length), np.float32))
    cfg = m._cfg(maxi)
    rc = m.lib.alm_omni_decode_prompted(m.ctx.h, p.data_ptr(), R, p.shape[-1], C.byref(cfg), o['n'].ctypes.data,
                                        o['pt'].ctypes.data, o['poly'].ctypes.data, o['rec'].ctypes.data,
                                        o['prob'].ctypes.data)
    return rc, o


@pytest.mark.gpu
def test_single_prompt_broadcast_is_the_classic_path(golden_dir):
    gold = _fixture(golden_dir)
    m = _fixture_model(gold)
    v = m.vocab
    B, maxi = 2, max(1, v.pt_seq_length // 2)
    for window in gold['prompts']:
        prompt = torch.from_numpy(window)
        rc, o = _raw_decode(m, prompt.reshape(1, 1, -1).expand(B, 1, -1), 1)
        assert rc == 0
        n = np.zeros(B, np.int32)
        pt, poly = np.zeros((B, maxi, 2), np.int64), np.zeros((B, maxi, 32), np.int64)
        rec, prob = np.zeros((B, maxi, v.rec_length), np.int64), np.zeros((B, maxi, v.rec_length), np.float32)
        cfg = m._cfg(maxi)
        m.ctx.check(m.lib.alm_omni_decode(m.ctx.h, prompt.data_ptr(), prompt.numel(), C.byref(cfg), n.ctypes.data,
                                          pt.ctypes.data, poly.ctypes.data, rec.ctypes.data, prob.ctypes.data))
        assert np.array_equal(o['n'][:, 0], n)
        for k, ref in (('pt', pt), ('poly', poly), ('rec', rec), ('prob', prob)):
            assert np.array_equal(o[k][:, 0], ref), k   # bit for bit, all output arrays
        pts = m.decode_points_prompted(prompt[None])
        ref = m.decode_points(prompt[None])
        for b in range(B):
            assert torch.equal(pts[b][0][0], ref[b][0]) and torch.equal(pts[b][0][1], ref[b][1])


@pytest.mark.gpu
def test_per_sequence_eos_and_graph_replay(golden_dir):
    gold = _fixture(golden_dir)
    m = _fixture_model(gold)
    P = torch.from_numpy(gold['prompts'])
    runs = {}
    for graphs in (1, 0):
        m.ctx.set_option('use_graphs', graphs)
        runs[graphs] = (m.decode_points_prompted(P), m.decode_prompted(P))
    m.ctx.set_option('use_graphs', 1)
    pts, outs = runs[1]
    lens = set()
    for i in range(2):
        for j in range(P.shape[0]):
            single = m.decode_points(P[j][None])[i]
            # every window stops at its own EOS, and the loop runs on while any window of the batch is alive
            assert torch.equal(pts[i][j][0], single[0]) and torch.equal(pts[i][j][1], single[1]), (i, j)
            key = f'p{i}_r{j}_'
            ref_n = 0 if gold[key + 'none'][0] else gold[key + 'pt'].size
            assert pts[i][j][0].numel() == ref_n, (i, j)
            lens.add(ref_n)
    assert len(lens) > 1
    for a, b in zip(runs[1][0], runs[0][0]):
        for (t1, p1), (t0, p0) in zip(a, b):
            assert torch.equal(t1, t0) and torch.equal(p1, p0)
    for a, b in zip(runs[1][1], runs[0][1]):
        for o1, o0 in zip(a, b):
            assert (o1 is None) == (o0 is None)
            if o1 is not None:
                assert all(torch.equal(x, y) for x, y in zip(o1[0] + o1[1], o0[0] + o0[1]))


@pytest.mark.gpu
@pytest.mark.parametrize('B,nx,ny', [(16, 2, 2), (12, 3, 1), (4, 3, 3)])
def test_windows_are_independent_at_benchmark_scale(B, nx, ny):
    """16 x 1024^2 pages (config 2), pt_eos suppressed so every window decodes its pinned length: the prompted call
    against R separate single-window calls.  Point tokens and probabilities bit for bit (same skinny-path arithmetic per
    row, same cross-attention key runs); polygon / recognition ids equal and probabilities within 1e-5 relative in norm
    per (page, window), 1e-4 per element (their cross-attention schedule depends on the instances per image: the
    probabilities of these near-uniform synthetic heads are ~2e-3 and move by ~1e-5 relative)."""
    m = _model(0, -30.0)
    R = nx * ny
    pts_per_window = max(1, 64 // R)
    m.vocab.pt_seq_length, m.vocab.rec_length = 2 * pts_per_window, 25
    m.encode(torch.cat([config2_page(1000 + p)[0] for p in range(B)]).cuda())
    grid = m.vocab.grid_prompts(nx, ny)
    pts = m.decode_points_prompted(grid)
    outs = m.decode_prompted(grid)
    for r in range(R):
        single_pts = m.decode_points(grid[r][None])
        single = m.decode(grid[r][None])
        for b in range(B):
            assert pts[b][r][0].numel() == 2 * pts_per_window
            assert torch.equal(pts[b][r][0], single_pts[b][0]), (b, r)
            assert torch.equal(pts[b][r][1], single_pts[b][1]), (b, r)   # bit-identical probabilities
            (pt, poly, rec), (probs,) = outs[b][r]
            (pt1, poly1, rec1), (probs1,) = single[b]
            assert torch.equal(pt, pt1) and torch.equal(poly, poly1) and torch.equal(rec, rec1), (b, r)
            p, p1 = probs.double(), probs1.double()
            assert float((p - p1).norm() / p1.norm()) <= 1e-5, (b, r)
            assert float(((p - p1).abs() / p1.abs().clamp_min(1e-30)).max()) <= 1e-4, (b, r)


@pytest.mark.gpu
def test_error_paths_leave_the_context_usable(golden_dir):
    from advancedliteratemachinery_b200 import AlmError
    gold = _fixture(golden_dir)
    m = _fixture_model(gold)
    P = torch.from_numpy(gold['prompts'])
    B, V = 2, m.lib.alm_omni_vocab(m.ctx.h)
    ok = m.decode_prompted(P)

    def still_ok():
        again = m.decode_prompted(P)
        for a, b in zip(again, ok):
            for o1, o0 in zip(a, b):
                assert (o1 is None) == (o0 is None)
                if o1 is not None:
                    assert all(torch.equal(x, y) for x, y in zip(o1[0] + o1[1], o0[0] + o0[1]))

    full = P[None].expand(B, -1, -1)
    assert _raw_decode(m, full[:, :0], 0)[0] == -1           # R = 0
    still_ok()
    assert _raw_decode(m, P[[0] * 17][None].expand(B, -1, -1), 17)[0] == -1   # R = 17
    still_ok()
    bad = full.clone()
    bad[1, 2, 3] = V
    assert _raw_decode(m, bad, P.shape[0])[0] == -1          # prompt id >= V
    bad[1, 2, 3] = -1
    assert _raw_decode(m, bad, P.shape[0])[0] == -1          # negative id
    still_ok()
    assert _raw_decode(m, full, P.shape[0], maxi=PROMPT_PT_SEQ_LENGTH // 2 - 1)[0] == -1   # max_instances too small
    still_ok()
    # a window that never emits EOS with pt_seq_length 1024: the position-table error, as the reference raises
    m2 = _model(0, -30.0)
    m2.vocab.pt_seq_length, m2.vocab.rec_length = 1024, 25
    img, mask = _page(gold, 0)
    m2.encode(img.cuda(), mask.cuda())
    with pytest.raises(AlmError, match='position table'):
        m2.decode_prompted(m2.vocab.grid_prompts(2, 1))
    m2.vocab.pt_seq_length = 8
    assert all(o is not None for o in m2.decode_prompted(m2.vocab.grid_prompts(2, 1))[0])
    # KIE checkpoints: not supported by the prompted entry points
    k = _model(2, -30.0, vie=4)
    k.vocab.pt_seq_length = 9
    k.encode(img.cuda(), mask.cuda())
    rc, _ = _raw_decode(k, k.vocab.pt_prompt().reshape(1, 1, -1), 1)
    assert rc == -5
    assert k.decode_kie([(96.0, 128.0)]) is not None   # the context still decodes
