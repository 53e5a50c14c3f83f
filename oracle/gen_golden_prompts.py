"""Pin window-prompted decoding to the UNMODIFIED reference and write tests/golden/omni_prompts.npz.

TEST INFRASTRUCTURE ONLY -- runs in the build container (needs /root/reference).  Usage:

    python -m oracle.gen_golden_prompts

Same recipe as oracle/gen_golden.py: the reference OmniParser module is built as the reference drivers build it,
``load_state_dict(strict=True)`` with the synthetic checkpoint, and run at batch 1 once per (page, prompt) -- the reference
forward takes any pt prompt (model/transformer.py:234-241).  The restatement (oracle/omniparser_ref.py) is run on the same
inputs and must agree; every greedy step must clear the near-tie floor GAP_FLOOR, so the GPU test compares ids bit for bit.

The checkpoint carries an EOS bias chosen so that the prompts of one page stop at different lengths and some
(page, prompt) pairs decode no point at all (the reference returns None): per-sequence EOS is what is being pinned.
"""
from __future__ import annotations

import os
import sys
import tempfile

import numpy as np
import torch

from oracle.gen_golden import GAP_FLOOR, GOLD, REF, SHIM, _maxdiff, omni_inputs
from oracle import weights as W

NB = W.NUM_BINS
_CH = NB + len(W.CHARS)  # last character-window id of the whole character range (engine/val.py:25-28)

# Weights seed 0 with EOS bias 0.6 (0.2 / 0.3 / 0.45 / 0.6 / 0.8 tried): the prompts of one page stop after different
# numbers of points, and every page has a prompt that decodes none.
PROMPT_WEIGHTS = dict(wseed=0, pt_eos_bias=0.6)
PROMPT_PT_SEQ_LENGTH = 12
PROMPT_REC_LENGTH = 25

# The two pages: the canvases of the 'full' and 'masked' cases of gen_golden.py.  The input seed is the first of
# seed, seed + 100, ... whose decodes clear GAP_FLOOR and satisfy the length condition; the file records the one used
# (1000 and 1101: page 1 at seed 1001 had a 6e-5 polygon gap under the random-rectangle prompt).
PROMPT_PAGES = [dict(seed=1000, canvas=(96, 128)), dict(seed=1001, canvas=(96, 128), image=(80, 112))]
RESEED_TRIES = 6

# [x0, y0, x1, y1, char_lo, char_hi, pt_sos] (dataset/collate_fn.py:46-115 windows)
PROMPT_WINDOWS = [
    [0, 0, NB - 1, NB - 1, NB, _CH, W.PT_SOS],          # the default prompt (whole page, every character)
    [500, 0, NB - 1, 500, NB, _CH, W.PT_SOS],           # 2x2 grid, tile i = 1, j = 0 (collate_fn.py:55-69)
    [333, 0, 666, NB - 1, NB, _CH, W.PT_SOS],           # 3x1 grid, the middle strip
    [120, 250, 870, NB - 1, NB, _CH, W.PT_SOS],         # a rectangle of the random kind (collate_fn.py:73-77)
    [0, 0, NB - 1, NB - 1, NB + 10, NB + 40, W.PT_SOS],  # whole page, character sub-range 10..40 (:111-114)
]


def gen_prompts():
    sys.path[:0] = [SHIM, os.path.join(REF, 'OmniParser')]
    tmp = tempfile.mktemp(suffix='.pth')
    torch.save({'model': {}}, tmp)  # satisfies swin_transformer.py:636
    from oracle import omniparser_ref as O
    sys.argv = ['x', '--tfm_pre_norm', '--use_fpn', '--use_char_window_prompt', '--pretrained_file', tmp,
                '--pt_seq_length', str(PROMPT_PT_SEQ_LENGTH), '--rec_length', str(PROMPT_REC_LENGTH)]
    from utils.parser import DefaultParser
    from utils.nested_tensor import NestedTensor
    from model.backbone import build_backbone
    from model.transformer import build_transformer
    from model.omniparser import OmniParser
    args = DefaultParser().parse_args()
    assert (args.pt_sos_index, args.num_bins, len(args.chars)) == (W.PT_SOS, NB, len(W.CHARS))
    sd = W.omniparser_state_dict(seed=PROMPT_WEIGHTS['wseed'], pt_eos_bias=PROMPT_WEIGHTS['pt_eos_bias'])
    model = OmniParser(build_backbone(args), build_transformer(args), args.num_classes, True).eval()
    r = model.load_state_dict(sd, strict=True)
    assert not r.missing_keys and not r.unexpected_keys
    _, poly_prompt, rec_prompt = O.default_prompts(True)
    gold = dict(prompts=np.array(PROMPT_WINDOWS, dtype=np.int64), wseed=np.array([PROMPT_WEIGHTS['wseed']]),
                pt_eos_bias=np.array([PROMPT_WEIGHTS['pt_eos_bias']]),
                lengths=np.array([PROMPT_PT_SEQ_LENGTH, PROMPT_REC_LENGTH]))
    seeds = []
    for i, page in enumerate(PROMPT_PAGES):
        for k in range(RESEED_TRIES):
            case = dict(page, seed=page['seed'] + 100 * k)
            entry = _page_entries(model, sd, O, NestedTensor, case, i, poly_prompt, rec_prompt)
            if entry is not None:
                break
            print(f'page {i}: seed {case["seed"]} rejected, re-seeding')
        assert entry is not None, f'page {i}: no seed in {RESEED_TRIES} tries'
        gold.update(entry)
        seeds.append(case['seed'])
    gold['page_seeds'] = np.array(seeds)
    np.savez_compressed(os.path.join(GOLD, 'omni_prompts.npz'), **gold)
    print('omni_prompts: ok, page seeds', seeds)


def _page_entries(model, sd, O, NestedTensor, page, i, poly_prompt, rec_prompt):
    """Fixture entries of page i under every window, or None when a step is a near-tie or the EOS bias does not give
    different lengths and a None on this page."""
    img, mask = omni_inputs(page)
    mem, pos, kpm, _ = O.encode(img, mask, sd)
    gold, n_pts = {}, []
    for j, window in enumerate(PROMPT_WINDOWS):
        prompt = torch.tensor([window], dtype=torch.long)
        with torch.no_grad():
            out = model(NestedTensor(img, mask), [prompt, poly_prompt, rec_prompt, torch.tensor(page['canvas'])])
            res, logs = O.greedy_text_spotting(mem[0], kpm[0], pos[0], sd, prompt, PROMPT_PT_SEQ_LENGTH,
                                               PROMPT_REC_LENGTH, return_logits=True)
        key = f'p{i}_r{j}_'
        gaps = O.greedy_min_gaps(logs)
        # every step the loops took, including the EOS step of the pt loop (no poly / rec steps when None)
        if min(gaps.values()) < GAP_FLOOR:
            print(f'page {i} prompt {j}: near-tie {gaps}')
            return None
        gold[key + 'min_gap'] = np.array([gaps['pt'], gaps['poly'], gaps['rec']])
        if out is None:
            assert res is None, (i, j)
            gold[key + 'none'] = np.array([1])
            n_pts.append(0)
            continue
        (pt, poly, rec), (probs,) = out
        assert torch.equal(pt, res[0][0]) and torch.equal(poly, res[0][1]) and torch.equal(rec, res[0][2]), (i, j)
        assert _maxdiff(probs, res[1][0]) < 1e-5
        gold.update({key + 'none': np.array([0]), key + 'pt': pt.numpy(), key + 'poly': poly.numpy(),
                     key + 'rec': rec.numpy(), key + 'probs': probs.numpy()})
        n_pts.append(pt.numel() // 2)
    print(f'page {i} (seed {page["seed"]}): points per prompt {n_pts}')
    if len(set(n_pts)) < 2 or 0 not in n_pts:
        return None
    return gold


if __name__ == '__main__':
    torch.set_grad_enabled(False)
    os.makedirs(GOLD, exist_ok=True)
    gen_prompts()
