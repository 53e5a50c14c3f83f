"""OmniParserB200: the reference's ``OmniParser.forward`` call site served by libalm_ocr.so.

Reference boundary (relative to /root/reference/OCR/OmniParser/):
  ``output = model(samples, seqs)``                      engine/val.py:35
  OmniParser.forward                                     model/omniparser.py:19-32
  token-id layout                                        utils/parser.py:16,88-105
  checkpoint layout ``torch.load(path)['model']``        utils/checkpointer.py:20,44-47
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from types import SimpleNamespace
from typing import List, Optional

import numpy as np
import torch

from . import _lib
from .nested_tensor import NestedTensor

DEFAULT_CHARS = ' !"#$%&\'()*+,-./0123456789:;<=>?@ABCDEFGHIJKLMNOPQRSTUVWXYZ[\\]^_`abcdefghijklmnopqrstuvwxyz{|}~'


# entity classes of the two KIE datasets the reference supports (model/transformer.py:49-61); class id =
# padding_index + 1 + position
CLASSES_CORD = ['menu.cnt', 'menu.discountprice', 'menu.etc', 'menu.itemsubtotal', 'menu.nm', 'menu.num', 'menu.price',
                'menu.sub.cnt', 'menu.sub.nm', 'menu.sub.price', 'menu.sub.unitprice', 'menu.unitprice', 'menu.vatyn',
                'sub_total.discount_price', 'sub_total.etc', 'sub_total.othersvc_price', 'sub_total.service_price',
                'sub_total.subtotal_price', 'sub_total.tax_price', 'total.cashprice', 'total.changeprice',
                'total.creditcardprice', 'total.emoneyprice', 'total.menuqty_cnt', 'total.menutype_cnt', 'total.total_etc',
                'total.total_price', 'void_menu.nm', 'void_menu.price']
CLASSES_SROIE = ['company', 'address', 'date', 'total']


@dataclass
class OmniVocab:
    """Same derivation as DefaultParser.parse_args (utils/parser.py:88-105)."""
    chars: str = DEFAULT_CHARS
    num_bins: int = 1000
    rec_length: int = 25
    pt_seq_length: int = 1024
    vie_categories: int = 0
    use_char_window_prompt: bool = True
    classes: Optional[List[str]] = None   # KIE entity names; default: SROIE for 4 categories, CORD for 29

    def __post_init__(self):
        if self.vie_categories and self.classes is None:
            self.classes = {4: CLASSES_SROIE, 29: CLASSES_CORD}.get(self.vie_categories)
        n_char = len(self.chars) + 1
        self.recog_pad_index = self.num_bins + n_char
        self.pt_eos_index = self.recog_pad_index + 1
        self.poly_eos_index = self.pt_eos_index + 1
        self.rec_eos_index = self.poly_eos_index + 1
        self.pt_sos_index = self.rec_eos_index + 1
        self.poly_sos_index = self.pt_sos_index + 1
        self.rec_sos_index = self.poly_sos_index + 1
        self.padding_index = self.rec_sos_index + 1
        self.num_classes = self.padding_index + 1 + self.vie_categories

    def pt_prompt(self) -> torch.Tensor:
        """engine/val.py:25-28"""
        if self.use_char_window_prompt:
            p = [0, 0, self.num_bins - 1, self.num_bins - 1, self.num_bins, self.num_bins + len(self.chars),
                 self.pt_sos_index]
        else:
            p = [0, 0, self.num_bins - 1, self.num_bins - 1, self.pt_sos_index]
        return torch.tensor([p], dtype=torch.long)

    def window_prompt(self, x0: int, y0: int, x1: int, y1: int, char_lo: int = 0,
                      char_hi: Optional[int] = None) -> torch.Tensor:
        """[1, n_prompt] pt prompt for a spatial window in bins and a character window in character indices (0 ..
        len(chars)), the prompt layout the model is trained with (dataset/collate_fn.py:46-115; the decoder is meant to
        emit the points with x0 < x <= x1, y0 < y <= y1 whose text lies in the character range).  The 5-token form
        (no character window) when ``use_char_window_prompt`` is off."""
        p = [int(x0), int(y0), int(x1), int(y1)]
        if self.use_char_window_prompt:
            hi = len(self.chars) if char_hi is None else int(char_hi)
            p += [self.num_bins + int(char_lo), self.num_bins + hi]
        return torch.tensor([p + [self.pt_sos_index]], dtype=torch.long)

    def grid_prompts(self, nx: int, ny: int, char_window=None) -> torch.Tensor:
        """[nx * ny, n_prompt] prompts of the nx x ny grid tiles of dataset/collate_fn.py:55-69 (same tile size
        min(int(num_bins / n), num_bins - 1), same clamped ends, i over x outer, j over y inner).  char_window:
        optional (char_lo, char_hi) shared by every tile."""
        nb = self.num_bins
        ix, iy = min(int(nb / nx), nb - 1), min(int(nb / ny), nb - 1)
        lo, hi = char_window if char_window is not None else (0, None)
        rows = []
        for i in range(nx):
            for j in range(ny):
                x0, y0 = i * ix, j * iy
                rows.append(self.window_prompt(x0, y0, min(x0 + ix, nb - 1), min(y0 + iy, nb - 1), lo, hi))
        return torch.cat(rows, 0)


def merge_window_outputs(outs):
    """One reference-shaped output per page from its per-window outputs (prompt order, None windows skipped): the
    instances of every window of the page, as ``postprocess`` / ``alm_post_omni_json`` take them; None when no window
    decoded a point."""
    live = [o for o in outs if o is not None]
    if not live:
        return None
    return ([torch.cat([o[0][0] for o in live], 1), torch.cat([o[0][1] for o in live], 1),
             torch.cat([o[0][2] for o in live], 1)], [torch.cat([o[1][0] for o in live], 0)])


class OmniParserB200:
    """Inference-only stand-in for the reference ``OmniParser`` module (``--tfm_pre_norm --use_fpn``)."""

    def __init__(self, state_dict, vocab: Optional[OmniVocab] = None, device: int = 0, stream: Optional[int] = None,
                 ctx: Optional[_lib.Context] = None, workspace_mb: Optional[int] = None,
                 share_from: Optional['OmniParserB200'] = None):
        """state_dict: the reference checkpoint ``torch.load(path)['model']``; or None together with
        ``share_from=other`` (another OmniParserB200 on the same GPU): this instance becomes a second execution
        context over the SAME device weights (alm_share_weights) -- one model, several batches in flight; or None
        when the weights were already put into ``ctx`` (multi-GPU start-up, dist.load_weights_broadcast).

        Device inputs: the context enqueues on its own stream; CUDA tensors handed to encode()/forward() are ordered
        after torch's current stream automatically (alm_stream_wait)."""
        self.vocab = vocab or OmniVocab()
        self.ctx = ctx or _lib.Context(device, stream)
        if workspace_mb:
            self.ctx.set_option('workspace_mb', workspace_mb)
        if share_from is not None:
            assert state_dict is None, 'pass either a state dict or share_from'
            self.ctx.share_weights(share_from.ctx)
        elif state_dict is not None:
            kind = _lib.MODEL_OMNI_KIE if self.vocab.vie_categories else _lib.MODEL_OMNI_SPOT
            self.ctx.load_state_dict(kind, state_dict)
        self.lib = self.ctx.lib

    # nn.Module look-alikes so reference drivers keep working
    def eval(self):
        return self

    def to(self, *_a, **_k):
        return self

    def __call__(self, samples, sequence=None):
        return self.forward(samples, sequence)

    # ---------------------------------------------------------------------------------------- stages
    def encode(self, tensors: torch.Tensor, mask: Optional[torch.Tensor] = None):
        """Swin-B -> FPN -> input_proj (model/omniparser.py:20-31).  Host or CUDA tensors."""
        assert tensors.dim() == 4 and tensors.shape[1] == 3 and tensors.dtype == torch.float32
        t = tensors.contiguous()
        B, _, H, W = t.shape
        mp = None
        if mask is not None:
            m8 = mask.to(torch.uint8).contiguous()
            if bool(m8.any()):
                self._keep_mask = m8
                mp = m8.data_ptr()
        self._keep_img = t
        self.ctx.wait_torch(t, mask)  # device inputs: order the context's stream after torch's current stream
        self.ctx.check(self.lib.alm_omni_encode(self.ctx.h, t.data_ptr(), mp, B, H, W))
        return self.memory_shape()

    def memory_shape(self):
        b, h, w = C.c_int(), C.c_int(), C.c_int()
        self.ctx.check(self.lib.alm_omni_memory_shape(self.ctx.h, C.byref(b), C.byref(h), C.byref(w)))
        return b.value, h.value, w.value

    def features(self, level: int) -> torch.Tensor:
        """LN'd Swin stage output, NCHW like ``features[level].tensors`` (backbone/joiner.py:10-18)."""
        B, mh, mw = self.memory_shape()
        H, W = self._keep_img.shape[2:]
        hs, ws = (H + 3) // 4, (W + 3) // 4
        for _ in range(level):
            hs, ws = (hs + 1) // 2, (ws + 1) // 2
        out = torch.empty(B, hs, ws, 128 << level, dtype=torch.float32)
        self.ctx.check(self.lib.alm_omni_get_feature(self.ctx.h, level, out.data_ptr(), out.numel()))
        return out.permute(0, 3, 1, 2)

    def memory(self, which: int = 0) -> torch.Tensor:
        """which 0: memory [B,M,512] (input_proj output, flattened); 1: sine position embedding."""
        B, mh, mw = self.memory_shape()
        out = torch.empty(B, mh * mw, 512, dtype=torch.float32)
        self.ctx.check(self.lib.alm_omni_get_memory(self.ctx.h, which, out.data_ptr(), out.numel()))
        return out

    def _cfg(self, max_instances):
        v = self.vocab
        return _lib.DecodeCfg(v.num_bins, v.pt_eos_index, v.poly_eos_index, v.rec_eos_index, v.pt_sos_index,
                              v.poly_sos_index, v.rec_sos_index, v.recog_pad_index, v.pt_seq_length, v.rec_length, 32,
                              v.vie_categories, max_instances)

    def decode(self, pt_prompt: Optional[torch.Tensor] = None):
        """Greedy pt / poly / rec decoding of every encoded image (model/transformer.py:234-286).
        Returns per-image reference-shaped outputs (None where no point was produced)."""
        v = self.vocab
        B, _, _ = self.memory_shape()
        prompt = (pt_prompt if pt_prompt is not None else v.pt_prompt()).reshape(-1).to(torch.long).cpu().contiguous()
        maxi = max(1, v.pt_seq_length // 2)
        n_inst = np.zeros(B, dtype=np.int32)
        pt = np.zeros((B, maxi, 2), dtype=np.int64)
        poly = np.zeros((B, maxi, 32), dtype=np.int64)
        rec = np.zeros((B, maxi, v.rec_length), dtype=np.int64)
        prob = np.zeros((B, maxi, v.rec_length), dtype=np.float32)
        cfg = self._cfg(maxi)
        self.ctx.check(self.lib.alm_omni_decode(self.ctx.h, prompt.data_ptr(), prompt.numel(), C.byref(cfg),
                                                n_inst.ctypes.data, pt.ctypes.data, poly.ctypes.data, rec.ctypes.data,
                                                prob.ctypes.data))
        outs = []
        for b in range(B):
            n = int(n_inst[b])
            if n == 0:
                outs.append(None)  # transformer.py:240-241
                continue
            outs.append(([torch.from_numpy(pt[b, :n].reshape(1, -1).copy()),
                          torch.from_numpy(poly[b, :n].reshape(1, -1).copy()),
                          torch.from_numpy(rec[b, :n][None].copy())],
                         [torch.from_numpy(prob[b, :n].copy())]))
        return outs

    def decode_points(self, pt_prompt: Optional[torch.Tensor] = None):
        """`decode_pt_seq` alone (model/transformer.py:102-141) for every encoded image: list of (tokens int64 [n],
        probs f32 [n]) -- the long single-sequence decode of structure heads (BASELINE config 5: 512 tokens)."""
        v = self.vocab
        B, _, _ = self.memory_shape()
        prompt = (pt_prompt if pt_prompt is not None else v.pt_prompt()).reshape(-1).to(torch.long).cpu().contiguous()
        P = v.pt_seq_length
        n_tok = np.zeros(B, dtype=np.int32)
        toks = np.zeros((B, P), dtype=np.int64)
        prob = np.zeros((B, P), dtype=np.float32)
        cfg = self._cfg(max(1, P // 2))
        self.ctx.check(self.lib.alm_omni_decode_points(self.ctx.h, prompt.data_ptr(), prompt.numel(), C.byref(cfg),
                                                       n_tok.ctypes.data, toks.ctypes.data, prob.ctypes.data))
        return [(torch.from_numpy(toks[b, :n_tok[b]].copy()), torch.from_numpy(prob[b, :n_tok[b]].copy())) for b in range(B)]

    def _prompts(self, prompts: torch.Tensor):
        """[R, L] (the same windows for every page) or [B, R, L] (per page) -> int64 [B, R, L] on the host."""
        B, _, _ = self.memory_shape()
        p = torch.as_tensor(prompts).to(torch.long).cpu()
        if p.dim() == 2:
            p = p.unsqueeze(0).expand(B, -1, -1)
        if p.dim() != 3 or p.shape[0] != B:
            raise ValueError(f'prompts must be [R, L] or [{B}, R, L], got {tuple(p.shape)}')
        return p.contiguous()

    def decode_prompted(self, prompts: torch.Tensor, merge: bool = False):
        """Greedy decoding of every encoded page under R window prompts each (``OmniVocab.window_prompt`` /
        ``grid_prompts``), over one encode.  prompts: [R, L] or [B, R, L].  Returns per page a list of R
        reference-shaped outputs (None where a window decoded no point), each what ``decode`` returns for that page
        under that prompt; with ``merge=True`` one output per page holding the instances of all its windows in prompt
        order (``merge_window_outputs``)."""
        v = self.vocab
        p = self._prompts(prompts)
        B, R, L = p.shape
        maxi = max(1, v.pt_seq_length // 2)
        n_inst = np.zeros((B, R), dtype=np.int32)
        pt = np.zeros((B, R, maxi, 2), dtype=np.int64)
        poly = np.zeros((B, R, maxi, 32), dtype=np.int64)
        rec = np.zeros((B, R, maxi, v.rec_length), dtype=np.int64)
        prob = np.zeros((B, R, maxi, v.rec_length), dtype=np.float32)
        cfg = self._cfg(maxi)
        self.ctx.check(self.lib.alm_omni_decode_prompted(self.ctx.h, p.data_ptr(), R, L, C.byref(cfg), n_inst.ctypes.data,
                                                         pt.ctypes.data, poly.ctypes.data, rec.ctypes.data,
                                                         prob.ctypes.data))
        pages = []
        for b in range(B):
            outs = []
            for r in range(R):
                n = int(n_inst[b, r])
                outs.append(None if n == 0 else
                            ([torch.from_numpy(pt[b, r, :n].reshape(1, -1).copy()),
                              torch.from_numpy(poly[b, r, :n].reshape(1, -1).copy()),
                              torch.from_numpy(rec[b, r, :n][None].copy())],
                             [torch.from_numpy(prob[b, r, :n].copy())]))
            pages.append(merge_window_outputs(outs) if merge else outs)
        return pages

    def decode_points_prompted(self, prompts: torch.Tensor):
        """`decode_pt_seq` alone under R window prompts per page: per page a list of R (tokens int64 [n], probs f32 [n])."""
        v = self.vocab
        p = self._prompts(prompts)
        B, R, L = p.shape
        P = v.pt_seq_length
        n_tok = np.zeros((B, R), dtype=np.int32)
        toks = np.zeros((B, R, P), dtype=np.int64)
        prob = np.zeros((B, R, P), dtype=np.float32)
        cfg = self._cfg(max(1, P // 2))
        self.ctx.check(self.lib.alm_omni_decode_points_prompted(self.ctx.h, p.data_ptr(), R, L, C.byref(cfg),
                                                                n_tok.ctypes.data, toks.ctypes.data, prob.ctypes.data))
        return [[(torch.from_numpy(toks[b, r, :n_tok[b, r]].copy()), torch.from_numpy(prob[b, r, :n_tok[b, r]].copy()))
                 for r in range(R)] for b in range(B)]

    def decode_kie(self, image_sizes, pt_prompt: Optional[torch.Tensor] = None):
        """KIE decoding of every encoded image (model/transformer.py:143-217): per image the reference's
        ``[(text, class_name, prob, [[x0,y0,x1,y1], ...]), ...]``.  image_sizes: (h, w) per image (seq[3])."""
        v = self.vocab
        assert v.vie_categories > 0 and v.classes is not None and len(v.classes) == v.vie_categories
        B, _, _ = self.memory_shape()
        prompt = (pt_prompt if pt_prompt is not None else v.pt_prompt()).reshape(-1).to(torch.long).cpu().contiguous()
        maxi, L, P = max(1, v.pt_seq_length // 2), v.rec_length, v.pt_seq_length
        n_tok = np.zeros(B, dtype=np.int32)
        toks = np.zeros((B, P), dtype=np.int64)
        tprob = np.zeros((B, P), dtype=np.float32)
        n_inst = np.zeros(B, dtype=np.int32)
        pos = np.zeros((B, maxi), dtype=np.int32)
        poly = np.zeros((B, maxi, 32), dtype=np.int64)
        rec = np.zeros((B, maxi, L), dtype=np.int64)
        prob = np.zeros((B, maxi, L), dtype=np.float32)
        cfg = self._cfg(maxi)
        self.ctx.check(self.lib.alm_omni_decode_kie(self.ctx.h, prompt.data_ptr(), prompt.numel(), C.byref(cfg),
                                                    n_tok.ctypes.data, toks.ctypes.data, tprob.ctypes.data,
                                                    n_inst.ctypes.data, pos.ctypes.data, poly.ctypes.data, rec.ctypes.data,
                                                    prob.ctypes.data))
        self.last_kie_raw = dict(n_tok=n_tok, tokens=toks, probs=tprob, n_inst=n_inst, inst_pos=pos, poly=poly, rec=rec)
        results = []
        for b in range(B):
            if n_tok[b] == 0:
                results.append(None)  # transformer.py:240-241
                continue
            h, w = [float(x) for x in image_sizes[b]]
            by_pos = {int(pos[b, n]): n for n in range(int(n_inst[b]))}
            out, words, rects = [], [], []
            i = 0
            while i < n_tok[b]:
                if i in by_pos:  # an (x, y) pair: polygon extent (:163-169) + transcription (:187-203)
                    n = by_pos[i]
                    pts = poly[b, n].reshape(-1, 2)
                    rects.append([w * float(pts[:, 0].min()) / v.num_bins, h * float(pts[:, 1].min()) / v.num_bins,
                                  w * float(pts[:, 0].max()) / v.num_bins, h * float(pts[:, 1].max()) / v.num_bins])
                    chars = []
                    for tok in rec[b, n].tolist():
                        if tok == v.recog_pad_index or tok == v.rec_eos_index:
                            break
                        if tok == v.recog_pad_index - 1:
                            continue
                        chars.append(v.chars[tok - v.num_bins])
                    words.append(''.join(chars))
                    i += 2
                elif toks[b, i] < v.num_bins:
                    i += 1
                else:  # class token closes the entity (:211-215)
                    out.append((' '.join(words), v.classes[int(toks[b, i]) - v.padding_index - 1], float(tprob[b, i]), rects))
                    words, rects = [], []
                    i += 1
            results.append(out)
        return results

    def kie_results_json(self, image_sizes) -> List[Optional[str]]:
        """The text `json.dump(output, f)` stores per image (engine/val.py:38-42) for the last `decode_kie` call, produced
        by the library's C++ entity walk (`alm_post_omni_kie_json`); None where nothing was decoded."""
        from . import postprocess
        raw, v = self.last_kie_raw, self.vocab
        args = SimpleNamespace(chars=v.chars, num_bins=v.num_bins, rec_length=v.rec_length,
                               recog_pad_index=v.recog_pad_index, rec_eos_index=v.rec_eos_index)
        out = []
        for b in range(len(raw['n_tok'])):
            nt, ni = int(raw['n_tok'][b]), int(raw['n_inst'][b])
            if nt == 0:
                out.append(None)
                continue
            out.append(postprocess.kie_json(raw['tokens'][b, :nt], raw['probs'][b, :nt], raw['inst_pos'][b, :ni],
                                            raw['poly'][b, :ni], raw['rec'][b, :ni], image_sizes[b], args, v.classes,
                                            v.padding_index + 1))
        return out

    def decode_logits(self, image: int, kind: str, seq: torch.Tensor) -> torch.Tensor:
        """Teacher-forced ``Transformer.decode`` (model/transformer.py:74-100): seq [n,len] -> [n,len,V]."""
        k = {'pt': 0, 'poly': 1, 'rec': 2}[kind]
        s = seq.to(torch.long).cpu().contiguous()
        V = self.lib.alm_omni_vocab(self.ctx.h)
        out = torch.empty(s.shape[0], s.shape[1], V, dtype=torch.float32)
        self.ctx.check(self.lib.alm_omni_decode_logits(self.ctx.h, image, k, s.data_ptr(), s.shape[0], s.shape[1],
                                                       out.data_ptr()))
        return out

    # ---------------------------------------------------------------------------------------- forward
    def forward(self, samples: NestedTensor, sequence=None):
        """Reference contract for batch 1 (engine/val.py:22,35): returns
        ``([pt[1,2N], poly[1,32N], rec[1,N,L]], [probs[N,L]])`` or ``None``.
        ``sequence`` = [pt_prompt, poly_prompt, rec_prompt, orig_size]; the poly/rec prompts are the fixed
        sos tokens (val.py:30-31) and are validated, the pt prompt is passed through."""
        outs = self.forward_batch(samples, sequence)
        if len(outs) != 1:
            raise ValueError('OmniParser.forward keeps the reference batch-1 contract; use forward_batch for B > 1')
        return outs[0]

    def forward_batch(self, samples: NestedTensor, sequence=None) -> List:
        pt_prompt = None
        if sequence is not None:
            pt_prompt = sequence[0]
            v = self.vocab
            if int(sequence[1].reshape(-1)[0]) != v.poly_sos_index or int(sequence[2].reshape(-1)[0]) != v.rec_sos_index:
                raise ValueError('poly/rec prompts must be the sos tokens of the vocabulary (engine/val.py:30-31)')
        self.encode(samples.tensors, samples.mask)
        if self.vocab.vie_categories:
            if sequence is None or len(sequence) < 4:
                raise ValueError('KIE needs the original image size as sequence[3] (engine/val.py:33)')
            size = sequence[3]
            sizes = [size] * samples.tensors.shape[0] if torch.as_tensor(size).dim() == 1 else size
            return self.decode_kie([tuple(float(x) for x in torch.as_tensor(sz).reshape(-1)[:2]) for sz in sizes], pt_prompt)
        return self.decode(pt_prompt)
