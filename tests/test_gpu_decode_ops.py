"""GPU: the kernels of the OmniParser decode step against plain fp64 references, through the unit-op C entry points.

Covered: the skinny exact-fp32 GEMV of the point loop (`gemv_rows`, every row class and K path, fused LayerNorm + query
position, the x / x2 column split), the cached self-attention step (wide and narrow kernels), the fused decoder
cross-attention (every `xattn_impl`, run boundaries, several images per launch, key-padding masks) and the greedy head
step (`head_select`).  The model-level tests check these kernels only end to end, where small per-kernel errors are
hidden behind four LayerNorm'd layers.

Bounds come from the arithmetic where one applies (u = 2^-24, the fp32 unit roundoff); each test records the largest
ratio error / bound it saw, printed at the end of the module (run with -s).  Out of scope: an image whose keys are all
masked -- the reference softmax is NaN there, and the key-padding mask of a real page always leaves a key live.
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

U = 2.0 ** -24
ALM_ERR_INVALID = -1
ALM_ERR_UNSUPPORTED = -5
NAN = float('nan')

_WORST = {}


def _record(name, ratio):
    _WORST[name] = max(_WORST.get(name, 0.0), float(ratio))


@pytest.fixture(scope='module')
def ctx():
    from advancedliteratemachinery_b200 import _lib
    assert torch.cuda.is_available(), 'GPU tests need a B200; there is no CPU fallback to test'
    c = _lib.Context(0)
    yield c
    print('\nlargest error / bound per check:', {k: f'{v:.3g}' for k, v in sorted(_WORST.items())})
    c.close()


def _ptr(t):
    return None if t is None else t.data_ptr()


def _ready():
    # the context enqueues on its own non-blocking stream: torch's pending fills / copies of the operands must be done
    torch.cuda.synchronize()


def _within(name, got, ref, bound):
    """|got - ref| <= bound elementwise (got finite); records the worst ratio."""
    got, ref, bound = got.double(), ref.double(), bound.double()
    assert torch.isfinite(got).all(), f'{name}: non-finite output'
    ratio = float(((got - ref).abs() / bound).max())
    _record(name, ratio)
    assert ratio <= 1.0, f'{name}: error is {ratio:.3g} x the bound'


# ============================================================================================ skinny GEMV
def _vocab_size():
    from advancedliteratemachinery_b200 import OmniVocab
    return OmniVocab().num_classes


def gemv(ctx, x, W, M, N, K, *, ldx=None, x2=None, n_split=1 << 30, bias=None, resid=None, ldr=0, out=None, ldo=None,
         act=0, ln=None, pos=None, pos_split=0, check=True):
    ldx = K if ldx is None else ldx
    ldo = N if ldo is None else ldo
    if out is None:
        out = torch.full((M, ldo), NAN, device='cuda')
    g, b = (None, None) if ln is None else ln
    _ready()
    rc = ctx.lib.alm_op_gemv(ctx.h, _ptr(x), _ptr(x2), n_split, ldx, _ptr(W), _ptr(bias), _ptr(resid), ldr, _ptr(out), ldo,
                             M, N, K, act, _ptr(g), _ptr(b), 1e-5, _ptr(pos), pos_split)
    if check:
        ctx.check(rc)
        return out
    return rc


def _act64(y, act):
    if act == 1:
        return 0.5 * y * (1.0 + torch.erf(y / math.sqrt(2.0)))
    return torch.relu(y) if act == 2 else y


def _gemv_bound(xa, Wa, ba, K, ref):
    """Recursive fp32 summation of K products: |err| <= K u (sum |x||w| + |b|); + 4u |out| for the bias / activation /
    residual roundings and erff (a few ulp).  Rigorous, not fitted: on a B200 the largest error is 0.03 of it."""
    s = xa.abs() @ Wa.abs().T
    if ba is not None:
        s = s + ba.abs()
    return K * U * s + 4 * U * ref.abs() + 1e-30


GEMV_M = [1, 7, 8, 9, 16, 17, 31, 32, 33, 63, 64]
GEMV_K = [64, 500, 512, 1024, 1536, 2048]


@pytest.mark.parametrize('K', GEMV_K)
@pytest.mark.parametrize('M', GEMV_M)
def test_gemv_matches_fp64(ctx, M, K):
    """Every row class (8/16/32/64 rows) x every K path (one chunk, 512-float chunks, 256-float chunks of the 64-row
    kernel; K = 1024 / 1536 leave trailing chunks empty).  Columns K..ldx-1 of x hold NaN and must not reach the output;
    output / residual strides wider than N; the output padding stays untouched."""
    Ns = [1, 3, 5, 512, 1536, 2048, _vocab_size()]
    i = GEMV_M.index(M) + GEMV_K.index(K)
    g = torch.Generator(device='cuda').manual_seed(1000 * M + K)
    for j, N in enumerate((Ns[i % len(Ns)], Ns[(i + 3) % len(Ns)])):
        act = (i + j) % 3
        with_bias, with_resid = (i + j) % 2 == 0, (i + j) % 4 < 2
        ldx = K + 4 * (1 + (i + j) % 3)
        ldo = N + (4 if j else 0)
        ldr = N + 8
        x = torch.randn(M, ldx, generator=g, device='cuda')
        x[:, K:] = NAN
        W = torch.randn(N, K, generator=g, device='cuda') / math.sqrt(K)
        b = torch.randn(N, generator=g, device='cuda') if with_bias else None
        r = torch.randn(M, ldr, generator=g, device='cuda') if with_resid else None
        out = gemv(ctx, x, W, M, N, K, ldx=ldx, bias=b, resid=r, ldr=ldr if with_resid else 0, ldo=ldo, act=act)
        xd, Wd = x[:, :K].double(), W.double()
        y = xd @ Wd.T + (b.double() if with_bias else 0)
        ref = _act64(y, act) + (r[:, :N].double() if with_resid else 0)
        _within('gemv', out[:, :N], ref, _gemv_bound(xd, Wd, None if b is None else b.double(), K, ref))
        assert torch.isnan(out[:, N:]).all(), 'gemv wrote the output padding'


@pytest.mark.parametrize('M', [1, 9, 33, 64])
@pytest.mark.parametrize('n_split', [0, 4, 1024, 1536])
def test_gemv_column_split_reads_x_then_x2(ctx, M, n_split):
    """Columns below n_split read x, the rest x2 (the packed q | k | v projection: q, k from LN(x) + pos, v from LN(x))."""
    K, N = 512, 1536
    g = torch.Generator(device='cuda').manual_seed(7 * M + n_split)
    x, x2 = torch.randn(M, K, generator=g, device='cuda'), torch.randn(M, K, generator=g, device='cuda') * 3
    W = torch.randn(N, K, generator=g, device='cuda') / math.sqrt(K)
    b = torch.randn(N, generator=g, device='cuda')
    out = gemv(ctx, x, W, M, N, K, x2=x2, n_split=n_split, bias=b)
    left = torch.arange(N, device='cuda')[None, :, None] < n_split
    xin = torch.where(left, x.double()[:, None, :], x2.double()[:, None, :])
    ref = torch.einsum('mnk,nk->mn', xin, W.double()) + b.double()
    bound = K * U * (torch.einsum('mnk,nk->mn', xin.abs(), W.double().abs()) + b.double().abs()) + 4 * U * ref.abs()
    _within('gemv_split', out, ref, bound)


def _ln64(x, g, b):
    xd = x.double()
    mu = xd.mean(-1, keepdim=True)
    rstd = 1.0 / torch.sqrt(((xd - mu) ** 2).mean(-1, keepdim=True) + 1e-5)
    y = (xd - mu) * rstd * g.double() + b.double()
    return y, (xd - mu).abs() * rstd * g.double().abs(), rstd * xd.abs().mean(-1, keepdim=True) * g.double().abs()


@pytest.mark.parametrize('M', [1, 9, 33, 64])
@pytest.mark.parametrize('pos_split', [0, 512, 1024, 1 << 30])
def test_gemv_fused_layernorm_and_position_match_fp64(ctx, M, pos_split):
    """Fused pre-LayerNorm (K = 512) and the query position added to the output columns below pos_split only."""
    K, N = 512, 1536
    gen = torch.Generator(device='cuda').manual_seed(M * 31 + (pos_split & 4095))
    x = torch.randn(M, K, generator=gen, device='cuda') * 2 + 0.5
    lg, lb = torch.randn(K, generator=gen, device='cuda'), torch.randn(K, generator=gen, device='cuda')
    pos = torch.randn(K, generator=gen, device='cuda')
    W = torch.randn(N, K, generator=gen, device='cuda') / math.sqrt(K)
    b = torch.randn(N, generator=gen, device='cuda')
    out = gemv(ctx, x, W, M, N, K, bias=b, ln=(lg, lb), pos=pos, pos_split=pos_split)
    y, ydev, ymean = _ln64(x, lg, lb)
    live = (torch.arange(N, device='cuda') < pos_split)[None, :, None]
    yin = torch.where(live, (y + pos.double())[:, None, :], y[:, None, :])
    Wd = W.double()
    ref = torch.einsum('mnk,nk->mn', yin, Wd) + b.double()
    # LayerNorm in fp32: the mean and variance are sums of 512 terms summed to a depth of ~21 (16 per lane + the warp
    # tree), rsqrtf is within 2 ulp: 32 u on each normalised value (relative to |x - mean| rstd |g| and to the error of
    # the mean, rstd mean|x| |g|) and u on |b| and on the position add
    ey = 32 * U * (ydev + ymean) + U * (lb.double().abs() + y.abs())
    ey = torch.where(live, ey[:, None, :] + U * yin.abs(), ey[:, None, :])
    bound = (K * U * (torch.einsum('mnk,nk->mn', yin.abs(), Wd.abs()) + b.double().abs())
             + torch.einsum('mnk,nk->mn', ey, Wd.abs()) + 4 * U * ref.abs())
    _within('gemv_ln', out, ref, bound)


@pytest.mark.parametrize('K', [512, 2048])
def test_gemv_rows_are_independent_of_the_row_class(ctx, K):
    """A row's result is bit-identical whatever the launch's row class (8/16/32/64) and the row's position in it: the
    kernel documents it, and a window decoded with others relies on it."""
    N = 1104
    g = torch.Generator(device='cuda').manual_seed(K)
    x = torch.randn(64, K, generator=g, device='cuda')
    W = torch.randn(N, K, generator=g, device='cuda') / math.sqrt(K)
    b = torch.randn(N, generator=g, device='cuda')
    full = gemv(ctx, x, W, 64, N, K, bias=b, act=2)
    for r0, M in ((0, 1), (0, 8), (3, 5), (8, 16), (40, 8), (17, 32), (5, 9), (33, 31), (0, 33), (1, 63)):
        part = gemv(ctx, x[r0:], W, M, N, K, bias=b, act=2)
        assert torch.equal(part, full[r0:r0 + M]), (r0, M)


def test_gemv_fused_layernorm_is_the_unfused_arithmetic(ctx):
    """LN + pos inside the GEMV == alm_op_layernorm (gather_ln_kernel<4>), then the fp32 + pos, then the plain GEMV with
    the column split: bit for bit, for every row class."""
    K, N = 512, 1536
    gen = torch.Generator(device='cuda').manual_seed(5)
    lg, lb = torch.randn(K, generator=gen, device='cuda'), torch.randn(K, generator=gen, device='cuda')
    pos = torch.randn(K, generator=gen, device='cuda')
    W = torch.randn(N, K, generator=gen, device='cuda') / math.sqrt(K)
    b = torch.randn(N, generator=gen, device='cuda')
    for M in (1, 8, 13, 32, 47, 64):
        x = torch.randn(M, K, generator=gen, device='cuda') * 3 - 1
        fused = gemv(ctx, x, W, M, N, K, bias=b, ln=(lg, lb), pos=pos, pos_split=1024)
        y = torch.empty_like(x)
        _ready()
        ctx.check(ctx.lib.alm_op_layernorm(ctx.h, x.data_ptr(), lg.data_ptr(), lb.data_ptr(), 1e-5, y.data_ptr(), M, K))
        yp = y + pos  # one fp32 add per element, as the kernel's
        unfused = gemv(ctx, yp, W, M, N, K, x2=y, n_split=1024, bias=b)
        assert torch.equal(fused, unfused), M


def test_gemv_rejects_unsupported_shapes_and_the_context_stays_usable(ctx):
    g = torch.Generator(device='cuda').manual_seed(3)
    x = torch.randn(65, 2052, generator=g, device='cuda')
    W = torch.randn(16, 2052, generator=g, device='cuda')
    lg, lb = torch.ones(2048, device='cuda'), torch.zeros(2048, device='cuda')
    for M, K, ln in ((65, 512, None), (8, 768, None), (8, 2052, None), (8, 1024, (lg, lb)), (8, 64, (lg, lb))):
        rc = gemv(ctx, x, W, M, 16, K, ln=ln, check=False)
        assert rc == ALM_ERR_INVALID, (M, K, ln is not None)
    x, W = x[:8, :512].contiguous(), W[:, :512].contiguous()
    out = gemv(ctx, x, W, 8, 16, 512)
    ref = x.double() @ W.double().T
    _within('gemv', out, ref, _gemv_bound(x.double(), W.double(), None, 512, ref))


# ============================================================================================ self-attention step
def _sattn_case(ctx, S, Tmax, ts, gen):
    """Random caches for S sequences; for each t: rows < t random, rows > t NaN, one step, checks."""
    K0 = torch.randn(S, Tmax, 512, generator=gen, device='cuda')
    V0 = torch.randn(S, Tmax, 512, generator=gen, device='cuda')
    for ld_qk, ld_v in ((1536, 1536), (1024, 512)):
        qk = torch.randn(S, ld_qk, generator=gen, device='cuda')
        vn = qk[:, 1024:] if ld_v == 1536 else torch.randn(S, ld_v, generator=gen, device='cuda')
        vbase = qk if ld_v == 1536 else vn
        voff = 1024 if ld_v == 1536 else 0
        for t in ts:
            rows = torch.arange(Tmax, device='cuda')[None, :, None]
            kc0 = torch.where(rows < t, K0, torch.full_like(K0, NAN))
            vc0 = torch.where(rows < t, V0, torch.full_like(V0, NAN))
            for wide in (1, 0):
                ctx.set_option('sattn_wide', wide)
                kc, vc = kc0.clone(), vc0.clone()
                out = torch.full((S, 512), NAN, device='cuda')
                hi = torch.full((S, 512), NAN, device='cuda', dtype=torch.bfloat16)
                lo = torch.full((S, 512), NAN, device='cuda', dtype=torch.bfloat16)
                _ready()
                ctx.check(ctx.lib.alm_op_self_attn_step(ctx.h, qk.data_ptr(), ld_qk, vbase.data_ptr() + 4 * voff, ld_v,
                                                        kc.data_ptr(), vc.data_ptr(), S, t, Tmax, out.data_ptr(),
                                                        hi.data_ptr(), lo.data_ptr()))
                # row t is the appended k / v, exactly; every other row is untouched
                assert torch.equal(kc[:, t], qk[:, 512:1024]) and torch.equal(vc[:, t], vbase[:, voff:voff + 512])
                keep = torch.ones(Tmax, dtype=torch.bool, device='cuda')
                keep[t] = False
                assert torch.equal(kc[:, keep].isnan(), kc0[:, keep].isnan())
                assert torch.equal(torch.nan_to_num(kc[:, keep]), torch.nan_to_num(kc0[:, keep]))
                assert torch.equal(torch.nan_to_num(vc[:, keep]), torch.nan_to_num(vc0[:, keep]))
                # fp64 reference over keys 0..t
                q = qk[:, :512].double().view(S, 8, 64) / 8
                kk = kc[:, :t + 1].double().view(S, t + 1, 8, 64)
                vv = vc[:, :t + 1].double().view(S, t + 1, 8, 64)
                s = torch.einsum('shd,sjhd->shj', q, kk)
                p = torch.softmax(s, -1)
                ref = torch.einsum('shj,sjhd->shd', p, vv).reshape(S, 512)
                pv = torch.einsum('shj,sjhd->shd', p, vv.abs()).reshape(S, 512)
                # scores: 64-term fp32 dot products (64 u relative to sum |q||k|), a probability within twice that; the
                # softmax sum and the P.V sum run over t + 1 terms (t + 1 u each); expf (2 ulp), the 8-group / warp
                # reductions and the division (24 u).  On a B200 the largest error is 0.04 of this bound.
                ds = 64 * U * torch.einsum('shd,sjhd->shj', q.abs(), kk.abs()).amax(-1)
                bound = (2 * ds.repeat_interleave(64, -1) + (2 * (t + 1) + 24) * U) * pv + 1e-30
                _within('self_attn', out, ref, bound)
                joined = hi.double() + lo.double()
                assert torch.equal(hi, out.to(torch.bfloat16)), 'hi is not the bf16 rounding of the fp32 output'
                assert float(((joined - out.double()).abs() / out.double().abs().clamp_min(1e-30)).max()) <= 2.0 ** -17
    ctx.set_option('sattn_wide', 1)


def _sattn_S():
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    edge = 4 * sms // 8  # the wide kernel runs while S * 8 <= 4 * SMs (and "sattn_wide" is on)
    return [1, 2, edge, edge + 1, 300]


@pytest.mark.parametrize('Tmax', [3, 28, 1024])
@pytest.mark.parametrize('si', range(5))
def test_self_attention_step_matches_fp64(ctx, si, Tmax):
    """Both kernels (wide: CTA per (sequence, head), 128-thread key stride and 8 position groups; narrow: warp per pair,
    32-lane stride) on both sides of the wide / narrow boundary, with positions that cross every loop stride."""
    S = _sattn_S()[si]
    ts = sorted({t for t in (0, 1, 31, 32, 33, 127, 128, 129, Tmax - 1) if t < Tmax})
    if S == 300 and Tmax == 1024:
        ts = [0, 33, 129, 1023]  # 1.2 GB of caches per step: the strides are crossed by the other shapes too
    _sattn_case(ctx, S, Tmax, ts, torch.Generator(device='cuda').manual_seed(S * 7 + Tmax))


# ============================================================================================ cross-attention
XA_M = [1, 37, 64, 65, 127, 128, 129, 255, 1000, 4096]
XA_NCAP = [1, 2, 16, 17, 64, 65, 70]
XA_MASKS = ['none', 'rand30', 'tail', 'block64', 'block128', 'last_only']


def _mask(kind, B, M, gen):
    """u8 [B, M], 1 = padding; different for every image, never all keys of an image."""
    if kind == 'none':
        return None
    k = torch.zeros(B, M, dtype=torch.uint8, device='cuda')
    for b in range(B):
        if kind == 'rand30':
            k[b] = (torch.rand(M, generator=gen, device='cuda') < 0.3).to(torch.uint8)
        elif kind == 'tail':  # page padding: a right-hand tail of a different length per image
            k[b, max(1, (M * (3 + b % 5)) // 8):] = 1
        elif kind in ('block64', 'block128'):
            w = 64 if kind == 'block64' else 128
            blk = (b % 2) if M > 2 * w else 0
            k[b, blk * w:(blk + 1) * w] = 1
        elif kind == 'last_only':
            k[b, :-1] = 1
        if bool(k[b].all()):
            k[b, -1] = 0
    return k


def _xattn_ref(q, k, v, kpm, img0, nimg, Ncap):
    qd = q.double().view(nimg, Ncap, 8, 64).permute(0, 2, 1, 3) / 8
    kd, vd = k[img0:img0 + nimg].double(), v[img0:img0 + nimg].double()
    s = qd @ kd.transpose(-1, -2)                                   # [nimg, 8, Ncap, M]
    if kpm is not None:
        s = s.masked_fill(kpm[img0:img0 + nimg].bool()[:, None, None, :], float('-inf'))
    p = torch.softmax(s, -1)
    ref = (p @ vd).permute(0, 2, 1, 3).reshape(nimg * Ncap, 512)
    pv = (p @ vd.abs()).permute(0, 2, 1, 3).reshape(nimg * Ncap, 512)
    qk_abs = (qd.abs() @ kd.abs().transpose(-1, -2)).amax(-1)       # [nimg, 8, Ncap]
    return ref, pv, qk_abs.permute(0, 2, 1).repeat_interleave(64, -1).reshape(nimg * Ncap, 512)


def xattn(ctx, q, k, v, kpm, B, img0, nimg, Ncap, M, dl, q_split):
    out = torch.full((nimg * Ncap, 512), NAN, device='cuda')
    _ready()
    rc = ctx.lib.alm_op_cross_attention(ctx.h, q.data_ptr(), k.data_ptr(), v.data_ptr(), _ptr(kpm), B, img0, nimg, Ncap, M,
                                        dl, q_split, out.data_ptr())
    return rc, out


# Empirical: the fraction of the worst-case bound below that the kernels are held to.  On a B200 (1000 W) the largest
# error of any kernel was 0.065 of the worst-case bound with split operands and 0.079 in single-pass bf16, i.e. 0.26 /
# 0.32 of the tolerance.  Reading the key-padding mask of the wrong image fails 53 cases, each by 12x the tolerance or
# more; taking the last key of every 128-key block as live fails 41 cases, all but two by 28x or more.
XA_FIT = 0.25


def _xattn_bound(nsplit, pv, qk_abs):
    # split-bf16 operands: a product of two 3-term splits is within 2^-16 of the fp32 product (the dropped lo*lo term and
    # the two representation errors), so a score is within 2^-16 sum |q/8||k|, a probability within twice that; ex2.approx,
    # the split of P and V and the fp32 sums stay below 2^-14 relative.  Single-pass bf16: 2^-8 per score, 2^-7 in P.V.
    if nsplit == 3:
        return XA_FIT * (2 * 2.0 ** -16 * qk_abs + 2.0 ** -14) * pv + 1e-30
    return XA_FIT * (2 * 2.0 ** -8 * qk_abs + 2.0 ** -7) * pv + 1e-30


def _xattn_run(ctx, M, Ncap, idx, impls, nsplit):
    gen = torch.Generator(device='cuda').manual_seed(M * 100 + Ncap)
    geos = [(1, 0, 1), (3, 1, 2), (32, 0, 32) if M <= 255 else (3, 1, 2)]
    ctx.set_option('nsplit', nsplit)
    try:
        for n, impl in enumerate(impls):
            j = idx + n
            B, img0, nimg = geos[j % 3]
            dl = (0, 11)[j % 2]
            mask = XA_MASKS[j % len(XA_MASKS)]
            q_split = (j // 2) % 2 if impl != 1 else 0
            ctx.set_option('xattn_impl', impl)
            ctx.set_option('xattn_wg', 1 + j % 2)
            ctx.set_option('xattn_ctas_per_sm', 1 + j % 3)
            q = torch.randn(nimg * Ncap, 512, generator=gen, device='cuda')
            k = torch.randn(B, 8, M, 64, generator=gen, device='cuda')
            v = torch.randn(B, 8, M, 64, generator=gen, device='cuda')
            kpm = _mask(mask, B, M, gen)
            if impl == 1 and Ncap > 1:
                rc, _ = xattn(ctx, q, k, v, kpm, B, img0, nimg, Ncap, M, dl, 0)
                assert rc == ALM_ERR_UNSUPPORTED
                continue
            rc, out = xattn(ctx, q, k, v, kpm, B, img0, nimg, Ncap, M, dl, q_split)
            ctx.check(rc)
            ref, pv, qk_abs = _xattn_ref(q, k, v, kpm, img0, nimg, Ncap)
            tag = f'xattn impl {impl} nsplit {nsplit}'
            try:
                _within(tag, out, ref, _xattn_bound(nsplit, pv, qk_abs))
            except AssertionError as e:
                raise AssertionError(f'{e} (B, img0, nimg = {B, img0, nimg}, dl {dl}, mask {mask}, q_split {q_split}, '
                                     f'wg {1 + j % 2}, ctas/SM {1 + j % 3})') from None
            # a second launch over the self-reset merge counters gives the same bits
            rc, again = xattn(ctx, q, k, v, kpm, B, img0, nimg, Ncap, M, dl, q_split)
            ctx.check(rc)
            assert torch.equal(out, again), tag
    finally:
        ctx.set_option('nsplit', 3)
        ctx.set_option('xattn_impl', 0)
        ctx.set_option('xattn_wg', 1)
        ctx.set_option('xattn_ctas_per_sm', 2)


@pytest.mark.parametrize('Ncap', XA_NCAP)
@pytest.mark.parametrize('M', XA_M)
def test_cross_attention_matches_fp64(ctx, M, Ncap):
    """Every kernel the decode loops can pick (mma.sync 16- / 64-query, its TMA variant, tcgen05 for > 16 queries, the
    fp32 single-query kernel) at key counts below / at / across the 64- and 128-key blocks, 1..32 images per launch at
    an image offset, the first and last decoder-layer slot, masked blocks, tails and lone live keys, and the run
    boundaries of 1..3 CTAs per SM.  Every slice the call must not read holds NaN."""
    idx = XA_M.index(M) * len(XA_NCAP) + XA_NCAP.index(Ncap)
    _xattn_run(ctx, M, Ncap, idx, (0, 1, 2, 3, 0, 3), 3)


@pytest.mark.parametrize('M,Ncap', [(37, 1), (129, 16), (255, 17), (1000, 70), (4096, 65)])
def test_cross_attention_single_pass_bf16_within_bf16_bound(ctx, M, Ncap):
    _xattn_run(ctx, M, Ncap, M + Ncap, (0, 2, 3), 1)


def test_cross_attention_rejects_bad_arguments(ctx):
    q = torch.randn(4, 512, device='cuda')
    k = v = torch.randn(2, 8, 40, 64, device='cuda')
    for args in ((2, 1, 2, 2, 40, 0, 0), (2, 0, 2, 2, 40, 12, 0), (2, 0, 1, 2, 40, 0, 2), (2, -1, 1, 2, 40, 0, 0)):
        rc, _ = xattn(ctx, q, k, v, None, *args)
        assert rc == ALM_ERR_INVALID, args
    rc, out = xattn(ctx, q, k, v, None, 2, 0, 2, 2, 40, 0, 0)
    ctx.check(rc)


# ============================================================================================ head select
def _cfg(vie=0):
    from advancedliteratemachinery_b200 import OmniVocab, _lib
    v = OmniVocab(vie_categories=vie)
    return v, _lib.DecodeCfg(v.num_bins, v.pt_eos_index, v.poly_eos_index, v.rec_eos_index, v.pt_sos_index,
                             v.poly_sos_index, v.rec_sos_index, v.recog_pad_index, 8, 25, 32, vie, 8)


def _candidates(v, V, phase, gen_index):
    j = np.arange(V)
    if phase == 0:
        mode = (0, 1, 3)[gen_index % 3] if v.vie_categories else gen_index % 2
    else:
        mode = phase
    if mode == 0:
        return (j < v.num_bins) | (j == v.pt_eos_index)
    if mode == 1:
        return j < v.num_bins
    if mode == 2:
        return ((j >= v.num_bins) & (j <= v.recog_pad_index)) | (j == v.rec_eos_index)
    return j >= V - v.vie_categories


def head_select(ctx, cfg, logits, S, V, nsoft, phase, t, npm1, tokens, probs, finished=None, ntok=None):
    import ctypes
    _ready()
    ctx.check(ctx.lib.alm_op_head_select(ctx.h, logits.data_ptr(), S, V, nsoft, phase, ctypes.byref(cfg), t, npm1,
                                         tokens.data_ptr(), tokens.shape[1], _ptr(probs),
                                         0 if probs is None else probs.shape[1], _ptr(finished), _ptr(ntok)))


@pytest.mark.parametrize('vie', [0, 4])
@pytest.mark.parametrize('phase', [0, 1, 2])
def test_head_select_matches_fp64(ctx, phase, vie):
    """Top-1 over the candidates of each mode (pt: coordinate or EOS on even steps, coordinate on odd ones, the class slot
    of the KIE 3-cycle; poly: bins; rec: chars + EOS), softmax over the first nsoft logits only, planted exact ties
    resolved to the lowest index, and nothing written but tokens[s, t+1] and probs[s, t - n_prompt_m1]."""
    v, cfg = _cfg(vie)
    V, S, npm1, T = v.num_classes, 37, 6, 40
    gen = torch.Generator().manual_seed(phase * 10 + vie)
    nsofts = [V] if phase == 0 else [V, V - vie] if vie else [V, V - 3]
    for t in (npm1, npm1 + 1, npm1 + 2, npm1 + 5):
        gi = t - npm1
        cand = _candidates(v, V, phase, gi)
        for nsoft in nsofts:
            x = torch.randn(S, V, generator=gen, dtype=torch.float64) * 4
            ok = np.flatnonzero(cand[:nsoft])
            # planted ties among the candidates: same thread (stride 256), other lanes / warps, lowest in a later thread
            for s in range(0, S, 3):
                picks = ok[[(7 * s) % len(ok), (7 * s + 256) % len(ok), (11 * s + 1) % len(ok), len(ok) - 1 - s % 5]]
                x[s, picks] = float(x[s, :nsoft].max()) + 1.5
            x[S - 1, :nsoft] = 0.25  # a row of equal logits
            x = x.float()
            tokens = torch.full((S, T), -7, dtype=torch.int32, device='cuda')
            probs = torch.full((S, T), NAN, device='cuda')
            head_select(ctx, cfg, x.cuda(), S, V, nsoft, phase, t, npm1, tokens, probs)
            xd = x.double().numpy()
            masked = np.where(cand[None, :nsoft], xd[:, :nsoft], -np.inf)
            best = masked.argmax(1)  # first maximum: the lowest index
            m = xd[:, :nsoft].max(1)
            pref = np.exp(masked[np.arange(S), best] - m) / np.exp(xd[:, :nsoft] - m[:, None]).sum(1)
            tk, pr = tokens.cpu().numpy(), probs.cpu().numpy()
            assert (tk[:, t + 1] == best).all(), (t, nsoft, np.flatnonzero(tk[:, t + 1] != best))
            # expf within 2 ulp of exp(rounded (x - max)), which is off by u |x - max|; sums of depth <= 18 (8 strided
            # terms, a warp tree, 8 warps) and one division: (32 + |best - max|) u relative (0.23 of it at most on a B200)
            gap = np.abs(masked[np.arange(S), best] - m)
            err = np.abs(pr[:, gi] - pref) / ((32 + gap) * U * pref)
            _record('head_select prob', err.max())
            assert err.max() <= 1.0
            others = np.ones((S, T), dtype=bool)
            others[:, t + 1] = False
            assert (tk[others] == -7).all(), 'tokens written outside column t+1'
            others = np.ones((S, T), dtype=bool)
            others[:, gi] = False
            assert np.isnan(pr[others]).all(), 'probs written outside column t - n_prompt_m1'


@pytest.mark.parametrize('vie', [0, 4])
def test_head_select_eos_bookkeeping(ctx, vie):
    """finished / ntok per sequence: an EOS pick sets finished and keeps ntok, any other pick sets ntok = gen_index + 1,
    and a finished row's state is never touched again."""
    v, cfg = _cfg(vie)
    V, S, npm1, T = v.num_classes, 24, 2, 20
    gen = torch.Generator().manual_seed(11 + vie)
    finished = torch.zeros(S, dtype=torch.int32, device='cuda')
    finished[::5] = 1
    ntok = torch.arange(S, dtype=torch.int32, device='cuda') + 100
    fin_h, ntok_h = finished.cpu().numpy().copy(), ntok.cpu().numpy().copy()
    tokens = torch.zeros(S, T, dtype=torch.int32, device='cuda')
    for t in range(npm1, npm1 + 9):
        gi = t - npm1
        x = torch.randn(S, V, generator=gen) * 2
        if gi >= 2:  # rows 0, 3, 6, ... pick EOS from the first step where EOS is a candidate after step 2
            x[::3, v.pt_eos_index] = 20.0
        head_select(ctx, cfg, x.cuda(), S, V, V, 0, t, npm1, tokens, None, finished, ntok)
        cand = _candidates(v, V, 0, gi)
        pick = np.where(cand[None], x.double().numpy(), -np.inf).argmax(1)
        assert (tokens[:, t + 1].cpu().numpy() == pick).all()
        for s in range(S):
            if fin_h[s]:
                continue
            if pick[s] == v.pt_eos_index:
                fin_h[s] = 1
            else:
                ntok_h[s] = gi + 1
        assert (finished.cpu().numpy() == fin_h).all(), t
        assert (ntok.cpu().numpy() == ntok_h).all(), t
    assert 0 < fin_h.sum() < S
