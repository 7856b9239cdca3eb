"""One CDAE training step's raw gradient arena against a float64 reference, element by element.

The weight-level tests run Adam (and RMSprop, Adagrad, Adamax), whose updates do not depend on the scale of the gradient:
a kernel that sent 2x dW', dropped the 1 / (1 - q) factor of dW or added only part of a split reduction passes them.
Here one step runs through drb_cdae_step_phases(PREP | GRADS), the arena (data gradient only: L2 is folded in by the
update kernel) is read segment by segment and compared with a float64 restatement of oracle.cdae's gradients, on every
GEMM path (FFMA, fp16 and tf32 split products), the loss-epilogue branches (BCE / MSE, batch-mean / per-user labels,
fast and general fp16 BCE forms, Keras' clip), db' from the ones feature or from the loss epilogue's column sums, the
batch-split dW'^T, the sampled-output step and the balanced scatter of dW / dV.

Error model.  Every gradient element is a reduction; its scale S is the float64 sum of the absolute values of its terms,
carried through the chain (an input known to a relative c carries c * S of error into the next reduction):
  S(a1) = |x||W| + |V_u| + |b|            S(h) = h + h(1-h) S(a1)         S(z) = S(h)|W'| + |b'|
  S(dz) = |dz| + |d dz/dp| p(1-p) S(z)    S(dW'^T) = S(h)^T |dz| + h^T S(dz)        S(db') = sum_b S(dz)
  S(dh) = S(dz)|W'|^T                     S(dz1) = S(dh) h(1-h) + |dh| S(h)         S(db), S(dV) = sums of S(dz1)
  S(dW) = |x|^T S(dz1)
and (a) |got - ref| <= C_ELEM * S for every element, (b) ||got - ref|| <= C_NORM ||ref|| per segment, (c) the
least-squares scale of got on ref is within C_SCALE of 1 per segment.  C_ELEM = 1e-4: the split products keep ~22 bits,
MUFU sigmoid / lg2 ~21 bits, fp32 sums run over at most 26,744 terms.  Two rounding effects are not relative to S and
enter as absolute terms, each stated where it is formed: the fp16 operands' smallest step (2^-25 of the scaled value) and
the fp32 quantisation of p (the kernel's p is known to two fp32 steps, P_ULPS, which near p = 1 is a large part of
1 - p and so of dz in the general BCE form; the fast fp16 form takes only its numerator from the rounded p, so there
the term is small).  The second is also propagated on its own, and (b) / (c) allow its norm.  On the
tensor-core paths (b) / (c) also allow the scale bias of the MMA's round-toward-zero accumulation (_tc_scale_bias).
"""
import ctypes as C

import numpy as np
import pytest

C_ELEM, C_NORM, C_SCALE = 1e-4, 1e-5, 1e-5
EPS = float(np.float32(1e-7))                           # Keras epsilon as the kernels hold it (fp32)
ONE_M = float(np.float32(1.0) - np.float32(1e-7))       # 1 - 1.19e-7: the fp32 upper clip bound
# fp32 steps of p the kernels' p = rcp(1 + ex2(-z log2 e)) may be off by, near p = 1 where it matters: rounding 1 + e
# to fp32 moves p by at most half a step, rcp.approx.ftz.f32 adds at most one ulp, and ex2.approx's relative error on
# e = 1 - p << 1 moves p by a negligible (1 - p) 2^-22.  The clip guarantee of the engineered case (2 steps from one_m)
# rests on the same count.
P_ULPS = 2
LOG2E = 1.4426950408889634
FAST_ARG_MAX = 22.0      # umma_loss.cu: a 16-row x 32-item chunk takes the fast form when every |z log2 e| <= 22
F16_STEP = 2.0 ** -25    # half the smallest fp16 step: representation error of a scaled fp16 hi/lo operand pair
H_SCALE, DZ_SCALE = 2.0 ** 15, 2.0 ** 14                # fp16 scaling of h and of dz / inv_count (kernels.h)
SEGMENTS = ('W2T', 'W', 'b', 'b2', 'V')

PHASE_PREP, PHASE_UPDATE, PHASE_GRADS = 1, 4, 2 | 8 | 16


# ------------------------------------------------------------------------------------------------ float64 reference
def _ulp32(p):
    import torch
    p32 = p.float()
    return (torch.nextafter(p32, torch.full_like(p32, 2.0)) - p32).double()


def fast_chunks(z):
    """Elements the fp16 BCE batch-mean epilogue computes in its fast form: full 16-row x 32-item chunks (rows and items
    aligned from 0, as the kernel's warps take them) whose every |z| log2 e <= 22.  A chunk within 0.05 of the threshold
    counts as general, the form with the larger quantisation term, so the kernel's own rounding of z cannot make this
    classification claim more accuracy than the kernel has."""
    import torch
    B, I = z.shape
    nb, ni = B // 16, I // 32
    fast = torch.zeros_like(z, dtype=torch.bool)
    if nb and ni:
        arg = (z[:nb * 16, :ni * 32].abs() * LOG2E).view(nb, 16, ni, 32).amax(dim=(1, 3))
        ok = arg <= FAST_ARG_MAX - 0.05
        fast[:nb * 16, :ni * 32] = ok[:, None, :, None].expand(nb, 16, ni, 32).reshape(nb * 16, ni * 32)
    return fast


def reference(w, uids, y, keep, q, loss, label_mode, mult=None, inv=None, fast_form=False):
    """oracle.cdae.CDAEOracle.grads without the regulariser, in float64, from the same fp32 weights.

    w: float64 tensors W [I,K], W_ [K,I], V [U,K], b [K], b_ [I]; uids [B] (long); y [B,I] labels of the batch rows;
    keep [B,I] corruption mask (ignored when q == 0, as the step ignores it); mult [B,I]: how often each (row, item) is
    scored (sampled outputs: positives once plus every draw; None = the dense layer, every item once); inv: loss
    normalisation (default 1 / (B I)); fast_form: the step runs the fp16 BCE batch-mean epilogue, whose fast chunks
    (fast_chunks) never form p (1 - p) from a rounded p.  Returns the reference arena segments, their scales S and
    quantisation terms A (both in units of C_ELEM, see the module docstring), the batch loss term and its error bound,
    and the intermediates.
    """
    import torch
    W, W_, V, b, b_ = (w[k] for k in ('W', 'W_', 'V', 'b', 'b_'))
    B, I = y.shape
    s = float(np.float32(1.0 / (1.0 - q)))              # the step's (float)(1 / (1 - q))
    x = y * s if q == 0 else y * keep * s
    M = torch.ones_like(y) if mult is None else mult
    inv = 1.0 / (B * I) if inv is None else inv
    floor_h = F16_STEP / H_SCALE / C_ELEM
    floor_w = F16_STEP * float(W_.abs().max()) * 2.0 ** -14 / C_ELEM   # W' scaled by alpha_w, max |W' alpha_w| >= 2^14
    floor_dz = F16_STEP * inv / DZ_SCALE / C_ELEM

    Vu = V[uids]
    a1 = x @ W + Vu + b
    S_a1 = x.abs() @ W.abs() + Vu.abs() + b.abs()
    h = torch.sigmoid(a1)
    hd = h * (1 - h)
    S_h = h + hd * S_a1 + floor_h
    z = h @ W_ + b_
    S_z = S_h @ (W_.abs() + floor_w) + b_.abs()
    p = torch.sigmoid(z)
    pd = p * (1 - p)
    t = y.mean(0, keepdim=True).expand_as(y) if label_mode == 'batch_mean' else y
    if loss == 'bce':
        p32 = p.float().double()                         # the clip and `inside` are decided on fp32 p, as the kernels do
        inside = ((p32 >= EPS) & (p32 <= ONE_M)).double()
        pc = p.clamp(EPS, ONE_M)
        da, db = pc + EPS, 1 - pc + EPS
        elem = -(t * torch.log(da) + (1 - t) * torch.log(db))
        g = (da - t * (da + db)) / (da * db) * inside     # dL/dp
        dg = (1 / db ** 2 + t * (1 + 2 * EPS) * (db - da) / (da * db) ** 2) * inside
        dz_p = (dg * pd + g * (1 - 2 * p)) * inv          # d dz / dp
    else:
        inside = torch.ones_like(p)
        elem = p * p - 2 * p * t + t if label_mode == 'batch_mean' else (p - t) ** 2   # (B,B,I) broadcast: y^2 == y
        g = 2 * (p - t)
        dz_p = (2 * pd + 2 * (p - t) * (1 - 2 * p)) * inv
    dz = M * g * pd * inv                                # dL/dz, summed over the times (row, item) is scored
    dp_q = P_ULPS * _ulp32(p)
    S_dz = M * ((g * pd * inv).abs() + dz_p.abs() * pd * S_z + floor_dz)
    # the general form computes dz from the rounded p throughout: d dz / dp.  The fast form (umma_loss.cu) forms
    # p (1 - p) / (da db) = e / t12 from e = exp(-z) and only its numerator da - t (1 + 2 eps) from the rounded p
    # (da = p + eps): d dz / d da = inv p (1 - p) / (da db)
    dz_q = dz_p.abs()
    fast = None
    if fast_form and loss == 'bce' and label_mode == 'batch_mean':
        fast = fast_chunks(z)
        dz_q = torch.where(fast, inv * pd / (da * db), dz_q)
    A_dz = M * dz_q * dp_q / C_ELEM
    loss_ref = float((M * elem).sum()) * inv
    loss_tol = inv * float((M * (C_ELEM * (elem.abs() + g.abs() * pd * S_z) + g.abs() * dp_q + 2.0 ** -21)).sum())

    dh = dz @ W_.t()
    dz1 = dh * hd
    ref = {'W2T': dz.t() @ h, 'b2': dz.sum(0), 'b': dz1.sum(0), 'W': x.t() @ dz1,
           'V': torch.zeros_like(V).index_add_(0, uids, dz1)}

    def chain(S_h, S_dz, fw):          # scales of the arena segments from those of h and dz (fw: W' operand floor)
        S_dh = S_dz @ W_.abs().t() + dz.abs().sum(1, keepdim=True) * fw
        S_dz1 = S_dh * hd + dh.abs() * S_h
        return {'W2T': S_dz.t() @ h + dz.abs().t() @ S_h, 'b2': S_dz.sum(0),
                'b': S_dz1.sum(0), 'W': x.abs().t() @ S_dz1, 'V': torch.zeros_like(V).index_add_(0, uids, S_dz1)}
    S = chain(S_h, S_dz, floor_w)
    A = chain(torch.zeros_like(S_h), A_dz, 0.0)
    return {'ref': ref, 'S': {k: S[k] + A[k] for k in S}, 'A': A, 'loss': loss_ref, 'loss_tol': loss_tol,
            'h': h, 'dz': dz, 'x': x, 'dz1': dz1, 'p': p, 'z': z, 'fast': fast, 't': t, 'M': M, 'inv': inv}


def check_segment(name, got, ref, S, A, bias=0.0):
    """(a), (b), (c) of the module docstring for one segment; returns the observed ratios to their bounds (<= 1 passes)
    and raises AssertionError with them otherwise.  Elements whose scale is 0 (no term reaches them) must be exactly 0.
    bias: the relative shrinkage toward zero the tensor-core accumulation may add (_tc_scale_bias), allowed in (b), (c)."""
    got, ref, S, A = (t.double().flatten() for t in (got, ref, S, A))
    err = (got - ref).abs()
    zero = S == 0
    assert bool((got[zero] == 0).all()), f'{name}: {int((got[zero] != 0).sum())} elements without any term are not 0'
    ra = float((err[~zero] / (C_ELEM * S[~zero])).max()) if bool((~zero).any()) else 0.0
    nref = float(ref.norm())
    if nref == 0:
        return {'a': ra, 'b': 0.0, 'c': 0.0}
    nA = C_ELEM * float(A.norm())
    rb = float(err.norm()) / ((C_NORM + bias) * nref + nA)
    alpha = float(got @ ref) / nref ** 2
    rc = abs(alpha - 1) / (C_SCALE + bias + nA / nref)
    out = {'a': ra, 'b': rb, 'c': rc}
    assert ra <= 1 and rb <= 1 and rc <= 1, (
        f'{name}: worst |got-ref| / (c_elem S) = {ra:.3g}, ||got-ref|| / bound = {rb:.3g} '
        f'(relative {float(err.norm()) / nref:.3g}), |alpha-1| / bound = {rc:.3g} (alpha - 1 = {alpha - 1:.3g})')
    return out


# ------------------------------------------------------------------------------------------------ CPU-only tests
def _tiny_inputs(loss, label_mode, sampled, seed=0):
    import torch
    g = torch.Generator().manual_seed(seed)
    U, I, K, B = 7, 40, 6, 9
    W = (torch.rand(I, K, generator=g, dtype=torch.float64) - 0.5).float().double()
    W_ = (torch.rand(K, I, generator=g, dtype=torch.float64) - 0.5).float().double()
    V = (torch.rand(U, K, generator=g, dtype=torch.float64) - 0.5).float().double()
    b = torch.tensor([12.0, -12.0, 0.3, -0.2, 1.0, 0.0], dtype=torch.float64)
    # extreme logits: fast-form and general-form bands inside the clip, and clipped items on both sides
    bands = [0.0, 10.0, -10.0, 15.0, -15.0, -15.5, -16.0, 15.3, -16.5, 18.0, 30.0, -30.0, 100.0, -100.0]
    b_ = torch.tensor([bands[i % len(bands)] if i % 3 else 0.3 * (i % 5) for i in range(I)], dtype=torch.float64)
    W_[:, b_.abs() >= 10] *= 1e-3
    uids = torch.tensor([0, 3, 3, 6, 1, 2, 5, 3, 4])
    y = (torch.rand(B, I, generator=g, dtype=torch.float64) < 0.3).double()
    y[4] = 0                                             # a row without positives
    keep = (torch.rand(B, I, generator=g, dtype=torch.float64) < 0.8).double()
    mult, inv = None, None
    if sampled:
        mult = y.clone()
        draws = torch.randint(0, I, (B, 12), generator=g)
        mult.scatter_add_(1, draws, torch.ones_like(draws, dtype=torch.float64))
        inv = 1.0 / (B * 12)
    return {'W': W, 'W_': W_, 'V': V, 'b': b, 'b_': b_}, uids, y, keep, mult, inv


@pytest.mark.parametrize('loss,label_mode,sampled', [('bce', 'batch_mean', False), ('bce', 'per_user', False),
                                                     ('mse', 'batch_mean', False), ('mse', 'per_user', False),
                                                     ('bce', 'per_user', True), ('mse', 'per_user', True)])
def test_reference_matches_autograd(loss, label_mode, sampled):
    """The float64 reference against torch.autograd of the Keras loss (torch's clamp passes the gradient on the closed
    interval, as Keras' clip does), at a tiny shape with logits on both sides of the clip."""
    import torch
    w, uids, y, keep, mult, inv = _tiny_inputs(loss, label_mode, sampled)
    q = 0.2
    r = reference(w, uids, y, keep, q, loss, label_mode, mult, inv)
    p32 = r['p'].float().double()
    assert bool(((p32 - EPS).abs() > 0.1 * EPS).all()) and bool(((p32 - ONE_M).abs() >= 2 * 2.0 ** -24).all())
    assert bool((p32 > ONE_M).any()) and bool((p32 < EPS).any())          # both clips are exercised
    v = {k: t.clone().requires_grad_(True) for k, t in w.items()}
    B, I = y.shape
    x = y * keep * float(np.float32(1 / (1 - q)))
    h = torch.sigmoid(x @ v['W'] + v['V'][uids] + v['b'])
    p = torch.sigmoid(h @ v['W_'] + v['b_'])
    t = y.mean(0, keepdim=True) if label_mode == 'batch_mean' else y
    if loss == 'bce':
        pc = torch.clamp(p, EPS, ONE_M)
        elem = -(t * torch.log(pc + EPS) + (1 - t) * torch.log(1 - pc + EPS))
    else:
        elem = p * p - 2 * p * t + t if label_mode == 'batch_mean' else (p - t) ** 2
    M = torch.ones_like(y) if mult is None else mult
    L = (M * elem).sum() * (1.0 / (B * I) if inv is None else inv)
    L.backward()
    want = {'W2T': v['W_'].grad.t(), 'W': v['W'].grad, 'V': v['V'].grad, 'b': v['b'].grad, 'b2': v['b_'].grad}
    for k in SEGMENTS:
        scale = float(want[k].abs().max())
        assert scale > 0 and float((r['ref'][k] - want[k]).abs().max()) <= 1e-12 * scale, k
    assert abs(r['loss'] - L.item()) <= 1e-12 * abs(L.item())


def test_checker_rejects_scale_outlier_dropped_row_and_missing_plane():
    """check_segment passes the reference itself and fails each error the kernels could make without Adam noticing."""
    import torch
    w, uids, y, keep, mult, inv = _tiny_inputs('bce', 'batch_mean', False, seed=1)
    r = reference(w, uids, y, keep, 0.2, 'bce', 'batch_mean')
    for k in SEGMENTS:
        assert check_segment(k, r['ref'][k], r['ref'][k], r['S'][k], r['A'][k])['a'] == 0.0
        with pytest.raises(AssertionError):
            check_segment(k, r['ref'][k] * (1 + 1e-3), r['ref'][k], r['S'][k], r['A'][k])
        bad = r['ref'][k].clone().flatten()
        j = int(torch.argmax(r['S'][k].flatten()))
        bad[j] += 10 * C_ELEM * r['S'][k].flatten()[j]
        with pytest.raises(AssertionError):
            check_segment(k, bad.view_as(r['ref'][k]), r['ref'][k], r['S'][k], r['A'][k])
    h, dz, x, dz1 = r['h'], r['dz'], r['x'], r['dz1']
    B = h.shape[0]
    for name, ref, full, partial in (
            ('W2T', r['ref']['W2T'], lambda rows: dz[rows].t() @ h[rows], None),
            ('W', r['ref']['W'], lambda rows: x[rows].t() @ dz1[rows], None),
            ('b2', r['ref']['b2'], lambda rows: dz[rows].sum(0), None)):
        assert torch.allclose(full(slice(0, B)), ref, rtol=1e-12, atol=0)
        dropped = full(torch.tensor([j for j in range(B) if j != 1]))      # one batch row's contribution missing
        with pytest.raises(AssertionError):
            check_segment(name, dropped, ref, r['S'][name], r['A'][name])
        with pytest.raises(AssertionError):                               # one of two split planes missing
            check_segment(name, full(slice(0, B // 2)), ref, r['S'][name], r['A'][name])


def test_checker_rejects_errors_next_to_the_upper_clip():
    """Near p = 1 the rounding allowance is largest, so these are the errors easiest to hide: on the engineered logits,
    a fast-form dz that drops eps from db = 1 - p + eps (a factor 1.33 at z = 15) and a 1.2x error on the general-form
    items between the fast-form threshold and the clip must both fail, in dW'^T and in db'."""
    import torch
    U, I, K, B = 20, 256, 16, 32
    w = {k: torch.as_tensor(v).double() for k, v in _weights(U, I, K, seed=11, engineered=True).items()}
    g = torch.Generator().manual_seed(3)
    uids = torch.randint(0, U, (B,), generator=g)
    y = (torch.rand(B, I, generator=g, dtype=torch.float64) < 0.3).double()
    keep = (torch.rand(B, I, generator=g, dtype=torch.float64) < 0.8).double()
    r = reference(w, uids, y, keep, 0.2, 'bce', 'batch_mean', fast_form=True)
    z, p, fast, t, h, inv = r['z'], r['p'], r['fast'], r['t'], r['h'], r['inv']
    p32 = p.float().double()
    assert bool(((p32 - ONE_M).abs() >= 2 * 2.0 ** -24).all())
    fast_hi = fast & (z > 14.5)
    general_hi = ~fast & (z > 15.25) & (p32 <= ONE_M)
    assert bool(fast_hi.any()) and bool(general_hi.any())
    da = p + EPS
    no_eps = inv * (da - t * (da + 1 - p)) / (da * (1 - p)) * p * (1 - p)
    for bad in (torch.where(fast_hi, no_eps, r['dz']), torch.where(general_hi, 1.2 * r['dz'], r['dz'])):
        for name, got in (('W2T', bad.t() @ h), ('b2', bad.sum(0))):
            check_segment(name, r['ref'][name], r['ref'][name], r['S'][name], r['A'][name])
            with pytest.raises(AssertionError):
                check_segment(name, got, r['ref'][name], r['S'][name], r['A'][name])


# ------------------------------------------------------------------------------------------------ GPU harness
def _dataset(U, I, mean_deg, heavy_deg, seed):
    """Unique (user, item) pairs with ratings 2..5, except user 0, whose ratings are all 1: below the positive threshold
    1.5 the models use, so it has no positives.  User 1 has heavy_deg positives (several 256-entry scatter pieces)."""
    import drecpy_b200 as drb
    rng = np.random.default_rng(seed)
    deg = rng.integers(1, 2 * mean_deg, U)
    deg[1] = heavy_deg
    u = np.repeat(np.arange(U), deg)
    i = np.concatenate([rng.choice(I, d, replace=False) for d in deg])
    missing = np.setdiff1d(np.arange(I), i)
    u = np.concatenate([u, rng.integers(2, U, len(missing))])
    i = np.concatenate([i, missing])
    v = rng.integers(2, 6, len(u)).astype(np.float64)
    v[u == 0] = 1
    ds = drb.InteractionData(u + 1, i + 1, v)
    ds.assign_internal_ids()
    return ds


def _weights(U, I, K, seed, engineered=False):
    rng = np.random.default_rng(seed)

    def glorot(shape, fi, fo):
        lim = np.sqrt(6.0 / (fi + fo))
        return rng.uniform(-lim, lim, shape).astype(np.float32)
    w = {'W': glorot((I, K), I, K), 'W_': glorot((K, I), K, I), 'V': glorot((U, K), U, K),
         'b': glorot((K,), K, K), 'b_': glorot((I,), I, I)}
    if engineered:
        w['b_'], shrink = _logit_bands(I)
        w['W_'][:, shrink] *= 1e-3
        w['W_'] *= (2.0 ** rng.uniform(-14, 1, (K, 1))).astype(np.float32)   # hidden units over 15 binary orders
        w['b'][:6] = [12.0, -12.0, 12.5, -11.5, 12.0, -12.0]                   # saturated hidden units
    return w


FAST = [0.0, 10.0, -10.0, 15.0, -15.0]                  # fast fp16 BCE form (|z| < 15.25)
GENERAL = [-15.5, -16.0, 15.3]                          # general form, inside the clip
CLIPPED = [-16.5, 18.0, 30.0, -30.0, 100.0, -100.0]     # outside the clip: zero gradient, clipped loss term
# (+17 rounds to one fp32 step above the upper clip bound: a one-step difference in the kernel's sigmoid could move it
# inside, so +18 -- two steps -- stands for it)


def _logit_bands(I):
    """b' per item, by 32-item block (one epilogue warp's items): ordinary blocks, blocks of fast-form bands, ordinary
    blocks with one extreme item (the whole block takes the general form), and blocks of extreme items only."""
    rng = np.random.default_rng(4)
    lim = np.sqrt(6.0 / (2 * I))
    b_ = rng.uniform(-lim, lim, I).astype(np.float32)
    shrink = np.zeros(I, bool)
    extreme = GENERAL + CLIPPED
    for blk in range(I // 32):
        items = np.arange(32 * blk, 32 * blk + 32)
        kind = blk % 4
        if kind == 1:
            b_[items] = [FAST[j % len(FAST)] for j in range(32)]
            shrink[items] = True
        elif kind == 2:
            j = items[(7 * blk) % 32]
            b_[j] = extreme[blk % len(extreme)]
            shrink[j] = True
        elif kind == 3:
            b_[items] = [(FAST + extreme)[(j + blk) % (len(FAST) + len(extreme))] for j in range(32)]
            shrink[items] = True
    return b_, shrink


def _model(ds, K, B, w, gemm, loss, label_mode, q, output='dense', neg_groups=2, neg_per_group=24):
    import drecpy_b200 as drb
    m = drb.CDAE(hidden_factors=K, corruption_level=q, loss=loss, seed=10, verbose=False, rng_mode='philox',
                 label_mode=label_mode, gemm=gemm, output=output, neg_groups=neg_groups, neg_per_group=neg_per_group,
                 interaction_threshold=1.5)
    m.fit(ds, epochs=0, batch_size=B, learning_rate=1e-3, reg_rate=0.1, init_weights=w)
    return m


def _batch(m, B, seed):
    """Batch rows: the user without positives, the heavy user, one user listed twice, then uniform draws (with
    replacement, as the sampler draws them)."""
    deg = np.diff(m._h_indptr)
    rng = np.random.default_rng(seed)
    empty, heavy = int(np.flatnonzero(deg == 0)[0]), int(deg.argmax())
    special = [heavy] if B == 1 else [empty, heavy, 5, 5]
    uids = np.concatenate([special, rng.integers(0, m.n_users, max(0, B - len(special)))]).astype(np.int32)[:B]
    return uids


def _run_step(m, uids, keep_np, reg_rate=0.1):
    """PREP | GRADS, a copy of the arena, then UPDATE; returns (arena copy, [loss, batch term])."""
    import torch
    from drecpy_b200 import _lib
    lib = _lib.load()
    deg = np.diff(m._h_indptr)
    off = np.concatenate([[0], np.cumsum(deg[uids])]).astype(np.int32)
    d_u = torch.as_tensor(uids, device=m._dev)
    d_o = torch.as_tensor(off, device=m._dev)
    d_k = torch.as_tensor(np.concatenate([keep_np, [1]]).astype(np.uint8), device=m._dev)   # >= 1 byte
    loss = torch.zeros(2, dtype=torch.float32, device=m._dev)
    m._step = 1
    a = m.step_args(reg_rate)
    args = (m._native, _lib.t_ptr(d_u), _lib.t_ptr(d_o), _lib.t_ptr(d_k), len(uids), C.byref(a), _lib.t_ptr(loss))
    _lib.check(lib.drb_cdae_step_phases(*args, PHASE_PREP | PHASE_GRADS))
    grads = m._grads.clone()
    _lib.check(lib.drb_cdae_step_phases(*args, PHASE_UPDATE))
    torch.cuda.synchronize()
    return grads, loss.cpu().numpy()


def _segments(m, grads):
    L, I, U = m._L, m.n_items, m.n_users
    return {'W2T': grads[L.off_w2t:L.off_w2t + I * L.ld].view(I, L.ld), 'W': grads[L.off_w:L.off_w + I * L.ld].view(I, L.ld),
            'b': grads[L.off_b:L.off_b + L.ld], 'b2': grads[L.off_b2:L.off_v], 'V': grads[L.off_v:L.total].view(U, L.ld)}


def _tc_scale_bias(m, B):
    """Per segment, the scale bias the tensor-core paths may show.  The MMA's fp32 accumulation rounds toward zero (the
    aligned addends are truncated, as measured on earlier NVIDIA tensor cores by Fasi, Higham, Mikaitis and Pranesh,
    2021): each of the three split products of a k-step (16 fp16 or 8 tf32 elements) can drop up to one fp32 unit in the
    last place of the accumulator, always toward zero.  A reduction of n k-steps in one accumulator therefore comes out
    smaller by up to 3 n 2^-23 of its value -- a uniform scale, not noise: at the production shape dW'^T showed
    alpha - 1 = -1.5e-5 over 128 k-steps (B = 4096 in two planes), while the element-wise ratio stayed at 0.06 and the
    FFMA path shows no such bias.  n follows the split choices of api.cu (the model does not report them): dW'^T (and
    db' through the ones feature) over the batch in s2 planes (api.cu, s2), dh (and so dz1 -> dW, db, dV) over the items
    in `splits` parts (drb_cdae_create).  If those choices change to fewer parts, the kernels' bias outgrows this
    allowance and the test fails; if to more, the allowance is larger than needed but never above MAX_TC_BIAS, so a
    1e-3 scale error still fails.  At hidden = 256 db' is an fp32 column sum in the loss epilogue: no MMA, no bias."""
    import torch
    if m.output == 'sampled' or m.gemm == 'ffma':
        return dict.fromkeys(SEGMENTS, 0.0)
    k = 16 if _runs_fp16(m) else 8
    I, sm = m.n_items, torch.cuda.get_device_properties(m._dev).multi_processor_count
    mt2 = -(-I // 128)
    s2 = max(1, min(16, -(-2 * sm // mt2), B // 512)) if B >= 1024 else 1
    splits = max(1, min(32, (2 * sm) // -(-m._max_batch // 128), I // 256))
    steps_w, steps_h = -(-B // s2) // k + 4, -(-I // splits) // k + 4      # + 4: k-blocks rounded up per plane / part
    bw, bh = 3 * steps_w * 2.0 ** -23, 3 * steps_h * 2.0 ** -23
    assert max(bw, bh) <= MAX_TC_BIAS, (bw, bh)
    return {'W2T': bw, 'b2': 0.0 if m.hidden_factors == 256 else bw, 'W': bh, 'b': bh, 'V': bh}


MAX_TC_BIAS = 1e-4
# environment overrides of the step's tensor-core configuration (tuning / profiling only): with any of them set the
# split counts and operand forms above are not the ones the step runs
_TC_OVERRIDES = ('DRB_GEMM_SPLIT', 'DRB_DW_SPLITS', 'DRB_DH_SPLITS')


def _runs_fp16(m):
    """The step runs the fp16 split products (the default tensor-core path): dense outputs, gemm 'auto' or 'tcgen05'."""
    import os
    assert not any(os.environ.get(v) for v in _TC_OVERRIDES), f'unset {_TC_OVERRIDES} to run these tests'
    return m.output == 'dense' and m.gemm in ('auto', 'tcgen05')


def _check_step(m, w, uids, keep_np, q, reg_rate=0.1, engineered=False):
    """Runs one step and checks the arena against the reference; returns the worst ratios per check."""
    import torch
    from oracle.cdae import sampled_negatives
    dev = m._dev
    grads, loss = _run_step(m, uids, keep_np, reg_rate)
    K, I, B = m.hidden_factors, m.n_items, len(uids)
    indptr, indices = m._h_indptr, m._h_indices
    deg = np.diff(indptr)
    rows = np.repeat(np.arange(B), deg[uids])
    cols = np.concatenate([indices[indptr[u]:indptr[u + 1]] for u in uids]) if deg[uids].sum() else np.zeros(0, int)
    r_t, c_t = torch.as_tensor(rows, device=dev), torch.as_tensor(cols, dtype=torch.long, device=dev)
    y = torch.zeros(B, I, dtype=torch.float64, device=dev)
    y[r_t, c_t] = 1
    keep = torch.ones_like(y)
    keep[r_t, c_t] = torch.as_tensor(keep_np, dtype=torch.float64, device=dev)   # keep_off order = CSR order per row
    mult, inv = None, None
    if m.output == 'sampled':
        mult = y.clone()
        for bi in range(B):
            neg = sampled_negatives(I, m.neg_groups, m.neg_per_group, bi, 1, m._mask_seed)
            mult[bi].index_add_(0, torch.as_tensor(neg, device=dev), torch.ones(len(neg), dtype=torch.float64, device=dev))
        inv = 1.0 / (B * m.neg_groups * m.neg_per_group)
    w64 = {k: torch.as_tensor(v, device=dev).double() for k, v in w.items()}
    u_t = torch.as_tensor(uids.astype(np.int64), device=dev)
    r = reference(w64, u_t, y, keep, q, m.loss, m.label_mode, mult, inv, fast_form=_runs_fp16(m))
    if engineered:     # the data guarantee that keeps a one-step difference in the kernel's p from flipping the clip
        p32 = r['p'].float().double()
        assert bool(((p32 - EPS).abs() >= 0.1 * EPS).all()), 'a logit sits too close to the lower clip'
        assert bool(((p32 - ONE_M).abs() >= 2 * 2.0 ** -24).all()), 'a logit sits too close to the upper clip'
        z, fast = r['z'], r['fast']
        assert bool((p32 > ONE_M).any() & (p32 < EPS).any())
        # fast chunks next to the threshold and general-form items inside the clip on the upper side
        assert bool((fast & (z > 14.5)).any()) and bool((~fast & (z > 15.25) & (p32 <= ONE_M)).any())
    seg = _segments(m, grads)
    bias = _tc_scale_bias(m, B)
    out = {}
    for name in SEGMENTS:
        got = seg[name]
        n = I if name in ('b2', 'W2T', 'W') else (m.n_users if name == 'V' else K)
        if name in ('b', 'b2'):
            assert float(got[n:].abs().max()) == 0 if got.numel() > n else True, f'{name}: pad entries are not 0'
            got = got[:n]
        else:
            assert float(got[:, K:].abs().max()) == 0 if got.shape[1] > K else True, f'{name}: pad columns are not 0'
            got = got[:, :K]
        ref, S, A = r['ref'][name], r['S'][name], r['A'][name]
        if name == 'V':                # rows of users outside the batch: exactly 0; then the batch's distinct users
            inb = torch.zeros(m.n_users, dtype=torch.bool, device=dev)
            inb[u_t] = True
            assert float(got[~inb].abs().max()) == 0, 'dV rows of users outside the batch are not 0'
            got, ref, S, A = got[inb], ref[inb], S[inb], A[inb]
        out[name] = check_segment(name, got, ref, S, A, bias[name])
    # the batch term of the reported loss, from the pre-update weights
    assert abs(float(loss[1]) - r['loss']) <= r['loss_tol'], (float(loss[1]), r['loss'], r['loss_tol'])
    worst = {c: max(out[s][c] for s in SEGMENTS) for c in 'abc'}
    print(f'worst ratios (a, b, c) = ({worst["a"]:.3g}, {worst["b"]:.3g}, {worst["c"]:.3g}); per segment '
          + ', '.join(f'{s}: ({out[s]["a"]:.2g}, {out[s]["b"]:.2g}, {out[s]["c"]:.2g})' for s in SEGMENTS))
    return worst


# (name, gemm, K, B, loss, labels, q, output, data): every branch of the step at least once -- fp16 / tf32 / FFMA;
# K = 50 (pitch 52), 255 (ones feature in the last column of a 256-wide tile), 256 (db' from the loss epilogue's column
# sums); B = 1, 129 (a ragged 128-row tile), 2048 (dW'^T split over the batch, s2 = 4 planes at I = 5000); both losses
# and label modes; the sampled-output step; q = 0 (keep ignored) and 0.2.
CASES = [
    ('ffma_k16_b1_bce_mean', 'ffma', 16, 1, 'bce', 'batch_mean', 0.2, 'dense', 'small'),
    ('ffma_k50_b129_bce_user', 'ffma', 50, 129, 'bce', 'per_user', 0.2, 'dense', 'small'),
    ('ffma_k200_b129_mse_mean_q0', 'ffma', 200, 129, 'mse', 'batch_mean', 0.0, 'dense', 'small'),
    ('ffma_k255_b129_mse_user', 'ffma', 255, 129, 'mse', 'per_user', 0.2, 'dense', 'small'),
    ('ffma_k50_b2048_bce_mean', 'ffma', 50, 2048, 'bce', 'batch_mean', 0.2, 'dense', 'large'),
    ('f16_k16_b129_bce_mean', 'tcgen05', 16, 129, 'bce', 'batch_mean', 0.2, 'dense', 'small'),
    ('f16_k50_b1_bce_mean', 'tcgen05', 50, 1, 'bce', 'batch_mean', 0.2, 'dense', 'small'),
    ('f16_k50_b129_bce_user_q0', 'tcgen05', 50, 129, 'bce', 'per_user', 0.0, 'dense', 'small'),
    ('f16_k200_b129_mse_mean', 'tcgen05', 200, 129, 'mse', 'batch_mean', 0.2, 'dense', 'small'),
    ('f16_k255_b129_bce_mean', 'tcgen05', 255, 129, 'bce', 'batch_mean', 0.2, 'dense', 'small'),
    ('f16_k255_b129_mse_user', 'tcgen05', 255, 129, 'mse', 'per_user', 0.2, 'dense', 'small'),
    ('f16_k256_b129_bce_mean', 'tcgen05', 256, 129, 'bce', 'batch_mean', 0.2, 'dense', 'small'),
    ('f16_k256_b129_mse_user', 'tcgen05', 256, 129, 'mse', 'per_user', 0.2, 'dense', 'small'),
    ('f16_k50_b2048_bce_mean_q0', 'tcgen05', 50, 2048, 'bce', 'batch_mean', 0.0, 'dense', 'large'),
    ('f16_k256_b2048_bce_user', 'tcgen05', 256, 2048, 'bce', 'per_user', 0.2, 'dense', 'large'),
    ('tf32_k16_b1_bce_mean', 'tcgen05_tf32', 16, 1, 'bce', 'batch_mean', 0.2, 'dense', 'small'),
    ('tf32_k50_b129_bce_mean', 'tcgen05_tf32', 50, 129, 'bce', 'batch_mean', 0.2, 'dense', 'small'),
    ('tf32_k255_b129_bce_user', 'tcgen05_tf32', 255, 129, 'bce', 'per_user', 0.2, 'dense', 'small'),
    ('tf32_k256_b129_mse_mean', 'tcgen05_tf32', 256, 129, 'mse', 'batch_mean', 0.2, 'dense', 'small'),
    ('tf32_k200_b2048_mse_user', 'tcgen05_tf32', 200, 2048, 'mse', 'per_user', 0.2, 'dense', 'large'),
    ('sampled_k50_b129_bce', 'auto', 50, 129, 'bce', 'per_user', 0.2, 'sampled', 'small'),
    ('sampled_k200_b64_mse_q0', 'auto', 200, 64, 'mse', 'per_user', 0.0, 'sampled', 'small'),
]

DATA = {'small': (400, 1200, 30, 700), 'large': (3000, 5000, 30, 900)}


@pytest.fixture(scope='module')
def datasets():
    return {k: _dataset(*v, seed=3) for k, v in DATA.items()}


def _keep_bytes(m, uids, q, seed):
    nnz = int(np.diff(m._h_indptr)[uids].sum())
    keep = (np.random.default_rng(seed).random(nnz) >= max(q, 0.2)).astype(np.uint8)
    return keep               # q == 0: the step ignores keep, so zeros in it must change nothing


@pytest.mark.gpu
@pytest.mark.parametrize('case', CASES, ids=[c[0] for c in CASES])
def test_step_gradients_vs_float64(case, datasets):
    name, gemm, K, B, loss, label_mode, q, output, data = case
    ds = datasets[data]
    U, I = DATA[data][:2]
    w = _weights(U, I, K, seed=K + B)
    m = _model(ds, K, B, w, gemm, loss, label_mode, q, output)
    assert m._native is not None and (output == 'sampled') == (m.output == 'sampled')
    uids = _batch(m, B, seed=B)
    _check_step(m, w, uids, _keep_bytes(m, uids, q, seed=B), q)


@pytest.mark.gpu
@pytest.mark.parametrize('q', [0.2, 0.0])
def test_step_gradients_engineered_logits(datasets, q):
    """fp16 BCE with batch-mean labels (the only instantiation with the fast epilogue form): items whose logits sit in
    bands around the fast-form threshold (|z| < 15.25) and Keras' clip, arranged so that some 16-row x 32-item chunks
    are all fast, some hold one extreme item among ordinary ones and some are extreme only; W' over 15 binary orders
    of magnitude and saturated hidden units.  B = 256: every chunk is full."""
    U, I, K, B = 400, 1200, 64, 256
    w = _weights(U, I, K, seed=11, engineered=True)
    m = _model(datasets['small'], K, B, w, 'tcgen05', 'bce', 'batch_mean', q)
    uids = _batch(m, B, seed=7)
    _check_step(m, w, uids, _keep_bytes(m, uids, q, seed=7), q, engineered=True)


@pytest.mark.gpu
def test_step_gradients_production_shape():
    """The C3 shape bench.py times: 138,493 users x 26,744 items, 20 M interactions, K = 200, B = 4096, default (fp16
    tensor-core) path, q = 0.2.  The reference runs in float64 on the GPU."""
    import drecpy_b200 as drb
    u, i, v = drb.synthetic_interactions(138493, 26744, 20_000_000, seed=10, zipf_a=1.0)
    ds = drb.InteractionData(u, i, v)
    ds.assign_internal_ids()
    U, I, K, B = 138493, 26744, 200, 4096
    w = _weights(U, I, K, seed=5)
    m = drb.CDAE(hidden_factors=K, corruption_level=0.2, seed=10, verbose=False, rng_mode='philox')
    m.fit(ds, epochs=0, batch_size=B, learning_rate=1e-3, reg_rate=0.1, init_weights=w)
    uids = np.random.default_rng(1).integers(0, U, B).astype(np.int32)
    uids[1] = uids[0]
    _check_step(m, w, uids, _keep_bytes(m, uids, 0.2, seed=1), 0.2)
