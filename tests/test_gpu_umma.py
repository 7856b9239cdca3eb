"""tcgen05 (split-precision products, TMA, TMEM) GEMM paths -- 3xFP16 (default) and 3xTF32 -- against the exact-fp32 FFMA
path and the oracle (GPU only)."""
import numpy as np
import pytest

import drecpy_b200 as drb
from oracle.cdae import CDAEOracle

pytestmark = pytest.mark.gpu


def _setup(U, I, K, B, nnz, gemm, seed=3, **kw):
    u, i, v = drb.synthetic_interactions(U, I, nnz, seed=seed)
    ds = drb.InteractionData(u, i, v)
    ds.assign_internal_ids()
    rng = np.random.default_rng(7)

    def glorot(shape, fi, fo):
        lim = np.sqrt(6.0 / (fi + fo))
        return rng.uniform(-lim, lim, shape).astype(np.float32)
    w = {'W': glorot((I, K), I, K), 'W_': glorot((K, I), K, I), 'V': glorot((U, K), U, K),
         'b': glorot((K,), K, K), 'b_': glorot((I,), I, I)}
    m = drb.CDAE(hidden_factors=K, seed=10, verbose=False, rng_mode='philox', gemm=gemm, **kw)
    m.fit(ds, epochs=0, batch_size=B, init_weights=w)
    return ds, w, m


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


@pytest.mark.parametrize('U,I,K,B,nnz', [(300, 1682, 50, 64, 12000), (500, 777, 200, 300, 20000),
                                         (257, 1000, 130, 128, 9000), (400, 2049, 64, 129, 15000),
                                         (300, 640, 16, 40, 6000),
                                         # hidden 256: no room for the ones feature, db' summed in the loss epilogue
                                         (300, 900, 256, 200, 9000),
                                         # hidden 248: the ones feature in column 248 of a 256-wide tile
                                         (200, 600, 248, 64, 5000)])
@pytest.mark.parametrize('label_mode,loss', [('batch_mean', 'bce'), ('per_user', 'mse')])
@pytest.mark.parametrize('gemm', ['tcgen05', 'tcgen05_tf32'])
def test_tcgen05_step_matches_ffma_and_oracle(U, I, K, B, nnz, label_mode, loss, gemm):
    import torch
    ds, w, m_tc = _setup(U, I, K, B, nnz, gemm, label_mode=label_mode, loss=loss)
    _, _, m_ff = _setup(U, I, K, B, nnz, 'ffma', label_mode=label_mode, loss=loss)
    o = CDAEOracle(w['W'], w['W_'], w['V'], w['b'], w['b_'], ds.csr(), corruption_level=0.0, loss=loss,
                   label_mode=label_mode, learning_rate=1e-3)
    deg = np.diff(ds.csr(1e-3)[0])
    rng = np.random.default_rng(0)
    for step in range(3):
        uids = rng.integers(0, U, B).astype(np.int32)
        off = np.concatenate([[0], np.cumsum(deg[uids])]).astype(np.int32)
        losses = []
        for m in (m_tc, m_ff):
            m.corruption_level = 0.0
            loss_dev = torch.zeros(2, device='cuda')
            d_u, d_o = torch.as_tensor(uids, device='cuda'), torch.as_tensor(off, device='cuda')
            # q=0.2 philox mask is identical in both models (same seed / step); compare them against each other
            m.step_device(d_u, d_o, None, 1e-3, loss_dev)
            losses.append(loss_dev[0].item())
        assert abs(losses[0] - losses[1]) <= 2e-5 * abs(losses[1]), (step, losses)
        for name in ('W', 'V', 'b', 'b_'):
            a, b = getattr(m_tc, name).cpu().numpy(), getattr(m_ff, name).cpu().numpy()
            assert rel(a, b) < 5e-4, (step, name, rel(a, b))
        assert rel(m_tc.W_.cpu().numpy(), m_ff.W_.cpu().numpy()) < 5e-4
    # gradient-level check of the first Adam step against the oracle is covered by test_gpu_parity (default path)
