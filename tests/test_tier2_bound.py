"""The tier-2 bound of the int8 route's three-tier re-score (topk_finalize_kernel with db16, see pack_q_i8_kernel):

    eps16 = (e ||q|| + 1.25 D 2^-24 (x + e) ||q|| + 1.25 D 2^-24 x ||q||) * 1.001 + 1e-7

with e = max_r ||bf16(x_r) - x_r||, x = max_r ||x_r|| (Index.stats()[0], [1]), bounds |s16 - fp32| for every row,
s16 = the bf16-rounded row against the fp32 query summed in fp32.  Checked here with bf16 rounding emulated in numpy
(round to nearest even on the fp32 bits), on randn and heavy-tailed rows of mixed norms."""
import numpy as np
import pytest


def bf16(x):
    b = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    b = (b + 0x7FFF + ((b >> 16) & 1)) & 0xFFFF0000
    return b.astype(np.uint32).view(np.float32)


def eps16(db, q):
    e = np.sqrt(((bf16(db).astype(np.float64) - db) ** 2).sum(1).max())
    x = np.sqrt((db.astype(np.float64) ** 2).sum(1).max())
    qn = np.sqrt((q.astype(np.float64) ** 2).sum(1))
    acc = 1.25 * db.shape[1] * 2.0 ** -24
    return (e * qn + acc * (x + e) * qn + acc * x * qn) * 1.001 + 1e-7


@pytest.mark.parametrize("dist", ["randn", "heavy_tailed"])
def test_tier2_bound_covers_bf16_rows(dist):
    rs = np.random.RandomState(7)
    n, D, nq = 20000, 2048, 8
    db = rs.randn(n, D) if dist == "randn" else rs.standard_t(2, size=(n, D))
    db = (db / np.linalg.norm(db, axis=1, keepdims=True) * rs.uniform(0.25, 2.0, (n, 1))).astype(np.float32)
    q = rs.randn(nq, D)
    q = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    q[1:, :] = q[1:, :] * np.float32(1.5)                        # the bound scales with ||q||
    s16 = bf16(db) @ q.T                                          # fp32 sums (BLAS order; the bound holds for any order)
    s32 = db @ q.T
    s64 = db.astype(np.float64) @ q.astype(np.float64).T
    # a row-by-row sequential fp32 sum, the worst order for accumulation error
    seq = np.zeros((200, nq), np.float32)
    for d in range(D):
        seq += bf16(db[:200, d:d + 1]) * q[:, d][None, :]
    err = np.abs(np.concatenate([s16 - s32, seq - s32[:200]]).astype(np.float64))
    eps = eps16(db, q)
    ratio = (err / eps[None, :]).max()
    print("tier-2 bound %s: max |s16 - fp32| / eps16 = %.3f, eps16 %.2e .. %.2e" % (dist, ratio, eps.min(), eps.max()))
    assert ratio < 1.0
    assert np.abs(s32 - s64).max() < 1.25 * D * 2.0 ** -24 * 2.0 * 1.5          # the fp32 term itself is a bound
    # not vacuous: within ~20x of the largest error met, and <= 3e-3 of ||x|| ||q|| (the int8 bound is ~1e-2 at unit norms)
    x_q = np.sqrt((db.astype(np.float64) ** 2).sum(1).max()) * np.sqrt((q.astype(np.float64) ** 2).sum(1))
    assert ratio > 0.03 and (eps / x_q).max() < 3e-3
