"""mdir_b200.DiffusionTable (offline diffusion) on the GPU: every table row equals Diffusion.search of that row with
k_q = 1 bit for bit; the combine kernel matches tests/diffusion_offline_reference.py:offline_search on the GPU's own
table and top-k_q lists; results are batch-invariant; the chain mAP gain holds; a table built after remove + compact
equals one of a fresh index; out-of-range parameters and stale tables are refused."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import diffusion_offline_reference as oref  # noqa: E402
from test_gpu_diffusion import build_case, chains, map_at  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
N_DB, D, K = 20000, 128, 50
WIDTH, TRUNC = 100, 500
PARAMS = dict(alpha=0.99, iters=20, rtol=1e-6)
F_TOL = 1e-6          # max |f - f_ref| / max |f_ref|: only pow() of the weights can differ


@pytest.fixture(scope="module")
def m():
    import mdir_b200
    return mdir_b200


def _unit(x):
    return x / x.norm(dim=1, keepdim=True)


_CASES = {}


def case(m, dist):
    """(index, Diffusion(k=50), table(width 100, trunc 500), q), built once per module."""
    if dist not in _CASES:
        db, q = build_case(dist)
        index = m.Index(db, device=DEV)
        g = m.Diffusion(index, k=K, gamma=3.0)
        _CASES[dist] = (index, g, g.offline(width=WIDTH, trunc=TRUNC, **PARAMS), q)
    return _CASES[dist]


def check_rows(g, tab, rows, width, trunc):
    """Table rows equal Diffusion.search(db32[i:i+1], k=width, trunc, k_q=1) bit for bit."""
    t_ids, t_f = tab.table()
    for i in rows:
        f, ids = g.search(g.index.db32[i:i + 1], k=width, trunc=trunc, k_q=1, **PARAMS)
        assert torch.equal(ids[0], t_ids[i]) and torch.equal(f[0].view(torch.int32), t_f[i].view(torch.int32)), i


@pytest.mark.parametrize("dist", ["randn", "clusters", "near_dup"])
def test_table_rows_equal_diffusion_search(m, dist, monkeypatch):
    index, g, tab, _ = case(m, dist)
    rows = np.random.RandomState(1).choice(N_DB, 40, replace=False).tolist()
    if dist == "randn":
        rows += [999, 1000, 1040, 1079]                                    # the 81-copy clique: one seed, one table row
        t_ids, t_f = tab.table()
        assert torch.equal(t_ids[1000], t_ids[999]) and torch.equal(t_f[1079], t_f[999])
    check_rows(g, tab, rows, WIDTH, TRUNC)
    import mdir_b200.diffusion as dmod
    monkeypatch.setattr(dmod, "OFFLINE_CHUNK", 3001)                      # other chunks and 1,024-query scan passes
    monkeypatch.setattr(dmod, "OFFLINE_BLOCK_Q", 1024)
    other = g.offline(width=WIDTH, trunc=TRUNC, **PARAMS)
    assert torch.equal(other.tab_ids, tab.tab_ids) and torch.equal(other.tab_f.view(torch.int32), tab.tab_f.view(torch.int32))


def test_table_fewer_live_rows_than_trunc(m):
    db, _ = build_case("clusters", seed=5)
    index = m.Index(db[:600], device=DEV, capacity=1000)                  # 600 live rows, a free tail of 400
    g = m.Diffusion(index, k=10)
    tab = g.offline(width=1000, trunc=1000, **PARAMS)
    t_ids, t_f = tab.table()
    assert t_ids.shape == (600, 1000)
    assert (t_ids[:, 600:] == -1).all() and torch.isneginf(t_f[:, 600:]).all() and (t_ids[:, :600] >= 0).all()
    assert (tab.tab_ids[600:] == -1).all() and torch.isneginf(tab.tab_f[600:]).all()
    check_rows(g, tab, [0, 17, 311, 599], 1000, 1000)


def check_combine(m, tab, q, k, k_q):
    index = tab.index
    f, ids = tab.search(q, k=k, k_q=k_q)
    s, L = index.search(q, k_q, precision="fp32")
    t_ids, t_f = (t.cpu().numpy() for t in tab.table())
    _, _, fulls = oref.offline_search(t_ids, t_f, L.cpu().numpy(), s.cpu().numpy(), k, gamma=tab.gamma, slot_id=index._ids)
    f, ids = f.cpu().numpy(), ids.cpu().numpy()
    padded = 0
    for qi in range(f.shape[0]):
        ref = fulls[qi]
        u_ids = np.fromiter(ref.keys(), dtype=np.int64, count=len(ref))
        u_f = np.fromiter(ref.values(), dtype=np.float64, count=len(ref))
        bound = F_TOL * max(np.abs(u_f).max(initial=0), np.finfo(np.float32).tiny)
        mm = min(k, u_ids.size)
        padded += mm < k
        assert (ids[qi, mm:] == -1).all() and np.isneginf(f[qi, mm:]).all()
        got = ids[qi, :mm].astype(np.int64)
        assert np.unique(got).size == mm and all(int(j) in ref for j in got)
        got_f = np.array([ref[int(j)] for j in got])
        assert np.abs(f[qi, :mm] - got_f).max(initial=0) <= bound, qi
        want = u_ids[np.lexsort((u_ids, -u_f.astype(np.float32)))[:mm]]
        diff = got != want
        want_f = np.array([ref[int(j)] for j in want])
        assert np.all(np.abs(got_f[diff] - want_f[diff]) <= bound), qi
    return padded


@pytest.mark.parametrize("dist", ["randn", "clusters", "near_dup"])
@pytest.mark.parametrize("k,k_q", [(100, 10), (1000, 10), (7, 1), (8192, 81)])
def test_combine_matches_restatement(m, dist, k, k_q):
    _, _, tab, q = case(m, dist)
    padded = check_combine(m, tab, q, k, k_q)
    if k > k_q * WIDTH:
        assert padded == q.shape[0]                                       # the union is smaller than k: padding


def test_status_words(m):
    index, _, tab, q = case(m, "near_dup")
    tab.search(q, k=100, k_q=10)
    st = tab.status().clone()
    index.search(q, 10, precision="fp32")
    assert torch.equal(st, index.status()[:q.shape[0]])


def test_deterministic_and_batch_invariant(m):
    index, _, tab, _ = case(m, "clusters")
    g0 = torch.Generator(device=DEV).manual_seed(21)
    src = torch.randint(0, N_DB, (200,), device=DEV, generator=g0)
    q = _unit(index.db32[src] + 0.5 * torch.randn((200, D), device=DEV, generator=g0) / D ** 0.5)   # 200 > 128: two scan blocks
    f1, i1 = tab.search(q)
    f2, i2 = tab.search(q)
    assert torch.equal(f1.view(torch.int32), f2.view(torch.int32)) and torch.equal(i1, i2)
    for j in (0, 137, 199):
        fa, ia = tab.search(q[j:j + 1])
        assert torch.equal(fa[0].view(torch.int32), f1[j].view(torch.int32)) and torch.equal(ia[0], i1[j]), j
    fb, ib = tab.search(q[100:190])                                       # another batch composition
    assert torch.equal(fb.view(torch.int32), f1[100:190].view(torch.int32)) and torch.equal(ib, i1[100:190])


def test_map_on_chains(m):
    X, Q, lab = chains()
    index = m.Index(X, device=DEV)
    g = m.Diffusion(index, k=30, gamma=3.0)
    tab = g.offline(width=100, trunc=500, **PARAMS)
    f, ids = tab.search(Q, k=100, k_q=10)
    _, on_ids = g.search(Q, k=100, trunc=500, k_q=10, **PARAMS)
    _, L = index.search(Q, 100, precision="fp32")
    s10, L10 = index.search(Q, 10, precision="fp32")
    t_ids, t_f = (t.cpu().numpy() for t in tab.table())
    _, ref_ids, _ = oref.offline_search(t_ids, t_f, L10.cpu().numpy(), s10.cpu().numpy(), 100, gamma=3.0)
    m_off, m_ref = map_at(ids.cpu().numpy(), lab), map_at(ref_ids, lab)
    m_plain, m_on = map_at(L.cpu().numpy(), lab), map_at(on_ids.cpu().numpy(), lab)
    print("chain mAP@100: plain %.4f, online diffusion %.4f, offline table %.4f (restatement %.4f)" % (m_plain, m_on, m_off, m_ref))
    assert abs(m_off - m_ref) <= 0.005
    assert m_off >= m_plain + 0.03


def test_table_after_compact(m):
    db, q = build_case("clusters", seed=7)
    a = m.Index(db.clone(), device=DEV)                                  # compact() rewrites the master copy in place
    ga = m.Diffusion(a, k=K)
    gone = np.random.RandomState(0).choice(N_DB, 3000, replace=False)
    ga.remove(gone)
    ga.compact()
    ta = ga.offline(width=WIDTH, trunc=TRUNC, **PARAMS)
    live = np.setdiff1d(np.arange(N_DB), gone)
    b = m.Index(db[torch.from_numpy(live).to(DEV)], device=DEV)
    tb = m.Diffusion(b, k=K).offline(width=WIDTH, trunc=TRUNC, **PARAMS)
    (ia, fa), (ib, fb) = ([t.cpu().numpy() for t in x.table()] for x in (ta, tb))
    assert np.array_equal(fa.view(np.int32), fb.view(np.int32))
    assert np.array_equal(ia, np.where(ib >= 0, live[np.maximum(ib, 0)], -1))
    fa, ia = ta.search(q)
    fb, ib = tb.search(q)
    assert torch.equal(fa.view(torch.int32), fb.view(torch.int32))
    assert np.array_equal(ia.cpu().numpy(), live[ib.cpu().numpy()])


def test_refusals(m):
    db, q = build_case("randn", seed=9)
    index = m.Index(db[:5000], device=DEV, capacity=6000)
    g = m.Diffusion(index, k=20)
    tab = g.offline(width=50, trunc=200, **PARAMS)
    f0, i0 = tab.search(q, k=50, k_q=10)
    st0 = tab.status()
    for bad in (dict(width=0), dict(width=1025, trunc=2048), dict(width=300, trunc=200), dict(trunc=2049)):
        with pytest.raises(m.MdirError):
            g.offline(**{**dict(width=50, trunc=200), **bad})
    for bad in (dict(k_q=0), dict(k_q=129), dict(k=0), dict(k=8193)):
        with pytest.raises(m.MdirError):
            tab.search(q, **{**dict(k=50, k_q=10), **bad})
    wide = g.offline(width=100, trunc=200, **PARAMS)
    with pytest.raises(m.MdirError, match="k_q \\* width"):
        wide.search(q, k=50, k_q=82)                                      # 8,200 entries
    assert tab.status() is st0
    f1, i1 = tab.search(q, k=50, k_q=10)                                  # unchanged
    assert torch.equal(f1.view(torch.int32), f0.view(torch.int32)) and torch.equal(i1, i0)
    # a mutation through the Diffusion keeps the graph current, not the table
    g.add(db[5000:5010])
    with pytest.raises(m.MdirError, match="mutated"):
        tab.search(q, k=50, k_q=10)
    tab = g.offline(width=50, trunc=200, **PARAMS)                        # a rebuild works
    tab.search(q, k=50, k_q=10)
    # a mutation on the index directly: the table and the graph are both stale
    index.remove([5])
    with pytest.raises(m.MdirError, match="mutated"):
        tab.search(q, k=50, k_q=10)
    with pytest.raises(m.MdirError, match="mutated"):
        g.offline(width=50, trunc=200, **PARAMS)
    index.restore([5])                                                    # back to the same rows, but still a mutation
    with pytest.raises(m.MdirError, match="mutated"):
        tab.search(q, k=50, k_q=10)
