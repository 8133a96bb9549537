"""CPU: host side of PairwiseInteraction (fastselect_b200/_interaction.py) with the GPU hook
(``_interaction.open_interaction``) served by the numpy oracle (oracle/interaction_oracle.py): the fitted
attributes, the exact test (IPF, G, dof, p-values), the screening bound G <= L_KSA, and every parameter check."""
import pickle

import numpy as np
import pytest
from scipy.stats import chi2
from sklearn.base import clone

import fastselect_b200 as fsb
from fastselect_b200 import _interaction, _mdr, _native
from oracle import interaction_oracle as O
from oracle import mdr_oracle as M


@pytest.fixture
def hook(monkeypatch):
    opened = []

    def fake_open(X, y_enc):
        src = O.Source(X, y_enc)
        opened.append(src)
        return src

    monkeypatch.setattr(_interaction, "open_interaction", fake_open)
    monkeypatch.setattr(_native, "device_count", lambda: 1)
    return opened


def genotypes(seed, n, p, maf=None):
    """0/1/2 columns (some with a rare allele), a constant and a 2-valued column, a planted pair (2, 5)."""
    rs = np.random.RandomState(seed)
    X = rs.randint(0, 3, (n, p)).astype(np.int8)
    if maf is not None:
        X[:, 6:] = (rs.rand(n, p - 6) < maf) + (rs.rand(n, p - 6) < maf)
    X[:, 0] = 1
    X[:, 4] = rs.randint(0, 2, n)
    y = ((X[:, 2] == 1) & (X[:, 5] == 2)).astype(int)
    flip = rs.rand(n) < 0.3
    y[flip] = 1 - y[flip]
    return X, y


def assert_matches_oracle(est, want):
    for k in ("classes_", "pairs_", "dof_", "n_pairs_tested_"):
        assert np.array_equal(np.asarray(getattr(est, k)), np.asarray(want[k])), k
    for k in ("ksa_statistic_", "bound_"):            # the same oracle values through the hook: bitwise
        assert np.array_equal(np.asarray(getattr(est, k)).view(np.int64), np.asarray(want[k]).view(np.int64)), k
    np.testing.assert_allclose(est.statistic_, want["statistic_"], rtol=1e-7, atol=1e-7)
    np.testing.assert_allclose(est.p_values_, want["p_values_"], rtol=1e-6, atol=1e-300)


@pytest.mark.parametrize("n,p,n_top,maf", [(300, 12, 20, None), (120, 9, 36, 0.1), (500, 15, 105, 0.05),
                                           (60, 8, 1, None)])
def test_estimator_equals_oracle(hook, n, p, n_top, maf):
    X, y = genotypes(n + p, n, p, maf)
    est = fsb.PairwiseInteraction(n_top=n_top).fit(X, y)
    assert_matches_oracle(est, O.fit(X, y, n_top))
    assert hook[-1].calls == ["interaction_scan"]
    assert est.pairs_.dtype == np.int64 and est.pairs_.shape == (min(n_top, p * (p - 1) // 2), 2)
    assert np.all(est.pairs_[:, 0] < est.pairs_[:, 1])


def test_planted_pair_listed_first(hook):
    X, y = genotypes(3, 2000, 12)
    est = fsb.PairwiseInteraction(n_top=10).fit(X, y)
    assert tuple(est.pairs_[0]) == (2, 5)
    assert est.p_values_[0] < 0.05 / est.n_pairs_tested_
    assert est.n_pairs_tested_ == 66 and est.bound_ == est.ksa_statistic_[-1]


def test_every_pair_listed_bound_is_zero(hook):
    X, y = genotypes(4, 200, 6)
    est = fsb.PairwiseInteraction(n_top=2048).fit(X, y)          # clamps to the 15 pairs
    assert est.pairs_.shape == (15, 2) and est.bound_ == 0.0
    assert {tuple(r) for r in est.pairs_} == {(a, b) for a in range(6) for b in range(a + 1, 6)}


def test_list_order_and_ties(hook):
    X, y = genotypes(5, 400, 8)
    X = np.concatenate([X, X[:, [5, 2]]], axis=1)                 # 8 <- 5, 9 <- 2: exact copies, equal KSA
    est = fsb.PairwiseInteraction(n_top=45).fit(X, y)
    k = est.ksa_statistic_
    assert np.all(k[:-1] >= k[1:])
    idx = _mdr.encode_combinations(est.pairs_, 10)
    for q in range(k.size - 1):
        if k[q] == k[q + 1]:
            assert idx[q] < idx[q + 1]
    # (2, 5) = (2, 8) and (5, 9) = (8, 9) bitwise; the two groups hold the same table transposed, which the
    # cell-ordered sums may round differently
    top = [tuple(r) for r in est.pairs_[:4]]
    assert set(top) == {(2, 5), (2, 8), (5, 9), (8, 9)}
    assert top.index((2, 5)) < top.index((2, 8)) and top.index((5, 9)) < top.index((8, 9))


def test_ipf_recovers_a_no_three_way_table():
    """n_ijk = u_ij v_ik w_jk is itself in the model: the fit is n and G = 0 (up to the IPF tolerance)."""
    rs = np.random.RandomState(0)
    u, v, w = rs.randint(1, 6, (50, 3, 3)), rs.randint(1, 6, (50, 3, 2)), rs.randint(1, 6, (50, 3, 2))
    n = u[:, :, :, None] * v[:, :, None, :] * w[:, None, :, :]     # [m, i, j, k]
    n[:10, 2, :, :] = 0                                            # a column state never seen
    n[10:20, :, 1, :] = 0
    tab = n.transpose(0, 3, 1, 2).reshape(50, 2, 9)
    mu = _interaction.no_three_way_fit(n.astype(np.float64))
    np.testing.assert_allclose(mu, n, rtol=1e-6, atol=1e-6)           # margins within 1e-9 N
    G = _interaction.lr_statistic(tab)
    assert np.all(G >= 0) and np.all(G < 1e-6)
    for q in (0, 15, 49):
        assert O.lr_test(tab[q], 3, 3)[0] < 1e-6


def data_tables(seed, n, p, maf):
    X, y = genotypes(seed, n, p, maf)
    codes, n_states = M.cells(X)
    return O.tables(codes, y), n_states


@pytest.mark.parametrize("seed,n,maf", [(0, 60, None), (1, 80, 0.1), (2, 400, 0.05), (3, 3000, 0.02), (4, 1000, None)])
def test_g_is_bounded_by_ksa(seed, n, maf):
    tab, _ = data_tables(seed, n, 14, maf)
    assert (tab == 0).any(axis=(1, 2)).sum() > 0                    # zero cells, constant and 2-valued columns
    G = _interaction.lr_statistic(tab)
    L = O.ksa(tab)
    assert np.all(G >= 0)
    assert np.all(G <= L + 1e-9 * n + 1e-9 * np.abs(L)), np.max(G - L)
    for q in range(0, tab.shape[0], 13):                            # the per-table loop agrees
        assert abs(O.lr_test(tab[q], 3, 3)[0] - G[q]) <= 1e-7 * max(1.0, G[q])


def test_ksa_of_a_hand_table():
    """KSA from its definition on one table, summed in another order."""
    t = np.array([[[5, 3, 0], [2, 7, 1], [0, 4, 6]], [[1, 2, 3], [8, 0, 2], [3, 3, 9]]])  # [k, i, j]
    n = t.transpose(1, 2, 0).astype(float)
    N = n.sum()
    q = np.zeros_like(n)
    for i in range(3):
        for j in range(3):
            for k in range(2):
                num = n[i, j, :].sum() * n[i, :, k].sum() * n[:, j, k].sum()
                q[i, j, k] = num / (n[i].sum() * n[:, j].sum() * n[:, :, k].sum()) if num else 0.0
    eta = q.sum()
    pos = n > 0
    want = 2 * np.sum(n[pos] * np.log(n[pos] * eta / (N * q[pos])))
    got = O.ksa(t.reshape(1, 2, 9))[0]
    assert got == pytest.approx(want, rel=1e-12)
    assert got >= 0


def test_dof_and_p_values(hook):
    X, y = genotypes(6, 300, 7)                                     # column 0 constant, column 4 2-valued
    est = fsb.PairwiseInteraction(n_top=21).fit(X, y)
    states = np.array([1, 3, 3, 3, 2, 3, 3])
    for (a, b), d, g, pv in zip(est.pairs_, est.dof_, est.statistic_, est.p_values_):
        assert d == (states[a] - 1) * (states[b] - 1)
        if d == 0:
            assert pv == 1.0
        else:
            assert pv == pytest.approx(chi2.sf(g, d), rel=1e-12)
    assert set(est.dof_.tolist()) == {0, 2, 4}
    assert np.array_equal(_interaction.p_values(np.array([0.0, 3.0, 3.0]), [0, 0, 4]),
                          [1.0, 1.0, chi2.sf(3.0, 4)])


def test_ipf_cap_raises():
    tab, _ = data_tables(0, 300, 6, None)
    with pytest.raises(RuntimeError, match="did not converge"):
        _interaction.no_three_way_fit(tab.reshape(-1, 2, 3, 3).transpose(0, 2, 3, 1).astype(float), max_cycles=1)


def test_refit_clone_pickle(hook):
    X, y = genotypes(7, 200, 6)
    labels = np.where(y == 1, "case", "ctrl")
    est = fsb.PairwiseInteraction(n_top=5).fit(X, labels)
    assert list(est.classes_) == ["case", "ctrl"]
    est2 = pickle.loads(pickle.dumps(est))
    assert np.array_equal(est2.pairs_, est.pairs_)
    assert not any(isinstance(v, (_native.Dataset, _mdr.MDRData)) for v in vars(est).values())
    c = clone(est)
    assert c.get_params() == est.get_params() and not hasattr(c, "pairs_")
    est.set_params(n_top=3).fit(X, y)
    assert est.pairs_.shape == (3, 2)
    assert not hasattr(est, "predict") and not hasattr(est, "transform")


def test_value_errors(hook):
    X, y = genotypes(8, 60, 6)
    X4 = X.copy()
    X4[0, 1] = 7                                                    # a 4th state
    with pytest.raises(ValueError, match="at most 3"):
        fsb.PairwiseInteraction().fit(X4, y)
    with pytest.raises(ValueError, match="2 classes"):
        fsb.PairwiseInteraction().fit(X, np.arange(60) % 3)
    with pytest.raises(ValueError, match="2 classes"):
        fsb.PairwiseInteraction().fit(X, np.zeros(60))
    for bad in (0, -1, _native.FS_MDR_MAX_TOP + 1, 2.5, True):
        with pytest.raises(ValueError, match="n_top"):
            fsb.PairwiseInteraction(n_top=bad).fit(X, y)
    with pytest.raises(ValueError, match="numeric"):
        fsb.PairwiseInteraction().fit(X.astype(str).astype(object), y)
    with pytest.raises(ValueError):
        fsb.PairwiseInteraction().fit(np.where(X == 0, np.nan, X), y)
    with pytest.raises(ValueError, match="at least 2 features"):
        fsb.PairwiseInteraction().fit(X[:, :1], y)


def test_backends(hook, monkeypatch):
    X, y = genotypes(9, 60, 6)
    with pytest.raises(NotImplementedError):
        fsb.PairwiseInteraction(backend="cpu").fit(X, y)
    with pytest.raises(ValueError, match="backend"):
        fsb.PairwiseInteraction(backend="tpu").fit(X, y)
    monkeypatch.setattr(_native, "device_count", lambda: 0)
    with pytest.raises(RuntimeError):
        fsb.PairwiseInteraction().fit(X, y)
