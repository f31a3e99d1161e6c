"""The entrywise reference of the affine-coefficient hand-off (oracle/exact_affine.py), on the CPU.

Each coefficient Z_v[r, c] on the cover's upper triangle is held to |dev − ref| ≤ γ_N·abs + N·2⁻¹⁰⁷⁴, and
coefficients whose abs is 0 must be exactly 0 or absent.  Here:
- Z₀ + Σ γ_v Z_v, built from the exact coefficients, equals exact_z's Z(γ) exactly on every shape and output kind, so
  the two restatements pin each other;
- the per-variable order matches the literal assembly (oracle.affine_structure);
- the exact and extended modes agree;
- the nine committed device hand-offs (tests/golden/handoff_*.npz) meet the criterion, coefficient by coefficient
  and on every z0 entry;
- four bugs that the normwise check max |dev − ref| ≤ 1e-12·scale lets through are caught by it."""
import glob
import os
from fractions import Fraction

import numpy as np
import pytest

import exact_affine as ea
import exact_z as ez
import nnsdp_oracle as o
from helpers import assert_meets, rand_net, rand_query, wide_range_case

KINDS = ["safety", "hplaneS", "hplane", "circle", "ellipsoid"]
# the shapes of test_cpu_z_exact.py: β > a layer's width ([2, 1, 2, 2], 3) and β ≥ acdim ([2, 3, 2], 2)
SHAPES = [([2, 3, 2], 0), ([2, 3, 2], 2), ([2, 3, 3, 2], 1), ([3, 3, 3, 3, 4, 3, 3], 2), ([2, 10, 10, 10, 10, 2], 3),
          ([2, 4, 7, 3, 5, 2], 5), ([2, 1, 2, 2], 3), ([2] + [10] * 9 + [2], 7)]
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def ibp_case(xdims, beta, kind, seed):
    """(net, query, its IBP bounds as the given QC bounds)"""
    net = rand_net(xdims, seed=seed)
    q = rand_query(net, beta, np.random.default_rng(seed), kind=kind, radius=0.3)
    r = o.run_query(net, beta, q)
    return net, q, (r["qc_bounded"].acymin, r["qc_bounded"].acymax, r["qc_sector"].smin, r["qc_sector"].smax)


def gamma_vector(q):
    """the query's multipliers in the hand-off's variable order"""
    gout = [] if q.gout is None else np.atleast_1d(q.gout)
    return np.concatenate([q.gin, gout, q.gbnd, q.gsec])


def dyadic(rng, n):
    """random dyadic numbers spanning 2^±40"""
    return rng.integers(1, 2 ** 20, n) * 2.0 ** rng.integers(-60, 21, n)


def fp64_list(A):
    """(var, ent, val) of the reference rounded to FP64: what a correct device returns"""
    return A.var, A.ent, np.array([float(x) for x in A.ref])


# ---- Z₀ + Σ γ_v Z_v = exact_z, exactly ----------------------------------------------------------------------------

@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("xdims,beta", SHAPES)
def test_sum_of_coefficients_is_exact_z(xdims, beta, kind):
    rng = np.random.default_rng(len(xdims) * 8 + beta)
    for what, (net, q, bounds) in (("IBP", ibp_case(xdims, beta, kind, seed=beta + 1)),
                                   ("wide range", wide_range_case(xdims, beta, kind, seed=beta + 2))):
        q.gin, q.gbnd, q.gsec = dyadic(rng, len(q.gin)), dyadic(rng, len(q.gbnd)), dyadic(rng, len(q.gsec))
        if q.gout is not None:
            q.gout = dyadic(rng, 1)
        A = ea.exact_affine(net, beta, q, bounds)
        lay = A.lay
        g = gamma_vector(q)
        assert len(g) == lay.nvar
        assert lay.var_sec + len(q.gsec) == lay.nvar
        contrib = np.asarray([Fraction(x) for x in g], dtype=object)[A.var] * A.ref
        tot = np.empty(lay.nent, dtype=object)
        tot.fill(Fraction(0))
        np.add.at(tot, A.ent, contrib)
        Z0 = ea.exact_z0(net, beta, q, bounds).ref
        Z = ez.exact_z(net, beta, q, bounds).ref
        er, ec = lay.ent_row, lay.ent_col
        assert all(Z0[er, ec] + tot == Z[er, ec]), what
        off = lay.ent_of < 0
        off &= off.T
        assert all(Z[off] == 0) and all(Z0[off] == 0), what


# ---- the variable order -------------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", ["safety", "hplane", "circle", "ellipsoid"])
@pytest.mark.parametrize("xdims,beta", [([2, 3, 3, 2], 1), ([2, 4, 7, 3, 5, 2], 3), ([2, 1, 2, 2], 3)])
def test_variable_order_matches_the_literal_assembly(xdims, beta, kind):
    """Z_v = Z(e_v) − Z(0) of the literal assembly (its error relative to Z), variable by variable"""
    net, q, bounds = ibp_case(xdims, beta, kind, seed=11)
    A = ea.exact_affine(net, beta, q, bounds)
    Z0, Zv = o.affine_structure(net, beta, q.x1min, q.x1max, q.qc_out)
    assert len(Zv) == A.lay.nvar
    D = A.dense().astype(np.float64)
    er, ec = A.lay.ent_row, A.lay.ent_col
    for v in range(A.lay.nvar):
        ref = Zv[v][er, ec]
        scale = max(np.abs(ref).max(), np.abs(Z0).max())
        assert np.abs(D[:, v] - ref).max() <= 1e-12 * scale, v
        assert np.array_equal(D[:, v] != 0, np.abs(ref) > 1e-12 * scale), v


# ---- the two arithmetic modes agree --------------------------------------------------------------------------------

@pytest.mark.parametrize("beta", range(6))
def test_exact_and_extended_modes_agree(beta):
    xdims = [2, 4, 7, 3, 5, 2] if beta % 2 else [3, 3, 3, 3, 4, 3, 3]
    for i, kind in enumerate(KINDS):
        net, q, bounds = wide_range_case(xdims, beta, kind, seed=10 * beta + i)
        X = ea.exact_affine(net, beta, q, bounds, mode="exact")
        E = ea.exact_affine(net, beta, q, bounds, mode="extended")
        assert np.array_equal(X.key, E.key) and np.array_equal(X.N, E.N)
        assert np.array_equal(X.abs == 0, E.abs == 0) and (E.abs >= X.abs).all()
        ext = np.array([Fraction(*v.as_integer_ratio()) for v in E.ref], dtype=object)
        u = Fraction(ez.UEXT)
        assert all(abs(e - x) <= (n * u / (1 - n * u)) * a
                   for e, x, n, a in zip(ext, X.ref, E.N.tolist(), X.abs_exact)), kind


# ---- the committed device hand-offs --------------------------------------------------------------------------------

@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "handoff_*.npz"))), ids=os.path.basename)
def test_committed_handoff_meets_the_entrywise_criterion(path):
    """nnsdp_affine_create / get on the reference's W10 nets (CROWN bounds, ellipsoid): every summed COO coefficient
    and every z0 entry"""
    d = np.load(path)
    name = os.path.basename(path).split("handoff_")[1].split("_beta")[0]
    net = o.load_nnet(os.path.join(GOLDEN, f"scale-I2-O2-{name}.nnet"))
    beta = int(d["beta"])
    assert list(net.xdims) == d["xdims"].tolist()
    ac = net.acdim
    q = o.NumericQuery(x1min=d["x1min"], x1max=d["x1max"], gin=np.zeros(2), gbnd=np.zeros(ac),
                       gsec=np.zeros(o.sector_lambda_dim(ac, beta) + 2 * ac),
                       qc_out=o.QcReachEllipsoid(d["invP"], d["yc"]), gout=np.zeros(1))
    bounds = (d["ymin"], d["ymax"], d["smin"], d["smax"])
    A = ea.exact_affine(net, beta, q, bounds)
    assert np.array_equal(A.lay.ent_row + 1, d["ent_row"]) and np.array_equal(A.lay.ent_col + 1, d["ent_col"])
    assert int(d["nvar"]) == A.lay.nvar and int(d["var_sec"]) == A.lay.var_sec
    assert_meets(A, (d["coo_var"] - 1, d["coo_ent"] - 1, d["coo_val"]), path)
    Zd = np.zeros((net.Zdim, net.Zdim))
    er, ec = d["ent_row"] - 1, d["ent_col"] - 1
    Zd[er, ec] = Zd[ec, er] = d["z0"]
    assert_meets(ea.exact_z0(net, beta, q, bounds), Zd, f"{path} z0")


# ---- mutations the normwise criterion lets through -----------------------------------------------------------------

MUT_XDIMS, MUT_BETA, MUT_SEED = [2] + [4] * 8 + [2], 1, 7   # layer scales 2^±24: coefficients up to ~1e15


@pytest.fixture(scope="module")
def mut_case():
    net, q, bounds = wide_range_case(MUT_XDIMS, MUT_BETA, "safety", seed=MUT_SEED)
    A = ea.exact_affine(net, MUT_BETA, q, bounds)
    Z0 = ea.exact_z0(net, MUT_BETA, q, bounds).ref
    scale = max(np.abs(A.ref.astype(np.float64)).max(), np.abs(Z0.astype(np.float64)).max())
    return net, q, bounds, A, scale


def _caught_only_entrywise(A, scale, dev, mutated):
    """dev meets max |dev − ref| ≤ 1e-12·scale per variable (the normwise check) but breaks the entrywise bound at
    the (variable, entry) pairs `mutated` and nowhere else"""
    lay = A.lay
    var, ent, val = dev
    Dm = np.zeros((lay.nent, lay.nvar))
    np.add.at(Dm, (ent, var), val)
    assert np.abs(Dm - A.dense().astype(np.float64)).max() <= 1e-12 * scale
    assert_meets(A, fp64_list(A), "unmutated")
    ok, _ = A.check(dev)
    bad = {(int(k) // lay.nent, int(k) % lay.nent) for k in A._union[~ok]}
    assert bad and bad <= set(mutated), bad


def _layer1_gram_neuron(bounds):
    smin, smax = bounds[2], bounds[3]
    return next(j for j in range(2, MUT_XDIMS[1]) if smin[j] != 0 and smax[j] != 0)


def test_mutation_dropped_gram_coefficients_of_a_small_layer_neuron(mut_case):
    net, q, bounds, A, scale = mut_case
    j = _layer1_gram_neuron(bounds)
    v = A.lay.var_sec + j
    var, ent, val = fp64_list(A)
    r, c = A.lay.ent_row[ent], A.lay.ent_col[ent]
    n1, a = MUT_XDIMS[0], net.Zdim - 1
    gram = (var == v) & (r < n1) & ((c < n1) | (c == a))            # ρ ρ' on block 0 and column a
    gram |= (var == v) & (r == a)
    assert gram.sum() == n1 * (n1 + 1) // 2 + n1 + 1
    keep = ~gram
    _caught_only_entrywise(A, scale, (var[keep], ent[keep], val[keep]), list(zip(var[gram], ent[gram])))


def test_mutation_rho_i_and_rho_j_swapped_in_one_pair(mut_case):
    net, q, bounds, A, scale = mut_case
    ac, i = net.acdim, 2                                            # the pair (2, 3) of layer 1
    pairs = o.sector_pairs(ac, MUT_BETA) - 1
    k = int(np.nonzero((pairs[:, 0] == i) & (pairs[:, 1] == i + 1))[0][0])
    v = A.lay.var_sec + ac + k
    swapped = o.FeedFwdNet(xdims=list(net.xdims), Ms=[M.copy() for M in net.Ms])
    swapped.Ms[0][[i, i + 1]] = swapped.Ms[0][[i + 1, i]]
    S = ea.exact_affine(swapped, MUT_BETA, q, bounds, vars=[v])
    var, ent, val = fp64_list(A)
    mine = var == v
    svar, sent, sval = fp64_list(S)
    assert np.array_equal(ent[mine], sent)
    dev = (np.r_[var[~mine], svar], np.r_[ent[~mine], sent], np.r_[val[~mine], sval])
    changed = sent[sval != val[mine]]
    assert len(changed) >= 2 * (MUT_XDIMS[0] + 1)
    _caught_only_entrywise(A, scale, dev, [(v, e) for e in changed])


def test_mutation_eta_coefficient_sign_flipped(mut_case):
    net, q, bounds, A, scale = mut_case
    j = 3
    v = A.lay.var_sec + A.lay.lamdim + j                            # η_j
    e = A.lay.ent_of[MUT_XDIMS[0] + j, net.Zdim - 1]                # (e_j, a): the coefficient 1
    var, ent, val = fp64_list(A)
    at = np.nonzero((var == v) & (ent == e))[0]
    assert len(at) == 1 and val[at[0]] == 1.0
    val = val.copy()
    val[at] = -val[at]
    _caught_only_entrywise(A, scale, (var, ent, val), [(v, e)])


def test_mutation_coefficient_moved_to_the_next_entry_of_its_column(mut_case):
    net, q, bounds, A, scale = mut_case
    j = _layer1_gram_neuron(bounds)
    v = A.lay.var_sec + A.lay.lamdim + net.acdim + j                # ν_j: −smax w_r on (r, a)
    a = net.Zdim - 1
    e0, e1 = A.lay.ent_of[0, a], A.lay.ent_of[1, a]
    assert e1 == e0 + 1
    var, ent, val = fp64_list(A)
    at = np.nonzero((var == v) & (ent == e0))[0]
    assert len(at) == 1 and val[at[0]] != 0
    ent = ent.copy()
    ent[at] = e1
    _caught_only_entrywise(A, scale, (var, ent, val), [(v, e0), (v, e1)])
