"""Explicit-basis driver for the basis-update tests: one object (the oracle, a BLU, or the bases of a BLUBatch) goes
through a seeded sequence of basis changes while the test keeps B as an explicit matrix, and every step is checked
against real linear algebra on that matrix, not only against the oracle.

Per step: solve_for_update 'N' on the entering column, a leaving position (argmax |lhs| or a random eligible entry,
sometimes one where lhs is exactly zero so that the update is refused), solve_for_update 'T', update.  The branch the
update took is read off the nforrest_total / nsymperm_total deltas:

  ft       Forrest-Tomlin (a row eta was stored)
  sym      symmetric permutation (the spike has its diagonal, no intersection with the row eta)
  unsym    unsymmetric permutation through the BFS path (the spike lacks its diagonal; D4 / D14 repaired code)
  refused  SingularUpdate (-6): B stays as it was and the object is refactorized

The unsymmetric branch is hit on purpose: right after a factorization, `constructed_column` reads L and U and builds an
entering column whose spike is a single entry off the diagonal of the leaving position.

The bound.  After each accepted update the backward error of the object's solves with the new B' (dense 'N' / 'T' on a
random right-hand side, sparse 'N' / 'T', and the entering column itself) is compared with the backward error of a
fresh oracle factorization of the same explicit B' with the same tunables:

    eta_update <= C_BOUND * max(eta_fresh, m * eps) * (1 + max_eta) * max(1, max_pivot / max|B'|)

The last two factors are the growth an update allows: max_eta (the largest row-eta entry since the factorization)
because Forrest-Tomlin applies its row etas without pivoting, and max_pivot against the largest entry of B' because
the new column of U is the spike, unpivoted as well.  Steps where a fresh factorization finds B' singular are not
compared.  Measured on the oracle with droptol <= 1e-12, seeds 0..599 of draw_case (about 16,600 updates): the ratio
to the bound without C_BOUND is at most 1 on 16,599 of them and 328 on one, a symmetric permutation on the badly scaled
seed 60 (structured_matrix kind 4) whose backward error is 2e-12; so C_BOUND = 1000.

Steps where that bound reaches 1 cannot fail (a normwise backward error is at most 1); Stats counts them apart as
vacuous: 680 of the 8,524 accepted updates of test_oracle_updates' 300 seeds.

The pivot.  newpiv = xtbl * oldpiv in exact arithmetic, because det(B') = xtbl * det(B).  The update reports
pivot_error = |newpiv - xtbl oldpiv| / (1 + |newpiv|); it must stay below C_BOUND * m * eps * growth * max(1,
max_pivot) (measured at most 0.004 of that without C_BOUND).  Independently, the determinants of fresh factorizations
of B and B' must give det(B') / det(B) = xtbl within C_BOUND * m * eps * cond * growth, cond the larger of the two
fresh factorizations' condest_l * condest_u (measured at most 0.013 of that without C_BOUND); checked where that
bound is below 1.

The backward errors the plain bound of 1e-9 flags are all kind 4 (entries 1e-16 .. 1e4, diagonal down to 1e-12) after
Forrest-Tomlin updates: row etas of 1e10 .. 1e30 and pivots growing to 1e11 .. 1e19, with errors up to 1 where B' is
numerically singular to a fresh factorization.  For them the bound above is vacuous, so the verdict rests on other
evidence.  Seeds 18, 32, 46 and 74 of the first exploration of this (kind 4, default tunables, 1e-8 .. 1.4e-6 after 2 ..
37 updates) reach max_eta 3.4e22, 7.5e15, 8.5e12 and 7.9e12 and max_pivot 2.4e16, 1.7e12, 2.1e9 and 6.5e15, while a
fresh factorization of the same B' solves to 3.7e-19, 2.2e-19, 8.2e-20 and 3.0e-22 and the update's pivot_error stays
at 1.2e-14, 4.7e-12, 0 and 1.5e-16; along each run the error grows step by step with the etas, eps * growth being far
above what is seen.  That is the growth the algorithm allows, not a defect; the defects that were tried on purpose
(an eta entry or a reach entry dropped) fail the bound on steps where it is not vacuous.  droptol is capped at 1e-12
because solve_for_update drops spike entries below droptol by design: droptol = 1e-6 perturbs the entering column by
up to 1e-6 and gives backward errors of that size on well-conditioned bases (4e-7 measured; they vanish at droptol
1e-12)."""
import numpy as np
import scipy.sparse as sp

from blu_b200 import gen
from oracle_lib import Oracle
from parity import SPARSE_STATS, _csc, draw_tunables, structured_matrix
from subset_cases import layout

EPS = np.finfo(np.float64).eps
BRANCHES = ("ft", "sym", "unsym", "refused")
C_BOUND = 1000.0
# the getters an update changes, compared bit for bit between the oracle and a device object after every step
STEP_STATS = [n for n in SPARSE_STATS if n != "update_cost"]


def backward_error(B, x, b):
    """normwise backward error ||B x - b||_inf / (||B||_inf ||x||_inf + ||b||_inf), accumulated in long double"""
    Bl = np.asarray(B, dtype=np.longdouble)
    r = Bl @ np.asarray(x, dtype=np.longdouble) - np.asarray(b, dtype=np.longdouble)
    den = np.abs(Bl).sum(1).max() * np.abs(np.asarray(x, np.longdouble)).max() + np.abs(np.asarray(b, np.longdouble)).max()
    return float(np.abs(r).max() / den) if den > 0 else float(np.abs(r).max())


def draw_case(seed, mmin=8, mmax=120):
    """m, structure (structured_matrix kinds 0..5 or gen.basis as kind 6), tunables (default on even seeds, else
    draw_tunables with droptol capped at 1e-12) and the case's random stream"""
    rng = np.random.default_rng(seed)
    m = int(rng.integers(mmin, mmax + 1))
    kind = seed % 7
    cp, ri, v = structured_matrix(kind, m, rng) if kind < 6 else gen.basis(seed, m, m // 3, 3.0)
    t = draw_tunables(seed) if seed % 2 else {}
    if "droptol" in t:
        t["droptol"] = min(t["droptol"], 1e-12)
    B = sp.csc_matrix((v, ri, cp), shape=(m, m)).toarray()
    return m, kind, B, t, rng


def csc_of(B):
    return _csc(sp.csc_matrix(B))


def fresh_oracle(B, t):
    """a fresh oracle factorization of the explicit B with the tunables t: (status, oracle)"""
    m = B.shape[0]
    cp, ri, v = csc_of(B)
    o = Oracle(m, 400 * len(v) + 2000)
    for k, x in t.items():
        o.set_param(k, x)
    return o.factorize(cp[:-1], cp[1:], ri, v), o


def constructed_column(factors, m, rng):
    """From fresh factors B[rowperm, colperm] = L U: an entering column a = B[:, colperm] U^{-1} e_t' (column t' of L,
    rows mapped back through rowperm) and a leaving position j = colperm[t] with U[t, t'] != 0, t < t'.  Its spike
    L^{-1} a is e_t' exactly (the forward solve cancels every other entry to 0.0), so it lacks the diagonal of row t and
    the update takes the BFS / unsymmetric-permutation path.  None if U is diagonal."""
    rp, cpm = factors["rowperm"], factors["colperm"]
    U = sp.csc_matrix((factors["u_value"], factors["u_rowidx"], factors["u_colptr"]), shape=(m, m)).tocoo()
    off = np.flatnonzero((U.row < U.col) & (U.data != 0))
    if len(off) == 0:
        return None
    e = off[int(rng.integers(len(off)))]
    t, tp = int(U.row[e]), int(U.col[e])
    L = sp.csc_matrix((factors["l_value"], factors["l_rowidx"], factors["l_colptr"]), shape=(m, m))
    lo, hi = L.indptr[tp], L.indptr[tp + 1]
    rows, vals = L.indices[lo:hi], L.data[lo:hi]
    a = np.zeros(m)
    a[rp[rows]] = vals
    a[rp[tp]] = 1.0
    idx = np.flatnonzero(a)
    return idx, a[idx], int(cpm[t])


def random_column(m, rng, nz_range=(1, 5)):
    nz = int(rng.integers(*nz_range))
    idx = np.sort(rng.choice(m, nz, replace=False))
    return idx, rng.uniform(-1, 1, nz)


def leaving_position(lhs, rng, zero_rate):
    """argmax |lhs| half of the time, else a random entry with |lhs| > 1e-3 max; with probability zero_rate a
    position where lhs is exactly zero (the update must refuse it).  None if lhs is zero."""
    a = np.abs(lhs)
    if a.max() == 0:
        return None
    if rng.random() < zero_rate and (a == 0).any():
        z = np.flatnonzero(a == 0)
        return int(z[rng.integers(len(z))])
    if rng.random() < 0.5:
        return int(np.argmax(a))
    cand = np.flatnonzero(a > 1e-3 * a.max())
    return int(cand[rng.integers(len(cand))])


class Stats:
    """branch counts and the worst ratio of the bound over a run of cases.  A step whose bound is 1 or more cannot
    fail (a normwise backward error is at most 1): it is counted in `vacuous`, not in `steps`."""

    def __init__(self):
        self.count = {b: 0 for b in BRANCHES}
        self.count.update(realloc=0, singular_basis=0)
        self.worst_ratio = 0.0
        self.worst_eta = {b: 0.0 for b in ("ft", "sym", "unsym")}
        self.steps = 0
        self.vacuous = 0
        self.det_checked = 0

    def merge_ratio(self, branch, eta, ratio, bound):
        if bound >= 1.0:
            self.vacuous += 1
            return
        self.worst_ratio = max(self.worst_ratio, ratio)
        self.worst_eta[branch] = max(self.worst_eta.get(branch, 0.0), eta)
        self.steps += 1

    def __str__(self):
        return (f"branches {self.count}, checked steps {self.steps}, steps with a vacuous bound {self.vacuous}, "
                f"determinant ratios checked {self.det_checked}, worst ratio to the bound {self.worst_ratio:.3g}, "
                f"worst backward error per branch " + ", ".join(f"{k} {v:.2e}" for k, v in self.worst_eta.items()))


def classify(before, after, status):
    if status == -6:
        return "refused"
    if status == 1:
        return "realloc"
    assert status == 0, status
    if after["nforrest_total"] > before["nforrest_total"]:
        return "ft"
    if after["nsymperm_total"] > before["nsymperm_total"]:
        return "sym"
    return "unsym"


def log_det(o):
    """(sign, log|det|) of the basis a fresh oracle factorization holds: B[rowperm, colperm] = L U with unit L"""
    st, f = o.get_factors()
    assert st == 0
    m = o.m
    U = sp.csc_matrix((f["u_value"], f["u_rowidx"], f["u_colptr"]), shape=(m, m))
    d = U.diagonal()
    sign = np.prod(np.sign(d)) * perm_sign(f["rowperm"]) * perm_sign(f["colperm"])
    return sign, float(np.sum(np.log(np.abs(d))))


def perm_sign(p):
    p, seen, s = np.asarray(p), np.zeros(len(p), bool), 1
    for i in range(len(p)):
        if not seen[i]:
            n, j = 0, i
            while not seen[j]:
                seen[j] = True
                j = p[j]
                n += 1
            s *= -1 if n % 2 == 0 else 1
    return s


def check_step(info, solve_dense, solve_sparse, B, a, j, t, branch, before, m, seed, stats, what, xtbl=None, fo_prev=None):
    """The checks of one accepted update against the explicit B' (= B with column j replaced by a).  info(name) and
    the solve callables belong to the object under test; the solves return x as a dense float64 array.  With xtbl
    and fo_prev (a fresh factorization of B before the update): det(B') = xtbl det(B), from the two fresh
    factorizations, and the object's pivot_error.  Returns the fresh factorization of B' (None if it is singular)."""
    nupdate, nforrest = info("nupdate"), info("nforrest")
    assert nupdate == before["nupdate"] + 1, (what, nupdate, before["nupdate"])
    assert nforrest <= nupdate, (what, nforrest, nupdate)
    if branch == "ft":
        assert info("r_nz") >= before["r_nz"], (what, "r_nz fell across a Forrest-Tomlin update")
    else:
        assert info("r_nz") == before["r_nz"] and nforrest == before["nforrest"], what
    rng = np.random.default_rng(seed)
    b = rng.uniform(-1, 1, m)
    st, fo = fresh_oracle(B, t)
    eta_fresh = 0.0
    if st == 0:
        for tr, M in (("N", B), ("T", B.T)):
            eta_fresh = max(eta_fresh, backward_error(M, fo.solve_dense(b, tr)[1], b))
    else:
        eta_fresh = np.inf        # B' numerically singular for a fresh factorization: nothing to compare with
    eta = 0.0
    for tr, M in (("N", B), ("T", B.T)):
        eta = max(eta, backward_error(M, solve_dense(b, tr), b))
    x = solve_dense(a, "N")
    eta = max(eta, backward_error(B, x, a))
    si, sv = gen.sparse_rhs(seed + 1, m, min(m, 3))
    bs = np.zeros(m)
    bs[si] = sv
    for tr, M in (("N", B), ("T", B.T)):
        eta = max(eta, backward_error(M, solve_sparse(si, sv, tr), bs))
    growth = (1.0 + info("max_eta")) * max(1.0, info("max_pivot") / np.abs(B).max())
    ratio = eta / (max(eta_fresh, m * EPS) * growth)
    assert ratio <= C_BOUND, (what, branch, eta, eta_fresh, growth)
    stats.merge_ratio(branch, eta, ratio, C_BOUND * max(eta_fresh, m * EPS) * growth)
    # B'^{-1} a = e_j: where the update made no growth the entering column must solve to the unit vector
    if growth < 1e3 and eta_fresh < 1e-12:
        ej = np.zeros(m)
        ej[j] = 1.0
        cond = fo.info("condest_l") * fo.info("condest_u")
        assert np.abs(x - ej).max() <= C_BOUND * m * EPS * growth * max(cond, 1.0), (what, np.abs(x - ej).max(), cond)
    # the pivot: newpiv = xtbl * oldpiv, as det(B') = xtbl * det(B).  The update reports how far apart the two are
    # (pivot_error); the determinants of two fresh factorizations tell whether xtbl itself is right.
    pe = info("pivot_error")
    assert pe <= C_BOUND * m * EPS * growth * max(1.0, info("max_pivot")), (what, branch, pe, growth)
    if xtbl is not None and fo_prev is not None and st == 0:
        s0, l0 = log_det(fo_prev)
        s1, l1 = log_det(fo)
        cond = max(fo_prev.info("condest_l") * fo_prev.info("condest_u"), fo.info("condest_l") * fo.info("condest_u"))
        bound = C_BOUND * m * EPS * cond * growth
        if bound < 1.0:
            dev = abs(s1 * s0 * np.sign(xtbl) * np.exp(l1 - l0 - np.log(abs(xtbl))) - 1.0)
            assert dev <= bound, (what, branch, dev, cond, growth)
            stats.det_checked += 1
    return fo if st == 0 else None


def single_case(seed, make_objs, nsteps=40, construct_rate=0.5, zero_rate=0.04, stats=None, mmin=8, mmax=120,
                case=None):
    """One seeded case on the objects make_objs(m, nnz, tunables) returns: objs[0] is the oracle, every other object
    must match it bit for bit after every call; the explicit-basis checks run on the last object's own outputs."""
    stats = Stats() if stats is None else stats
    m, kind, B, t, rng = case if case is not None else draw_case(seed, mmin, mmax)
    objs = make_objs(m, int((B != 0).sum()), t)
    dev = objs[-1]
    need_factor, since = True, 0
    for it in range(nsteps):
        what = (seed, kind, m, it)
        if need_factor:
            cp, ri, v = csc_of(B)
            sts = [o.factorize(cp[:-1], cp[1:], ri, v) for o in objs]
            assert len(set(sts)) == 1, (what, sts)
            if sts[0] != 0:
                stats.count["singular_basis"] += 1
                return stats
            need_factor, since = False, 0
            fo_prev = fresh_oracle(B, t)[1]
        col = None
        if since == 0 and rng.random() < construct_rate:
            col = constructed_column(objs[0].get_factors()[1], m, rng)
        idx, val, j = col if col is not None else random_column(m, rng) + (None,)
        sts = [o.solve_for_update(len(idx), idx, val, "N", want_solution=1) for o in objs]
        assert len(set(sts)) == 1 and sts[0] == 0, (what, sts)
        same_solution(objs, what)
        lhs = objs[0].lhs.copy()
        if j is None or lhs[j] == 0:
            j = leaving_position(lhs, rng, zero_rate)
            if j is None:
                continue
        sts = [o.solve_for_update(1, np.array([j]), None, "T", want_solution=it % 2) for o in objs]
        assert len(set(sts)) == 1 and sts[0] == 0, (what, sts)
        if it % 2:
            same_solution(objs, what)
        before = {n: dev.info(n) for n in ("nforrest_total", "nsymperm_total", "nupdate", "nforrest", "r_nz")}
        sts = [o.update(lhs[j]) for o in objs]
        assert len(set(sts)) == 1, (what, sts)
        for o in objs[1:]:
            for n in STEP_STATS:
                assert o.info(n) == objs[0].info(n), (what, n, o.info(n), objs[0].info(n))
        after = {n: dev.info(n) for n in ("nforrest_total", "nsymperm_total")}
        branch = classify(before, after, sts[0])
        stats.count[branch] += 1
        if branch in ("refused", "realloc"):
            need_factor = True
            continue
        a = np.zeros(m)
        a[idx] = val
        B[:, j] = a
        since += 1

        def dense(b, tr):
            xs = [o.solve_dense(b, tr) for o in objs]
            assert all(s == 0 for s, _ in xs) and all(np.array_equal(x, xs[0][1]) for _, x in xs), what
            return xs[-1][1]

        def sparse(si, sv, tr):
            assert all(o.solve_sparse(len(si), si, sv, tr) == 0 for o in objs), what
            same_solution(objs, what)
            return dev.lhs.copy()

        fo_prev = check_step(dev.info, dense, sparse, B, a, j, t, branch, before, m, seed * 1000 + it, stats, what,
                             lhs[j], fo_prev)
        if dev.info("nforrest") >= min(m - 1, 30):
            need_factor = True
    return stats


def same_solution(objs, what):
    o = objs[0]
    n = o.nzlhs
    for g in objs[1:]:
        assert g.nzlhs == n, (what, g.nzlhs, n)
        assert np.array_equal(g.ilhs[:n], o.ilhs[:n]) and np.array_equal(g.lhs, o.lhs), what


class Cols:
    """An explicit basis kept as its m columns (index and value arrays), for bases too large to keep dense: products
    with B and B^T accumulate in long double."""

    def __init__(self, cp, ri, v):
        self.m = len(cp) - 1
        self.cols = [(ri[cp[j]:cp[j + 1]].astype(np.int64), v[cp[j]:cp[j + 1]].astype(np.float64)) for j in range(self.m)]
        self._flat = None

    def replace(self, j, col):
        self.cols[j] = col
        self._flat = None

    def flat(self):
        if self._flat is None:
            lens = [len(r) for r, _ in self.cols]
            self._flat = (np.repeat(np.arange(self.m), lens), np.concatenate([r for r, _ in self.cols]),
                          np.concatenate([x for _, x in self.cols]))
        return self._flat

    def csc(self):
        jj, ii, vv = self.flat()
        return np.searchsorted(jj, np.arange(self.m + 1)).astype(np.int64), ii, vv

    def backward_error(self, x, b, trans):
        jj, ii, vv = self.flat()
        prod = vv.astype(np.longdouble) * np.asarray(x, np.longdouble)[ii if trans == "T" else jj]
        r = np.zeros(self.m, np.longdouble)
        np.add.at(r, jj if trans == "T" else ii, prod)
        r -= np.asarray(b, np.longdouble)
        norm = np.zeros(self.m, np.longdouble)
        np.add.at(norm, jj if trans == "T" else ii, np.abs(vv).astype(np.longdouble))
        den = norm.max() * np.abs(np.asarray(x, np.longdouble)).max() + np.abs(np.asarray(b, np.longdouble)).max()
        return float(np.abs(r).max() / den)

    def absmax(self):
        return np.abs(self.flat()[2]).max()


def batch_rounds(b, oracles, bases, t, rounds, seed, update_dev=None, stats=None, construct_rate=0.3, zero_rate=0.04,
                 run_rate=0.75, fresh=True, dev_only=False, nz_range=(1, 5)):
    """Every basis of the BLUBatch b through `rounds` rounds of basis changes, each basis with its own oracle (bit for
    bit after every call) and its explicit basis (bases[k], a Cols).  Each round a random subset runs (the rest stay
    idle); rounds alternate between update_subset and update_dev with a run mask, update_dev getting its tensors
    through update_dev(array, dtype) (every round with dev_only).  Bases whose update was refused are refactorized through factorize_subset.
    After each round every basis that changed is checked against its explicit B' with the bound of this module, on
    the batch's own dense (solve_dense_multi) and sparse (solve_sparse) solves.  Returns stats; stats.count also
    counts 'realloc_subset' / 'realloc_dev', the update calls inside which the batch grew a store; entering columns
    with more entries (nz_range) give longer spikes, which outgrow the row file sooner."""
    import torch
    stats = Stats() if stats is None else stats
    stats.count.setdefault("realloc_subset", 0)
    stats.count.setdefault("realloc_dev", 0)
    rng = np.random.default_rng(seed)
    n, m = b.nmat, b.m
    since = [0] * n
    refactor = []
    for rd in range(rounds):
        if refactor:
            st, stat = b.factorize_subset(refactor, *layout([bases[k].cols for k in refactor]))
            for r, k in enumerate(refactor):
                cp, ri, v = bases[k].csc()
                assert oracles[k].factorize(cp[:-1], cp[1:], ri, v) == stat[r] == 0, (k, stat[r])
                since[k] = 0
            refactor = []
        sel = [k for k in range(n) if rng.random() < run_rate] or [int(rng.integers(n))]
        cols, fixed_j = {}, {}
        for k in sel:
            c = constructed_column(b.get_factors(k)[1], m, rng) if since[k] == 0 and rng.random() < construct_rate else None
            if c is None:
                cols[k] = random_column(m, rng, nz_range)
            else:
                cols[k] = c[:2]
                fixed_j[k] = c[2]
        st, stat, out = b.solve_for_update_subset(sel, [cols[k] for k in sel], "N", want_solution=1)
        assert st == 0 and (stat == 0).all(), (rd, stat)
        leave, xt = {}, {}
        for r, k in enumerate(sel):
            o = oracles[k]
            assert o.solve_for_update(len(cols[k][0]), cols[k][0], cols[k][1], "N", want_solution=1) == 0
            nz = o.nzlhs
            assert np.array_equal(out[r][0], o.ilhs[:nz]) and np.array_equal(out[r][1], o.lhs[o.ilhs[:nz]]), (rd, k)
            lhs = o.lhs
            j = fixed_j.get(k)
            if j is None or lhs[j] == 0:
                j = leaving_position(lhs, rng, zero_rate)
            if j is not None:
                leave[k], xt[k] = j, lhs[j]
        sel = sorted(leave)
        if not sel:
            continue
        st, stat, _ = b.solve_for_update_subset(sel, [(np.array([leave[k]]), None) for k in sel], "T", want_solution=0)
        assert st == 0 and (stat == 0).all()
        before = {k: {q: b.info(k, q) for q in ("nforrest_total", "nsymperm_total", "nupdate", "nforrest", "r_nz")}
                  for k in sel}
        nr = b.info(0, "nrealloc")
        if update_dev is not None and (dev_only or rd % 2):
            x = np.full(n, np.nan)
            run = np.zeros(n, np.int32)
            for k in sel:
                x[k], run[k] = xt[k], 1
            st, sd = b.update_dev(update_dev(x, torch.float64), run=update_dev(run, torch.int32))
            sd = sd.cpu().numpy()
            ust = [int(sd[k]) for k in sel]
            stats.count["realloc_dev"] += b.info(0, "nrealloc") > nr
        else:
            st, stat = b.update_subset(sel, [xt[k] for k in sel])
            ust = [int(s) for s in stat]
            stats.count["realloc_subset"] += b.info(0, "nrealloc") > nr
        changed = {}
        for r, k in enumerate(sel):
            o = oracles[k]
            assert o.solve_for_update(1, np.array([leave[k]]), None, "T", want_solution=0) == 0
            assert o.update(xt[k]) == ust[r], (rd, k, ust[r])
            for q in STEP_STATS:
                assert b.info(k, q) == o.info(q), (rd, k, q, b.info(k, q), o.info(q))
            after = {q: b.info(k, q) for q in ("nforrest_total", "nsymperm_total")}
            branch = classify(before[k], after, ust[r])
            stats.count[branch] += 1
            if branch == "refused":
                refactor.append(k)
                continue
            bases[k].replace(leave[k], cols[k])
            since[k] += 1
            changed[k] = branch
            if b.info(k, "nforrest") >= min(m - 1, 30):
                refactor.append(k)
        if changed:
            check_batch(b, bases, t, changed, rng, stats, fresh, rd, oracles, before, cols)
    return stats


def check_batch(b, bases, t, changed, rng, stats, fresh, rd, oracles=None, before=None, cols=None):
    """check_step for the bases of a batch in `changed` ({basis: branch}), with one batched call per kind of solve.
    With oracles, every basis' solves must equal its oracle's; with before (the getters before the update), the update
    counters are checked; with cols (the entering columns), the second dense right-hand side of a basis is its
    entering column, else a random vector."""
    n, m = b.nmat, b.m
    rhs = rng.uniform(-1, 1, (n, 2, m))
    for k in changed if cols is not None else ():
        rhs[k, 1] = 0.0
        rhs[k, 1, cols[k][0]] = cols[k][1]
    xs = {}
    for tr in "NT":
        st, x, stat = b.solve_dense_multi(rhs, tr)
        xs[tr] = x
    sp_rhs = [gen.sparse_rhs(int(rng.integers(1 << 30)), m, min(m, 3)) for _ in range(n)]
    sps = {}
    for tr in "NT":
        st, out, ustat = b.solve_sparse([[sp_rhs[k]] for k in range(n)], tr)
        sps[tr] = out
    if oracles is not None:
        # the oracles run the same solves on every basis: solves compact the pivot sequence and count flops
        xo = {tr: [[o.solve_dense(rhs[k, r], tr)[1] for r in range(2)] for k, o in enumerate(oracles)] for tr in "NT"}
        for tr in "NT":
            for k, o in enumerate(oracles):
                assert o.solve_sparse(len(sp_rhs[k][0]), sp_rhs[k][0], sp_rhs[k][1], tr) == 0
                nz = o.nzlhs
                assert np.array_equal(sps[tr][k][0][0], o.ilhs[:nz]) and np.array_equal(sps[tr][k][0][1], o.lhs[o.ilhs[:nz]]), (rd, k)
    for k, branch in changed.items():
        B = bases[k]
        what = (rd, k)
        if before is not None:
            nupdate, nforrest = b.info(k, "nupdate"), b.info(k, "nforrest")
            assert nupdate == before[k]["nupdate"] + 1 and nforrest <= nupdate, what
            if branch == "ft":
                assert b.info(k, "r_nz") >= before[k]["r_nz"], what
        if oracles is not None:
            for tr in "NT":
                assert np.array_equal(xs[tr][k, 0], xo[tr][k][0]) and np.array_equal(xs[tr][k, 1], xo[tr][k][1]), (what, tr)
        eta = max(B.backward_error(xs["N"][k, 0], rhs[k, 0], "N"), B.backward_error(xs["T"][k, 0], rhs[k, 0], "T"),
                  B.backward_error(xs["N"][k, 1], rhs[k, 1], "N"), B.backward_error(xs["T"][k, 1], rhs[k, 1], "T"))
        for tr in "NT":
            il, xl = sps[tr][k][0]
            x = np.zeros(m)
            x[il] = xl
            bs = np.zeros(m)
            bs[sp_rhs[k][0]] = sp_rhs[k][1]
            eta = max(eta, B.backward_error(x, bs, tr))
        growth = (1.0 + b.info(k, "max_eta")) * max(1.0, b.info(k, "max_pivot") / B.absmax())
        floor = m * EPS
        if eta > C_BOUND * floor * growth and fresh:
            cp, ri, v = B.csc()
            fo = Oracle(m, 40 * len(v) + 2000)
            for a, x in t.items():
                fo.set_param(a, x)
            if fo.factorize(cp[:-1], cp[1:], ri, v) != 0:
                continue
            for tr in "NT":
                floor = max(floor, B.backward_error(fo.solve_dense(rhs[k, 0], tr)[1], rhs[k, 0], tr))
        ratio = eta / (floor * growth)
        assert ratio <= C_BOUND, (what, eta, floor, growth)
        stats.merge_ratio(branch, eta, ratio, C_BOUND * floor * growth)


def check_maxvolume(b, pools, status, basis, t, rng, stats):
    """After batch maxvolume: rebuild each basis that ended OK from the returned `basis` (its pool's columns) and check
    the batch's later dense and sparse solves against that explicit basis with the bound of this module."""
    bases, ok = [], {}
    for k, p in enumerate(pools):
        cols = [(p.a_i[p.a_p[c]:p.a_p[c + 1]], p.a_x[p.a_p[c]:p.a_p[c + 1]]) for c in basis[k]]
        cp = np.concatenate([[0], np.cumsum([len(r) for r, _ in cols])]).astype(np.int64)
        bases.append(Cols(cp, np.concatenate([r for r, _ in cols]), np.concatenate([x for _, x in cols])))
        if status[k] == 0:
            ok[k] = "maxvolume"
    check_batch(b, bases, t, ok, rng, stats, True, "maxvolume")
    return len(ok)
