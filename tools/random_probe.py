"""Differential probe: random small configurations of the retirement and Deaton models against the compiled reference
(or, without it, the stored outputs of tests/golden/stored.npz)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
from egdst_b200 import examples
from oracle import ref
from tests.parity import solution_errors
from tests.goldens import sims_errors
from tests.oracles import oracle_for

def draw(rng, kinds=("retirement", "deaton")):
    kind = rng.choice(list(kinds))
    T = int(rng.integers(3, 13)); n = int(rng.integers(20, 601)); ny = int(rng.integers(1, 13))
    a0 = float(rng.choice([-5.0, -1.0, 0.0])); mmax = float(rng.uniform(8, 20))
    if kind == "retirement":
        kw = dict(T=T, ngridm=n, ngridmax=2 * n + 50, nthrhmax=max(n, 20), ny=ny, interest=float(rng.uniform(0, 0.03)),
                  duw=float(rng.uniform(0.2, 0.8)), wage=float(rng.uniform(0.8, 1.5)), a0=a0, mmax=mmax)
        return kind, kw, examples.retirement(**kw)
    if kind == "retirement_large":  # wide launch shapes: several compaction / envelope chunks, long node loops
        n = int(rng.integers(600, 6001))
        kw = dict(T=int(rng.integers(3, 9)), ngridm=n, ngridmax=2 * n + 50, nthrhmax=n, ny=int(rng.integers(4, 41)), interest=float(rng.uniform(0, 0.02)),
                  duw=float(rng.uniform(0.2, 0.8)), wage=float(rng.uniform(0.8, 1.5)), a0=a0, mmax=mmax)
        return kind, kw, examples.retirement(**kw)
    if kind == "occ3":      # three occupations, CRRA utility, decision-dependent shock variance; parameters set after
        m = examples.occ3(ngridm=int(rng.integers(20, 120)), ngridmax=1000, ny=max(ny, 2), T=int(rng.integers(3, 15)))  # the reference itself crashes on larger occ3 grids
        vals = dict(crra=float(rng.uniform(1.1, 2.0)), coefleisure=float(rng.uniform(0.05, 0.4)), wagegap=float(rng.uniform(1.1, 1.6)),
                    entrkap=float(rng.uniform(0.3, 0.7)), interest=float(rng.uniform(0.0, 0.05)))
        for k, v in vals.items():
            m.setparam(k, v)
        return kind, vals, m
    if kind == "model2":    # lecture model: two labour-market states (absorbing retirement), lognormal returns
        kw = dict(T=int(rng.integers(2, 9)), ngridm=int(rng.integers(20, 400)), nquad=max(ny, 2), mmax=float(rng.uniform(50, 150)),
                  cc=0.0, df=float(rng.uniform(0.9, 1.0)), rho=0.0, r=float(rng.uniform(0.0, 0.04)), sigma=float(rng.uniform(0.05, 0.4)),
                  duw=float(rng.uniform(0.5, 2.0)), wage=float(rng.uniform(2.0, 8.0)))
        return kind, kw, examples.model2(**kw)
    if kind == "humancapital":  # continuous state: wage scales with human capital, z' = depr*z + gain*work
        kw = dict(T=int(rng.integers(3, 12)), ngridm=int(rng.integers(20, 300)), ny=max(ny, 2), interest=float(rng.uniform(0.0, 0.04)),
                  duw=float(rng.uniform(0.1, 0.8)), wage=float(rng.uniform(0.6, 1.5)), depr=float(rng.uniform(0.8, 0.98)), gain=float(rng.uniform(0.02, 0.25)))
        return kind, kw, examples.humancapital(**kw)
    # shock strings stay the shipped ones: they are part of the generated source, and the reference-built checker
    # (oracle/_ref) only exists for the shipped images where /root/reference is absent
    kw = dict(T=T, ngridm=n, ngridmax=2 * n + 50, ny=max(ny, 2), interest=float(rng.uniform(0, 0.03)), income=float(rng.uniform(0.7, 1.6)),
              a0=a0 * 5, mmax=mmax * 5)
    return kind, kw, examples.deaton2(**kw)

def main(seed0, count, kinds=("retirement", "deaton")):
    bad = 0
    for seed in range(seed0, seed0 + count):
        rng = np.random.default_rng(seed)
        kind, kw, m = draw(rng, kinds)
        m.compile(); m.solve()
        st = m._solution.status()
        try:
            r = oracle_for(m); Mr, Dr = r.solve(); rerr = None
        except Exception as e:  # the reference aborts (mexErrMsgTxt)
            rerr = str(e).splitlines()[0][:80]
        if rerr is not None or st[0]:
            print(seed, kind, "status", st, "reference:", rerr, kw, flush=True)
            bad += (rerr is None) != (st[0] == 0)
            continue
        e = solution_errors(m.M, m.D, Mr, Dr)
        nsim = 64
        cont = any(v["continuous"] for v in m.s)  # the reference addresses only first-grid-point initial cells correctly
        init = np.column_stack([np.ones(nsim) if cont else np.full(nsim, float(m.nst)), m.a0 + (m.mmax - m.a0) * (0.02 + 0.6 * rng.random(nsim))])
        skip = [3] if cont else []            # and leaves the value column unassigned (DESIGN 6a)
        rs = rng.random(4 * nsim * m.nt)
        m.sim(init, "own_shocks", randstream=rs)
        sr = r.simulate(Mr, Dr, init, rs, 0)
        se = sims_errors(m.sims, sr, skip)
        # noise floor of the configuration: the reference against itself, built with contraction allowed (oracle/ref.py
        # variant "noise").  Consumption next to the borrowing limit makes log(c) amplify last-bit differences of the
        # math library; such configurations are held to twice what the reference's own two builds differ by.
        # (the stored outputs of a machine without the reference have no noise floor: held to the base tolerances)
        if r.kind == "reference":
            rn = ref.Reference(m, variant="noise"); Mn, Dn = rn.solve()
            en = solution_errors(Mn, Dn, Mr, Dr)
            sn = sims_errors(rn.simulate(Mn, Dn, init, rs, 0), sr, skip)
        else:
            en, sn = {"C": 0.0, "V": 0.0, "TH": 0.0, "rowdiff": 0}, {"discrete_mismatch": 0, "max": 0.0}
        tol = lambda k, base: max(base, 2.0 * en[k])  # noqa: E731
        ok = (e["C"] < tol("C", 1e-9) and e["V"] < tol("V", 1e-9) and e["TH"] < tol("TH", 1e-8) and e["Dseq"] and e["rowdiff"] <= en["rowdiff"]
              and se["nan_mismatch"] == 0 and se["discrete_mismatch"] <= sn["discrete_mismatch"] and se["max"] < max(1e-9, 2.0 * sn["max"]))
        if not ok:
            bad += 1
            print(seed, kind, "MISMATCH", {k: v for k, v in e.items() if k != "where"}, se, "noise:", {k: v for k, v in en.items() if k != "where"}, sn, kw, flush=True)
    print("checked", count, "bad", bad)
    return bad

if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 0, int(sys.argv[2]) if len(sys.argv) > 2 else 40,
         tuple(sys.argv[3].split(",")) if len(sys.argv) > 3 else ("retirement", "deaton"))
