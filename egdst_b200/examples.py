"""The reference's example models, transcribed property-for-property.

Sources: egdst_examples/model_{deaton1,deaton2,retirement1,retirement2,occ3,cake1,cake2}.m and
lecture_code/model2.m.  Only the model definitions are transcribed (the ``.m`` scripts also
compile/solve/plot); sizes and parameters can be overridden by keyword, which is how the scaled
BASELINE configs (SURVEY 8(d): S1, S1b, S5) are built.
"""
from __future__ import annotations

from .model import EgdstModel


def _common(m: EgdstModel, T, mmax, ngridmax, ngridm, nthrhmax, ny):
    m.t0 = 1
    m.T = T
    m.mmax = mmax
    m.ngridmax = ngridmax
    m.ngridm = ngridm
    m.nthrhmax = nthrhmax
    m.ny = ny


def _singleton(m: EgdstModel):
    m.s = ("Singleton state", [0, "dummy state"])
    m.trpr = ("true", [[1]])
    m.feasible = ("defaultfeasible", True)


def _log_utility(m: EgdstModel, util="log(consumption)"):
    m.u = ("utility", util)
    m.u = ("marginal", "1/consumption")
    m.u = ("marginalinverse", "1/mutility")
    m.u = ("extrap", "log(x)")


def deaton(label="deaton1", a0=0.0, sigma="0", mu="0", mmax=50, ny=2, T=25, ngridm=100, ngridmax=1000,
           interest=0.01, income=1.25, shocktype="lognormal") -> EgdstModel:
    """egdst_examples/model_deaton1.m:6-46 (and model_deaton2.m with a0=-25, sigma=0.75, mmax=100, ny=10)."""
    m = EgdstModel(label)
    _common(m, T, mmax, ngridmax, ngridm, 10, ny)
    _singleton(m)
    m.d = ("Dummy decision", [0, "dummy decision"])
    m.choiceset = ("defaultallow", True)
    _log_utility(m)
    m.budget = ("cashinhand", "savings*(1+interest)+income_level")
    m.budget = ("marginal", "1+interest")
    m.discount = "1/(1+interest)"
    m.param = ("interest", "return on savings", interest)
    m.eq = ("income_level", "Realized income", "income*shock", "next")
    m.param = ("income", "income (times multiplicator shock)", income)
    m.a0 = a0
    m.shock = shocktype
    m.shock = ("sigma", sigma)
    m.shock = ("mu", mu)
    return m


def deaton_meanstest(penalty=4.0, cut=2.0, **kw) -> EgdstModel:
    """Deaton model whose cash-in-hand drops by ``penalty`` once savings exceed ``cut`` (a means test).  Not shipped by the
    reference: next period's cash is then non-monotone in savings, which is what makes the zero-consumption signal fire
    AFTER the seed stage of the savings grid (egdst_solver.c:1080-1099) and the grid fold back with one decision."""
    args = dict(label="deaton_mt", a0=0.0, sigma="0.25", mu="-0.5*sigma*sigma", mmax=20, ny=5, T=6, ngridm=80, ngridmax=400)
    args.update(kw)
    label = args.pop("label")
    m = deaton(label, **args)
    m.budget = ("cashinhand", "savings*(1+interest)+income_level-%r*(savings>%r)" % (float(penalty), float(cut)))
    m.nthrhmax = 200
    return m


def deaton1(**kw) -> EgdstModel:
    return deaton("deaton1", **kw)


def deaton_normal(**kw) -> EgdstModel:
    """Deaton model with normally distributed income multiplier (DISTRIB=2): not shipped by the reference, used to
    cover the normal-shock code path (egdst_lib.c:66-101)."""
    args = dict(label="deaton_normal", a0=0.0, sigma="0.15", mu="1.0", mmax=60, ny=12, T=15, ngridm=300, ngridmax=1000, shocktype="normal")
    args.update(kw)
    label = args.pop("label")
    return deaton(label, **args)


def deaton2(**kw) -> EgdstModel:
    args = dict(a0=-25.0, sigma="0.75", mu="-0.5*sigma*sigma", mmax=100, ny=10)
    args.update(kw)
    return deaton("deaton2", **args)


def retirement(label="retire2", sigma="0.25", mu="-0.5*sigma*sigma", T=25, ngridm=100, ngridmax=1000, nthrhmax=10,
               ny=10, interest=0.045, mmax=10, a0=-5.0, duw=0.5, wage=1.05) -> EgdstModel:
    """egdst_examples/model_retirement2.m:6-46 (model_retirement1.m is the sigma=0 case)."""
    m = EgdstModel(label)
    _common(m, T, mmax, ngridmax, ngridm, nthrhmax, ny)
    _singleton(m)
    m.d = ("Labour supply", [0, "retire", 1, "work"])
    m.choiceset = ("defaultallow", True)
    m.u = ("utility", "log(consumption)+duw*(id==0)")
    m.param = ("duw", "disutility of work", duw)
    m.u = ("marginal", "1/consumption")
    m.u = ("marginalinverse", "1/mutility")
    m.u = ("extrap", "log(x)")
    m.budget = ("cashinhand", "savings+wage_income*(id!=0)")
    m.budget = ("marginal", "1+interest")
    m.discount = "1/(1+interest)"
    m.param = ("interest", "return on savings", interest)
    m.eq = ("wage_income", "Realized wage income", "wage*shock", "next")
    m.param = ("wage", "wage (times multiplicator shock)", wage)
    m.a0 = a0
    m.shock = "lognormal"
    m.shock = ("sigma", sigma)
    m.shock = ("mu", mu)
    return m


def retirement1(**kw) -> EgdstModel:
    args = dict(label="retire1", sigma="0", mu="0")
    args.update(kw)
    return retirement(**args)


def retirement2(**kw) -> EgdstModel:
    return retirement(**kw)


def retirement2_scaled(T=50, ngridm=10000, ny=100, interest=0.02) -> EgdstModel:
    """S1 of SURVEY 8(d): retirement2 at 10k grid x 100 nodes x 50 periods; ``interest=0.02`` because the
    reference itself aborts at this size with the shipped 0.045 (SURVEY 0, fact 7); nthrhmax=ngridm (fact 8)."""
    return retirement(T=T, ngridm=ngridm, ngridmax=2 * ngridm, nthrhmax=ngridm, ny=ny, interest=interest)


def occ3(ngridm=50, ngridmax=100, ny=10, T=40) -> EgdstModel:
    """egdst_examples/model_occ3.m:3-44."""
    m = EgdstModel("occ3")
    m.t0 = 0
    m.T = T
    m.s = ("Dummy state", [0, "dummy"])
    m.trpr = ("true", [[1]])
    m.feasible = ("defaultfeasible", True)
    m.d = ("Occupational choice", [0, "public sector (lower pay, secure)", 1, "private sector (hight pay, less secure)",
                                   2, "entrepreneurship"])
    m.choiceset = ("defaultallow", True)
    m.u = ("utility", "(pow(consumption,1-crra)-1)/(1-crra) - coefleisure*disutility[1][(int)dc1+1]")
    m.coef = ("disutility", "Disutility of work", [0.0, 1.0, 0.75])
    m.param = ("crra", "CRRA coefficient in utility", 1.2)
    m.param = ("coefleisure", "Weight with leisure in utility", 0.2)
    m.u = ("marginal", "pow(consumption,-crra)")
    m.u = ("marginalinverse", "pow(mutility,-1/crra)")
    m.u = ("extrap", "pow(x,1-crra)")
    m.discount = "0.93"
    m.shock = "lognormal"
    m.shock = ("sigma", "sigs[1][(int)dc1+1]")
    m.coef = ("sigs", "Sigmas for different occupations", [0.15, 0.35, 0.75])
    m.shock = ("mu", "-0.5*sigs[1][(int)dc1+1]*sigs[1][(int)dc1+1]")
    m.eq = ("wage1", "Realized wage in the public sector", "max(ssinc,shock*0.5)", "next")
    m.eq = ("wage2", "Realized wage in the private sector", "max(ssinc,shock*0.5*wagegap)", "next")
    m.param = ("ssinc", "Guaranteed social security income", 0.01)
    m.param = ("wagegap", "Wage gap between public and private sector", 1.35)
    m.eq = ("entrep", "Entrepreneurial income (realized)", "max(ssinc,log(savings+1)*entrkap*shock)", "next")
    m.param = ("entrkap", "Return on capital", 0.56)
    m.budget = ("cashinhand", "savings*(1+interest)+(dc1==0)*wage1+(dc1==1)*wage2+(dc1==2)*entrep")
    m.budget = ("marginal", "1+interest+(dc1==2)*max(0,entrkap*shock/(savings+1))")
    m.param = ("interest", "return on savings", 0.05)
    m.a0 = 0.0
    m.mmax = 5
    m.ngridm = ngridm
    m.ngridmax = ngridmax
    m.nthrhmax = 100
    m.ny = ny
    return m


def cake(label="cake1", discount="1", T=25, ngridm=100) -> EgdstModel:
    """egdst_examples/model_cake1.m:6-41 (cake2: discount='.75')."""
    m = EgdstModel(label)
    _common(m, T, 10, 1000, ngridm, 10, 2)
    _singleton(m)
    m.d = ("Dummy decision", [0, "dummy decision"])
    m.choiceset = ("defaultallow", True)
    _log_utility(m)
    m.budget = ("cashinhand", "savings")
    m.budget = ("marginal", "1")
    m.discount = discount
    m.a0 = 0.0
    m.shock = "normal"
    m.shock = ("sigma", "0")
    m.shock = ("mu", "0")
    return m


def cake1(**kw) -> EgdstModel:
    return cake("cake1", "1", **kw)


def cake2(**kw) -> EgdstModel:
    return cake("cake2", ".75", **kw)


def model2(T=3, ngridm=100, nquad=10, mmax=100, cc=0.0, df=1.0, rho=0.0, r=0.0, sigma=0.0, duw=1.0, wage=5.0) -> EgdstModel:
    """lecture_code/model2.m:1-77 -- the only shipped model with more than one state (absorbing retirement)."""
    m = EgdstModel("model2")
    m.t0 = 1
    m.T = T
    m.mmax = mmax
    m.ngridmax = 10 * ngridm
    m.ngridm = ngridm
    m.nthrhmax = ngridm
    m.ny = nquad
    m.a0 = 0.0
    m.s = ("Labour market state", [0, "retired", 1, "working"])
    m.d = ("Retirement decision", [0, "Retirement", 1, "Work"])
    m.feasible = ("defaultfeasible", True)
    m.trpr = ("dc1==0", [[1, 0], [1, 0]])
    m.trpr = ("dc1==1", [[0, 1], [0, 1]])
    m.choiceset = ("defaultallow", True)
    m.choiceset = ("ist==0 && id==1", "Retirement is absorbing")
    m.u = ("utility", "(fabs(rho)<1e-10?log(consumption):(pow(consumption,rho)-1)/rho)  - (id?duw:0.0)")
    m.u = ("marginal", "pow(consumption,rho-1)")
    m.u = ("marginalinverse", "pow(mutility,1/(rho-1))")
    m.param = ("rho", "1-crra parameter", rho)
    m.param = ("duw", "scale parameter for disutility of work", duw)
    m.u = ("extrap", "pow(x,rho)")
    m.budget = ("cashinhand", "savings*(1+r)*shock  + (id?wage:0.0)")
    m.budget = ("marginal", "(1+r)*shock")
    m.param = ("r", "risk free return", r)
    m.discount = "df"
    m.param = ("df", "discount factor", df)
    m.param = ("wage", "Workers wage", wage)
    m.a0 = cc
    m.shock = "lognormal"
    m.shock = ("sigma", "sig")
    m.shock = ("mu", "-sigma*sigma/2")
    m.param = ("sig", "sigma parameter in lognormal return", sigma)
    return m


def humancapital(T=12, ngridm=100, ngridmax=1000, ny=8, nz=5, nthrhmax=20, sigma="0.2", interest=0.03, duw=0.4, wage=1.0,
                 depr=0.9, gain=0.15, zlim=(0.4, 1.6), mmax=20.0, a0=0.0, health=False, nh=3) -> EgdstModel:
    """Work/retire model whose wage scales with a CONTINUOUS human-capital state z: z' = depr*z + gain*work, on a
    uniform grid of ``nz`` points.  Not shipped by the reference (none of its examples has a continuous state); it
    exercises the motion-rule code path (egdstmodel.m:629-648 and :1000-1004, compile.m:527-537 and :556-575,
    egdst_simulator.c:309-365).  ``health=True`` adds a second continuous state (worn down by work, valued in utility),
    so that the simulator mixes four grid cells."""
    m = EgdstModel("humancap2" if health else "humancap")
    _common(m, T, mmax, ngridmax, ngridm, nthrhmax, ny)
    m.s = ("Human capital", list(zlim), nz)
    m.trpr = (1, "true", "depr*st1+gain*dc1")
    if health:
        m.s = ("Health", [0.5, 1.0], nh)
        m.trpr = (2, "dc1==1", "0.93*st2+0.05")
        m.trpr = (2, "dc1==0", "0.93*st2+0.07")
    m.feasible = ("defaultfeasible", True)
    m.d = ("Labour supply", [0, "retire", 1, "work"])
    m.choiceset = ("defaultallow", True)
    m.u = ("utility", "log(consumption)+duw*(dc1==0)" + ("+0.3*log(st2)" if health else ""))
    m.param = ("duw", "disutility of work", duw)
    m.u = ("marginal", "1/consumption")
    m.u = ("marginalinverse", "1/mutility")
    m.u = ("extrap", "log(x)")
    m.budget = ("cashinhand", "savings*(1+interest)+wage_income*dc1")
    m.budget = ("marginal", "1+interest")
    m.discount = "1/(1+interest)"
    m.param = ("interest", "return on savings", interest)
    m.eq = ("wage_income", "Realized wage income", "wage*st1*shock", "next")
    m.param = ("wage", "wage per unit of human capital", wage)
    m.param = ("depr", "human capital carried over", depr)
    m.param = ("gain", "human capital gained by working", gain)
    m.a0 = a0
    m.shock = "lognormal"
    m.shock = ("sigma", sigma)
    m.shock = ("mu", "-0.5*sigma*sigma")
    return m


def retirement_mortal(**kw) -> EgdstModel:
    """retirement2 with age-dependent mortality: survival enters only the simulator (egdst_simulator.c:261-265: a
    death event ends the agent's record, the remaining rows stay NaN).  Not shipped by the reference -- none of its
    examples sets ``survival`` -- it exercises the death path and the NaN bookkeeping of the moment accumulators."""
    m = retirement(label="retire_mortal", **kw)
    m.survival = "0.995-0.002*age"
    return m


def retirement_jobloss(T=15, ngridm=100, ngridmax=1000, nthrhmax=50, ny=8, interest=0.02, mmax=12.0, a0=0.0, duw=0.4, wage=1.0,
                       sigma="0.3") -> EgdstModel:
    """Work/retire model with an employment state whose transition probabilities depend on the realised shock (a low
    draw costs the job, a high one finds one).  Not shipped by the reference: it takes the branch none of the shipped
    examples takes -- optim_TRPRnoSH = 0: trpr evaluated per quadrature node and per simulated draw
    (egdst_solver.c:507-530, egdst_simulator.c:280-290), no per-CTA shock table.  (optim_MUnoD = 0 cannot be reached:
    compile.m rejects a marginal utility that depends on the decision as "not yet implemented".)"""
    m = EgdstModel("jobloss")
    _common(m, T, mmax, ngridmax, ngridm, nthrhmax, ny)
    m.s = ("Employment", [0, "unemployed", 1, "employed"])
    m.trpr = ("true", [["1-0.5*(shock>1.0)", "0.5*(shock>1.0)"], ["0.3*(shock<0.7)", "1-0.3*(shock<0.7)"]])
    m.feasible = ("defaultfeasible", True)
    m.d = ("Labour supply", [0, "retire", 1, "work"])
    m.choiceset = ("defaultallow", True)
    m.u = ("utility", "log(consumption)+duw*(id==0)")
    m.param = ("duw", "utility of leisure", duw)
    m.u = ("marginal", "1/consumption")
    m.u = ("marginalinverse", "1/mutility")
    m.u = ("extrap", "log(x)")
    m.budget = ("cashinhand", "savings*(1+interest)+wage_income*(id!=0)")
    m.budget = ("marginal", "1+interest")
    m.discount = "1/(1+interest)"
    m.param = ("interest", "return on savings", interest)
    m.eq = ("wage_income", "Realized wage income", "wage*shock*(0.4+0.6*st1)", "next")
    m.param = ("wage", "wage (times multiplicator shock)", wage)
    m.a0 = a0
    m.shock = "lognormal"
    m.shock = ("sigma", sigma)
    m.shock = ("mu", "-0.5*sigma*sigma")
    return m


def humancapital2(**kw) -> EgdstModel:
    return humancapital(health=True, **kw)


def retirement2_smooth(sigma_eps=0.2, **kw) -> EgdstModel:
    """retirement2 with extreme-value taste shocks of scale ``sigma_eps`` on the labour-supply choice -- the opt-in
    smoothing mode (an extension: the reference has a hard max only, SURVEY 0 fact 2)."""
    m = retirement(**kw)
    m.sigma_eps = sigma_eps
    return m


def retirement_two_period(sigma_eps=0.5, ngridm=2000) -> EgdstModel:
    """Closed-form case of the smoothing mode (tests/smoothing_checks.py): periods t=1,2, no income risk, zero interest
    (discount 1), a0 = 0."""
    m = retirement(label="retire_kat", sigma="0", T=2, ngridm=ngridm, ngridmax=2 * ngridm, nthrhmax=50, ny=1, interest=0.0,
                   mmax=10, a0=0.0, duw=0.5, wage=1.05)
    m.sigma_eps = sigma_eps
    return m


def humancapital_smooth(sigma_eps=0.2, **kw) -> EgdstModel:
    """humancapital (one continuous state) with extreme-value taste shocks of scale ``sigma_eps`` on the labour-supply
    choice: choice draws and the choice likelihood at the exact human capital z."""
    m = humancapital(**kw)
    m.sigma_eps = sigma_eps
    return m


def humancapital2_smooth(sigma_eps=0.2, **kw) -> EgdstModel:
    """humancapital2 (two continuous states: four corner cells) with taste shocks of scale ``sigma_eps``."""
    m = humancapital(health=True, **kw)
    m.sigma_eps = sigma_eps
    return m


# images of the smoothing mode (compiled with EGDST_SMOOTHING, codegen.emit_devspec)
SMOOTH = {"retirement2_smooth": retirement2_smooth, "retirement_two_period": retirement_two_period,
          "humancapital_smooth": humancapital_smooth, "humancapital2_smooth": humancapital2_smooth}

EXTRA = {"deaton_normal": deaton_normal, "deaton_meanstest": deaton_meanstest, "humancapital": humancapital, "humancapital2": humancapital2,
         "retirement_mortal": retirement_mortal, "retirement_jobloss": retirement_jobloss}

ALL = {
    "deaton1": deaton1, "deaton2": deaton2, "retirement1": retirement1, "retirement2": retirement2,
    "occ3": occ3, "cake1": cake1, "cake2": cake2, "model2": model2,
}
