"""``EgdstModel`` -- host-side mirror of the reference's ``@egdstmodel`` handle class.

The reference's host language is MATLAB (absent in this image), so the class API is restated in
Python with the same property names, the same *append-on-assignment* setters and the same methods
(``compile``, ``solve``, ``sim``, ``call``, ``setparam``, ``getparam``):

    m = EgdstModel('retire2')
    m.t0 = 1; m.T = 25; m.mmax = 10; m.ngridm = 100 ...
    m.s = ('Singleton state', [0, 'dummy state'])            # egdstmodel.m:574-660
    m.d = ('Labour supply', [0, 'retire', 1, 'work'])        # egdstmodel.m:661-716
    m.u = ('utility', 'log(consumption)+duw*(id==0)')        # egdstmodel.m:717-741
    m.param = ('duw', 'disutility of work', 0.5)             # egdstmodel.m:912-948
    m.compile(); m.solve(); m.sim([[1, 0.25]])

``solve``/``sim``/``call`` go through the C-ABI of the per-model CUDA library
(include/egdst_b200.h); there is no CPU path -- a missing library or GPU raises.

Reference: @egdstmodel/egdstmodel.m (properties :356-425, setters :527-1009, solve :1141-1178,
call :1181-1207, sim :1210-1276, buildstates/stepmult :1432-1461).
"""
from __future__ import annotations

import itertools
import os
import time
from typing import Any, Dict, List

import numpy as np

from . import codegen
from .quadrature import model_quadrature

_APPEND_PROPS = ("s", "d", "u", "transform", "budget", "shock", "eq", "coef", "choiceset", "feasible", "param", "trpr",
                 "discount", "survival", "ngridm", "ngridmax")

_new_id = itertools.count(1)


def _numstr(v: float, fmt: str = "%.25f") -> str:
    return "0.0" if float(v) == 0.0 else (fmt % float(v))


class EgdstModel:
    def __init__(self, label: str = "<no name>", directory: str | None = None):
        d = self.__dict__
        d["label"] = label
        d["t0"] = float("nan")
        d["T"] = float("nan")
        d["s"] = []
        d["d"] = []
        d["mmax"] = float("nan")
        d["ngridm"] = 10
        d["ngridmax"] = 100
        d["nthrhmax"] = 100
        d["ny"] = 1
        d["a0"] = 0.0
        d["sigma_eps"] = 0.0  # EXTENSION (no reference counterpart): scale of extreme-value taste shocks on the discrete choice; 0 = the reference's hard max
        d["discount"] = ""
        d["survival"] = "1.0"
        d["u"] = {"utility": None, "marginal": None, "marginalinverse": None, "extrap": None}
        d["transform"] = {"direct": "log(x+1)", "inverse": "exp(x)-1"}
        d["budget"] = {"cashinhand": None, "marginal": None}
        d["shock"] = {"type": "lognormal", "mu": None, "sigma": None}
        d["trpr"] = []
        d["choiceset"] = {"defaultallow": True, "rules": []}
        d["feasible"] = {"defaultfeasible": True, "rules": []}
        d["eq"] = []
        d["coef"] = []
        d["param"] = []
        d["cflags"] = {"TOLERANCE": "1e-10", "ZEROCONSUMPTION": "1e-10", "DOUBLEPOINT_DELTA": "1e-10", "VERBOSE": "0"}
        # private-set properties
        d["nd"] = 0
        d["nnd"] = 0
        d["nst"] = 0
        d["nnst"] = 0
        d["stm"] = []
        d["dm"] = []
        d["M"] = None
        d["D"] = None
        d["states"] = np.zeros((0, 0))
        d["decisions"] = np.zeros((0, 0))
        d["sims"] = None
        d["simlabels"] = []
        d["init"] = None
        d["randstream"] = None
        d["optim"] = {"optim_MUnoD": False, "optim_UnoD": False, "optim_UasD": False, "optim_TRPRnoSH": False}
        d["quadrature"] = None
        d["quiet"] = True
        d["needtocompile"] = True
        d["lastrun_solver"] = None
        d["id"] = next(_new_id)
        d["dir"] = directory
        d["_lib"] = None
        d["_solution"] = None
        d["device"] = 0

    # ------------------------------------------------------------------ property plumbing
    def __setattr__(self, name: str, value: Any) -> None:
        if name in _APPEND_PROPS:
            getattr(self, "_set_" + name)(value)
        elif name == "cflags":
            self.__dict__["cflags"] = dict(value)
            self.__dict__["needtocompile"] = True
        else:
            self.__dict__[name] = value

    @property
    def nt(self) -> int:
        res = int(self.T) - int(self.t0) + 1
        if res < 1:
            raise ValueError("Error: t0>T!")
        return res

    # grids (egdstmodel.m:532-545)
    def _set_ngridm(self, value):
        self.__dict__["ngridm"] = int(value)
        if self.ngridm * 1.5 > self.ngridmax:
            self.__dict__["ngridmax"] = 2 * self.ngridm

    def _set_ngridmax(self, value):
        self.__dict__["ngridmax"] = int(value)
        if self.ngridm * 1.5 > self.ngridmax:
            self.__dict__["ngridmax"] = 2 * self.ngridm

    def _set_discount(self, value):
        self.__dict__["discount"] = value if isinstance(value, str) else _numstr(value)
        self.__dict__["needtocompile"] = True

    def _set_survival(self, value):
        self.__dict__["survival"] = value if isinstance(value, str) else _numstr(value)
        self.__dict__["needtocompile"] = True

    @staticmethod
    def _stepmult(a: List[int]) -> List[int]:
        """[a1..aN] -> [a2*..*aN, a3*..*aN, .., 1]  (egdstmodel.m:1432-1437)."""
        return [int(np.prod(a[i + 1:])) if i + 1 < len(a) else 1 for i in range(len(a))]

    def _variable(self, value, kind: str) -> Dict[str, Any]:
        name, spec = value[0], value[1]
        if len(value) == 3:
            # name + grid limits + number of grid points: a continuous variable on a uniform grid whose points double
            # as the enumerated "values" (egdstmodel.m:629-648)
            lim, npts = [float(x) for x in value[1]], int(value[2])
            if kind != "state" or len(lim) != 2 or npts < 2:
                raise ValueError("Unrecognized structure for %s variable!" % kind)
            if not lim[0] < lim[1]:
                # the reference accepts any pair; its grid search and the interpolation weights assume an increasing grid
                raise ValueError("Grid limits of a continuous state variable must be increasing!")
            grid = np.linspace(lim[0], lim[1], npts)
            return {"name": name, "type": "continuous", "discrete": False, "continuous": True,
                    "values": [{"value": float(g), "description": "grid point"} for g in grid],
                    "gridlimits": lim, "gridpoints": npts, "grid": [float(g) for g in grid]}
        vals = []
        if len(spec) and not any(isinstance(v, str) for v in spec):
            # numeric vector of values (egdstmodel.m:618-634)
            vals = [{"value": float(v), "description": "value %1.3f" % float(v)} for v in spec]
        else:
            if len(spec) % 2 != 0:
                raise ValueError("Unrecognized structure for %s variable!" % kind)
            for i in range(len(spec) // 2):
                if not isinstance(spec[2 * i], (int, float)):
                    raise ValueError("Non-numeric value of the %s variable detected!" % kind)
                vals.append({"value": float(spec[2 * i]), "description": str(spec[2 * i + 1])})
        return {"name": name, "type": "discrete", "discrete": True, "continuous": False, "values": vals}

    def _build(self, wh: str) -> np.ndarray:
        """Enumerate state/decision vectors, first variable slowest (egdstmodel.m:1439-1461)."""
        vars_ = self.s if wh == "s" else self.d
        lists = [[v["value"] for v in var["values"]] for var in vars_]
        rows = list(itertools.product(*lists))
        return np.asarray(rows, dtype=np.float64).reshape(len(rows), len(vars_))

    def _set_s(self, value):
        self.__dict__["needtocompile"] = True
        if not value:
            self.__dict__.update(s=[], nnst=0, trpr=[], stm=[], nst=0)
            return
        var = self._variable(value, "state")
        var["index"] = self.nnst + 1
        self.s.append(var)
        self.__dict__["nnst"] = self.nnst + 1
        sizes = [len(v["values"]) for v in self.s]
        self.__dict__["stm"] = sizes + self._stepmult(sizes)
        self.__dict__["nst"] = int(np.prod(sizes))
        self.__dict__["states"] = self._build("s")

    def _set_d(self, value):
        self.__dict__["needtocompile"] = True
        if not value:
            self.__dict__.update(d=[], nnd=0, dm=[], nd=0)
            return
        var = self._variable(value, "decision")
        var["index"] = self.nnd + 1
        self.d.append(var)
        self.__dict__["nnd"] = self.nnd + 1
        sizes = [len(v["values"]) for v in self.d]
        self.__dict__["dm"] = sizes + self._stepmult(sizes)
        self.__dict__["nd"] = int(np.prod(sizes))
        self.__dict__["decisions"] = self._build("d")

    def _set_u(self, value):
        self.__dict__["needtocompile"] = True
        key, val = value
        if key not in ("utility", "marginal", "marginalinverse", "extrap"):
            raise ValueError("Unrecognized structure for utility definition!")
        self.u[key] = val

    def _set_transform(self, value):
        self.__dict__["needtocompile"] = True
        if not value:
            self.__dict__["transform"] = {"direct": "log(x+1)", "inverse": "exp(x)-1"}
        else:
            self.__dict__["transform"] = {"direct": value[0], "inverse": value[1]}

    def _set_budget(self, value):
        self.__dict__["needtocompile"] = True
        key, val = value
        if key not in ("cashinhand", "marginal"):
            raise ValueError("Unrecognized structure for budget definition!")
        self.budget[key] = val

    def _set_shock(self, value):
        self.__dict__["needtocompile"] = True
        if isinstance(value, str):
            if value not in ("lognormal", "normal"):
                raise ValueError("Unrecognized structure for shock definition!")
            self.shock["type"] = value
            return
        key, val = value
        if key not in ("mu", "sigma"):
            raise ValueError("Unrecognized structure for shock definition!")
        self.shock[key] = val if isinstance(val, (str, list)) else _numstr(val)

    def _set_eq(self, value):
        self.__dict__["needtocompile"] = True
        if not value:
            self.__dict__["eq"] = []
            return
        ref, desc, expr = value[0], value[1], value[2]
        typ = value[3] if len(value) == 4 else "current"
        if typ not in ("current", "next"):
            raise ValueError("Unrecognized structure for equation definition!")
        new = {"ref": ref, "type": typ, "expression": expr, "description": desc}
        for i, e in enumerate(self.eq):
            if e["ref"] == ref:
                self.eq[i] = new
                break
        else:
            self.eq.append(new)
        self._checkrefs()

    def _set_coef(self, value):
        self.__dict__["needtocompile"] = True
        if not value:
            self.__dict__["coef"] = []
            return
        ref, desc, arr = value
        arr = np.atleast_2d(np.asarray(arr, dtype=np.float64)).tolist()
        self.coef.append({"ref": ref, "array": arr, "description": desc})
        self._checkrefs()

    def _set_choiceset(self, value):
        self.__dict__["needtocompile"] = True
        if not value:
            self.__dict__["choiceset"] = {"defaultallow": True, "rules": []}
        elif value[0] == "defaultallow" and isinstance(value[1], (bool, int)):
            self.choiceset["defaultallow"] = bool(value[1])
        else:
            self.choiceset["rules"].append({"condition": value[0], "description": value[1]})

    def _set_feasible(self, value):
        self.__dict__["needtocompile"] = True
        if not value:
            self.__dict__["feasible"] = {"defaultfeasible": True, "rules": []}
        elif value[0] == "defaultfeasible" and isinstance(value[1], (bool, int)):
            self.feasible["defaultfeasible"] = bool(value[1])
        else:
            self.feasible["rules"].append({"condition": value[0], "description": value[1]})

    def _set_param(self, value):
        if not value:
            self.__dict__["param"] = []
            return
        ref, desc, val = value
        self.param.append({"ref": ref, "description": desc, "value": float(val)})
        self.__dict__["needtocompile"] = True
        self._checkrefs()

    def _set_trpr(self, value):
        """{condition, matrix} or {varindex, condition, matrix}; numbers become '%10.10f' strings
        (egdstmodel.m:950-1008)."""
        self.__dict__["needtocompile"] = True
        if not value:
            self.__dict__["trpr"] = []
            return
        value = list(value)
        if len(value) == 2:
            value = [len(self.s)] + value
        vi, cond, mat = value
        if not (1 <= vi <= self.nnst):
            raise ValueError("Unrecognized structure for trpr definition!")
        n = self.stm[vi - 1]
        while len(self.trpr) < vi:
            self.trpr.append({"varindex": None, "cases": []})
        if isinstance(mat, str):
            # varindex + condition + executable string: the deterministic motion rule of a continuous state
            # (egdstmodel.m:1000-1004)
            self.trpr[vi - 1]["varindex"] = vi
            self.trpr[vi - 1]["cases"].append({"condition": cond, "prob": mat})
            return
        rows = [list(r) for r in mat]
        if len(rows) != n or any(len(r) != n for r in rows):
            raise ValueError("Unrecognized structure for trpr definition!")
        prob = [[(x if x else "0.0") if isinstance(x, str) else ("%10.10f" % float(x)) for x in r] for r in rows]
        self.trpr[vi - 1]["varindex"] = vi
        self.trpr[vi - 1]["cases"].append({"condition": cond, "prob": prob})

    def _checkrefs(self):
        reserved = codegen.RESERVED_GLOBALS + [
            "age", "ist", "id1", "id", "consumption", "mutility", "discount", "survival", "utility",
            "utility_marginal", "utility_marginal_inverse", "trpr", "feasible", "inchoiceset", "cashinhand",
            "cashinhand_marginal", "shock", "mu_param", "sigma_param", "sigma", "mu", "cash", "savings", "min", "max"]
        reserved += ["st%d" % i for i in range(1, 16)] + ["dc%d" % i for i in range(1, 16)]
        refs = reserved + [e["ref"] for e in self.eq] + [c["ref"] for c in self.coef] + [p["ref"] for p in self.param]
        if len(set(refs)) != len(refs):
            dup = sorted({r for r in refs if refs.count(r) > 1})
            raise ValueError("Not unique refs: %s" % dup)

    # ------------------------------------------------------------------ parameters
    def setparam(self, *args):
        """egdstmodel.m:1078-1112: vector of values, or ref/index,value pairs."""
        if len(args) == 1:
            vals = np.atleast_1d(np.asarray(args[0], dtype=np.float64))
            if len(vals) != len(self.param):
                raise ValueError("Passed vector does not match the dimentionality of param vector in the model!")
            for p, v in zip(self.param, vals):
                p["value"] = float(v)
        elif len(args) % 2 == 0:
            for k in range(len(args) // 2):
                key, v = args[2 * k], args[2 * k + 1]
                if isinstance(key, int) and 1 <= key <= len(self.param):
                    self.param[key - 1]["value"] = float(v)
                elif isinstance(key, str) and key in [p["ref"] for p in self.param]:
                    for p in self.param:
                        if p["ref"] == key:
                            p["value"] = float(v)
                else:
                    raise ValueError("Unrecognized pairs 'name',value,.. or index,value,.. !")
        else:
            raise ValueError("Expected pairs 'name',value,.. or index,value,.. !")

    def getparam(self, key=None):
        if key is None:
            return np.array([p["value"] for p in self.param])
        if isinstance(key, int):
            return self.param[key - 1]["value"]
        for p in self.param:
            if p["ref"] == key:
                return p["value"]
        raise ValueError("Unrecognized parameter name or parameter index out of bounds")

    def param_vector(self) -> np.ndarray:
        return np.array([p["value"] for p in self.param], dtype=np.float64)

    # ------------------------------------------------------------------ compile / solve / sim / call
    def _check_complete(self):
        for k in ("utility", "marginal", "marginalinverse"):
            if not self.u[k]:
                raise ValueError("Missing .u.%s, can not proceed with compile!" % k)
        for k in ("cashinhand", "marginal"):
            if not self.budget[k]:
                raise ValueError("Missing .budget.%s, can not proceed with compile!" % k)
        for k in ("mu", "sigma"):
            if self.shock[k] is None:
                raise ValueError("Missing .shock.%s, can not proceed with compile!" % k)
        if not self.discount:
            raise ValueError("Missing .discount, can not proceed with compile!")
        if not self.trpr or any(t["varindex"] is None for t in self.trpr):
            raise ValueError("Missing .trpr, can not proceed with compile!")

    def prepare(self):
        """The host-only half of ``compile``: checks, optim_* inference, simlabels (compile.m:579-747)."""
        self._check_complete()
        self.__dict__["optim"] = codegen.infer_optim(self)
        labels = ["1  cash-in-hand (M)", "2  optimal consumption (C)", "3  optimal saving (A)", "4  value function",
                  "5  current discrete decision index (id)", "6  current period state index (ist)",
                  "7  mu parameter of shock distribution", "8  sigma parameter of shock distribution",
                  "9  income shock", "10 utility", "11 discount factor"]
        for i, sv in enumerate(self.s):
            labels.append("%2d %s (st%d)" % (12 + i, sv["name"], i + 1))
        for i, dv in enumerate(self.d):
            labels.append("%2d %s (dc%d)" % (12 + len(self.s) + i, dv["name"], i + 1))
        for i, e in enumerate(self.eq):
            labels.append("%2d %s (eq%d)" % (12 + len(self.s) + len(self.d) + i, e["description"], i + 1))
        self.__dict__["simlabels"] = labels
        return self

    def compile(self, force: bool = False):
        """Generate the model header and build the per-model CUDA library with nvcc for sm_100a
        (replaces compile.m:754-819, which runs ``mex`` three times)."""
        from . import build
        self.prepare()
        path = build.build_model_library(self, force=force)
        self.__dict__["_libpath"] = path
        self.__dict__["_lib"] = None
        self.__dict__["M"] = None
        self.__dict__["D"] = None
        self.__dict__["sims"] = None
        self.__dict__["needtocompile"] = False
        return self

    def _capi(self):
        from . import capi
        if self.needtocompile:
            raise RuntimeError("The model needs to be compiled first! Run <model>.compile()")
        if self._lib is None:
            self.__dict__["_lib"] = capi.ModelLibrary(self._libpath)
        return self._lib

    def solve(self):
        """[M, D] = egdst_solver(model) through the C-ABI (egdstmodel.m:1141-1178)."""
        lib = self._capi()
        if self.ngridmax <= self.ngridm:
            self.__dict__["ngridmax"] = 2 * self.ngridm
        if self.ny > 1:
            self.__dict__["quadrature"] = model_quadrature(self.ny)
        t = time.perf_counter()
        sol = lib.solve(self)
        self.__dict__["lastrun_solver"] = time.perf_counter() - t
        self.__dict__["_solution"] = sol
        self.__dict__["M"], self.__dict__["D"] = sol.M, sol.D
        return self

    def sim(self, init=None, shocks: str = "own_shocks", randstream=None, draw_choices: bool = False):
        """sims = egdst_simulator(model, rndtype), permuted to [nsim, nt, nsimout] (egdstmodel.m:1210-1276).

        ``draw_choices`` (smoothing mode, ``sigma_eps > 0``): draw each period's decision from the choice probabilities
        instead of taking the modal choice (egdst_solution_set_choice_draws); the uniform of period it is slot
        3*(nt-1)+it of each agent's randstream block."""
        lib = self._capi()
        if self._solution is None:
            raise RuntimeError("The model needs to be compiled and solved first!")
        if shocks not in ("own_shocks", "same_shocks"):
            raise ValueError("Could not recognize argument!")
        rndtype = 1 if shocks == "same_shocks" else 0
        if init is not None:
            self.__dict__["init"] = np.atleast_2d(np.asarray(init, dtype=np.float64))
        if self.init is None:
            self.__dict__["init"] = np.array([[1.0, 0.0]])
        self.init[:, 1] = np.maximum(self.init[:, 1], self.a0)
        if randstream is not None:
            self.__dict__["randstream"] = np.asarray(randstream, dtype=np.float64).ravel()
        if self.randstream is None:
            rng = np.random.default_rng()
            self.__dict__["randstream"] = rng.random(max(self.init.shape[0], 100) * self.nt * 100)
        self._solution.set_choice_draws(draw_choices)
        sims = lib.simulate(self, self._solution, self.init, self.randstream, rndtype)  # [nsim, nt, nsimout]
        self.__dict__["sims"] = sims
        return self

    def loglik(self, obs, sigma_c: float = 0.0) -> float:
        """Smoothing mode (``sigma_eps > 0``) only: log-likelihood of the observations ``obs`` [nobs, 4 + K or 5 + K] under the
        current solution (egdst_choice_loglik; ``capi.observations_from_sims`` builds ``obs`` from simulated records)."""
        lib = self._capi()
        if self._solution is None:
            raise RuntimeError("The model needs to be compiled and solved first!")
        return float(lib.choice_loglik(self, self._solution, obs, sigma_c=sigma_c)[0])

    def mixture_loglik(self, obs, start, type_params, weights, sigma_c: float = 0.0, posterior: bool = False):
        """Smoothing mode (``sigma_eps > 0``) only: log-likelihood of a finite mixture over unobserved types.  Solves the
        parameter vectors ``type_params`` [ntypes, nparam] as one batch and evaluates the mixture with type weights
        ``weights`` [ntypes] (normalised by the library) over the observations ``obs`` grouped by individual with
        offsets ``start`` (``capi.observations_from_sims(..., start=True)``).  Returns the total, or (total, post
        [ntypes, nind]) with ``posterior=True`` (egdst_mixture_loglik)."""
        from . import capi
        lib = self._capi()
        tp = np.atleast_2d(np.asarray(type_params, dtype=np.float64))
        sol = lib.solve_batch(self, tp)
        if sol.warning:
            import warnings
            warnings.warn(sol.warning, capi.EgdstWarning)
        # a one-vector solution takes its parameter values from the descriptor (as egdst_simulate does)
        desc = capi.Desc(self)
        desc.params[:] = tp[0]
        ntypes = tp.shape[0]
        res = lib.mixture_loglik(self, sol, obs, start, np.arange(ntypes), np.asarray(weights, dtype=np.float64).reshape(1, ntypes),
                                 sigma_c=sigma_c, posterior=posterior, desc=desc)
        return (float(res[0][0]), res[1][0]) if posterior else float(res[0])

    def _solve_vectors(self, lib, pv):
        from . import capi
        sol = lib.solve_batch(self, pv)
        if sol.warning:
            import warnings
            warnings.warn(sol.warning, capi.EgdstWarning)
        return sol

    def _free_index(self, free):
        names = [p["ref"] for p in self.param]
        free = [free] if isinstance(free, str) else list(free)
        for f in free:
            if f not in names:
                raise ValueError("unknown parameter %r (parameters: %s)" % (f, ", ".join(names)))
        if not free or len(set(free)) != len(free):
            raise ValueError("free must name distinct parameters")
        return [names.index(f) for f in free]

    def _scores_at(self, lib, theta, idx, obs, start, sigma_c, step):
        """(total, grad, opg) at the full parameter vector ``theta`` for the components ``idx``: one batch of 2P+1
        vectors (centre, then theta_p + h_p and theta_p - h_p per component) and one one-type mixture per vector."""
        npar, nv = len(idx), 2 * len(idx) + 1
        pv = np.tile(np.asarray(theta, dtype=np.float64), (nv, 1))
        for p, j in enumerate(idx):
            h = step * max(abs(theta[j]), 1.0)
            pv[1 + 2 * p, j] += h
            pv[2 + 2 * p, j] -= h
        mplus, mminus = 1 + 2 * np.arange(npar), 2 + 2 * np.arange(npar)
        hinv = 1.0 / (pv[mplus, idx] - pv[mminus, idx])  # from the values solved
        sol = self._solve_vectors(lib, pv)
        tot, grad, opg = lib.mixture_scores(self, sol, obs, start, np.arange(nv).reshape(nv, 1), np.ones((nv, 1)), mplus,
                                            mminus, hinv, sigma_c=sigma_c)
        return float(tot[0]), grad, opg

    def scores(self, obs, start, free, sigma_c: float = 0.0, step: float = 1e-4):
        """Smoothing mode (``sigma_eps > 0``) only: central-difference scores of the log-likelihood of ``obs`` grouped
        by individual with offsets ``start`` (``capi.observations_from_sims(..., start=True)``) in the parameters named
        by ``free``, at the model's current values.  The centre and theta_p +- h_p, h_p = step * max(|theta_p|, 1), are
        solved as one batch and evaluated in one call (egdst_mixture_scores).  Returns (total, grad [P], opg [P, P]):
        the log-likelihood, its gradient and the outer product of the per-individual scores."""
        return self._scores_at(self._capi(), self.param_vector(), self._free_index(free), obs, start, sigma_c, step)

    def fit(self, obs, start, free, sigma_c: float = 0.0, step: float = 1e-4, tol: float = 1e-8, maxiter: int = 100):
        """Smoothing mode only: maximum likelihood in the parameters named by ``free`` by BHHH, starting from the model's
        current values (which are left unchanged).  Each iteration takes the scores of ``scores`` (one batched solve
        and one call), the direction d = OPG^-1 grad, and tries the step lengths 1, 1/2, 1/4 and 1/8 as one more batched
        solve and one ``mixture_loglik`` call of one-type mixtures (so that the totals have the bits of the score
        call's), taking the best that improves the total.  Stops when grad' OPG^-1 grad < tol.  Returns (estimates [P],
        standard errors sqrt(diag(OPG^-1)) [P], total, grad [P], opg [P, P], iterations).  Raises FloatingPointError on
        a non-finite total or score, numpy.linalg.LinAlgError on an OPG that is not positive definite, and
        RuntimeError when no step length improves the total or maxiter iterations do not converge.  The numerical noise
        of the totals (the solve, and the rounding of totals of large panels) bounds the criterion that can be reached:
        on a 200 000-individual panel it stalled near 1e-7, a distance of 4e-4 standard errors, so a large panel may
        need a larger ``tol``."""
        lib = self._capi()
        idx = self._free_index(free)
        theta = self.param_vector()
        lam = np.array([1.0, 0.5, 0.25, 0.125])
        for it in range(maxiter + 1):
            total, grad, opg = self._scores_at(lib, theta, idx, obs, start, sigma_c, step)
            if not (np.isfinite(total) and np.all(np.isfinite(grad)) and np.all(np.isfinite(opg))):
                raise FloatingPointError("BHHH: non-finite total or scores at %s = %s (an individual with -inf "
                                         "likelihood?)" % (list(free), theta[idx]))
            try:
                chol = np.linalg.cholesky(opg)
            except np.linalg.LinAlgError:
                raise np.linalg.LinAlgError("BHHH: the OPG matrix at %s = %s is singular" % (list(free), theta[idx]))
            d = np.linalg.solve(chol.T, np.linalg.solve(chol, grad))
            crit = float(grad @ d)
            if crit < tol:
                cinv = np.linalg.solve(chol, np.eye(len(idx)))
                se = np.sqrt(np.sum(cinv * cinv, axis=0))  # diag(OPG^-1) = column norms of L^-1
                return theta[idx].copy(), se, total, grad, opg, it
            if it == maxiter:
                break
            pv = np.tile(theta, (lam.size, 1))
            pv[:, idx] += lam[:, None] * d
            sol = self._solve_vectors(lib, pv)
            tots = lib.mixture_loglik(self, sol, obs, start, np.arange(lam.size).reshape(-1, 1), np.ones((lam.size, 1)),
                                      sigma_c=sigma_c)
            ok = np.isfinite(tots) & (tots > total)
            if not ok.any():
                raise RuntimeError("BHHH: no step length improves the total %.17g at %s = %s (grad' OPG^-1 grad = %.3g; "
                                   "a larger tol stops at this point)"
                                   % (total, list(free), theta[idx], crit))
            theta = pv[int(np.argmax(np.where(ok, tots, -np.inf)))]
        raise RuntimeError("BHHH did not converge in %d iterations: grad' OPG^-1 grad = %.3g" % (maxiter, crit))

    def call(self, func: str, funcargs):
        """res = egdst_call(model, sw, args) (egdstmodel.m:1181-1207)."""
        lib = self._capi()
        table = {"utility": 1, "util": 1, "u": 1, "mutility": 2, "mu": 2, "discount": 3, "df": 3,
                 "budget": 4, "b": 4, "mbudget": 5, "mb": 5, "value": 6, "vf": 6}
        if self._solution is None:  # egdstmodel.m:1182-1184
            raise RuntimeError("The model needs to be compiled and solved first!")
        if func not in table:
            raise ValueError("Unknown internal model function to call!")
        return lib.call(self, self._solution, table[func], np.atleast_2d(np.asarray(funcargs, dtype=np.float64)))

    def nsimout(self) -> int:
        return 11 + self.nnst + self.nnd + len(self.eq)

    # ------------------------------------------------------------------ (de)serialisation of the public properties
    _SCALARS = ("label", "t0", "T", "mmax", "ngridm", "ngridmax", "nthrhmax", "ny", "a0", "discount", "survival", "sigma_eps")

    def to_dict(self) -> Dict[str, Any]:
        """The public properties as plain data, in the shape ``jsonencode(struct(model))`` gives in MATLAB."""
        d: Dict[str, Any] = {k: getattr(self, k) for k in self._SCALARS}
        d["s"] = [dict({"name": v["name"], "values": [dict(x) for x in v["values"]]},
                       **({"gridlimits": list(v["gridlimits"]), "gridpoints": v["gridpoints"]} if v["continuous"] else {}))
                  for v in self.s]
        d["d"] = [{"name": v["name"], "values": [dict(x) for x in v["values"]]} for v in self.d]
        d["u"] = dict(self.u)
        d["transform"] = dict(self.transform)
        d["budget"] = dict(self.budget)
        d["shock"] = dict(self.shock)
        d["trpr"] = [{"varindex": t["varindex"], "cases": [dict(c) for c in t["cases"]]} for t in self.trpr]
        d["choiceset"] = {"defaultallow": self.choiceset["defaultallow"], "rules": [dict(r) for r in self.choiceset["rules"]]}
        d["feasible"] = {"defaultfeasible": self.feasible["defaultfeasible"], "rules": [dict(r) for r in self.feasible["rules"]]}
        d["eq"] = [dict(e) for e in self.eq]
        d["coef"] = [dict(c) for c in self.coef]
        d["param"] = [dict(p) for p in self.param]
        d["cflags"] = dict(self.cflags)
        return d

    @classmethod
    def from_dict(cls, d: Dict[str, Any]) -> "EgdstModel":
        def lst(x):  # jsonencode collapses 1-element struct arrays to a struct
            return [] if x is None else (x if isinstance(x, list) else [x])
        m = cls(d.get("label", "<no name>"))
        m.t0, m.T, m.mmax = d["t0"], d["T"], d["mmax"]
        m.ngridmax = d.get("ngridmax", 100)
        m.ngridm = d.get("ngridm", 10)
        m.nthrhmax, m.ny, m.a0 = d.get("nthrhmax", 100), d.get("ny", 1), d.get("a0", 0.0)
        m.sigma_eps = float(d.get("sigma_eps", 0.0) or 0.0)
        for kind in ("s", "d"):
            for v in lst(d.get(kind)):
                if v.get("gridpoints"):
                    setattr(m, kind, (v["name"], list(v["gridlimits"]), int(v["gridpoints"])))
                    continue
                spec = []
                for x in lst(v["values"]):
                    spec += [x["value"], x["description"]]
                setattr(m, kind, (v["name"], spec))
        for k, v in d["u"].items():
            if v:
                m.u = (k, v)
        if d.get("transform"):
            m.transform = (d["transform"]["direct"], d["transform"]["inverse"])
        for k in ("cashinhand", "marginal"):
            m.budget = (k, d["budget"][k])
        m.shock = d["shock"].get("type", "lognormal")
        m.shock = ("mu", d["shock"]["mu"])
        m.shock = ("sigma", d["shock"]["sigma"])
        m.discount = d["discount"]
        m.survival = d.get("survival", "1.0")
        for p in lst(d.get("param")):
            m.param = (p["ref"], p.get("description", ""), p["value"])
        for c in lst(d.get("coef")):
            m.coef = (c["ref"], c.get("description", ""), c["array"])
        for e in lst(d.get("eq")):
            m.eq = (e["ref"], e.get("description", ""), e["expression"], e.get("type", "current"))
        for t in lst(d.get("trpr")):
            for c in lst(t["cases"]):
                m.trpr = (int(t["varindex"]), c["condition"], c["prob"])
        cs = d.get("choiceset") or {}
        m.choiceset = ("defaultallow", bool(cs.get("defaultallow", True)))
        for r in lst(cs.get("rules")):
            m.choiceset = (r["condition"], r.get("description", ""))
        fs = d.get("feasible") or {}
        m.feasible = ("defaultfeasible", bool(fs.get("defaultfeasible", True)))
        for r in lst(fs.get("rules")):
            m.feasible = (r["condition"], r.get("description", ""))
        if d.get("cflags"):
            m.cflags = {k: str(v) for k, v in d["cflags"].items()}
        return m


def env_dir(default: str) -> str:
    return os.environ.get("EGDST_B200_BUILD_DIR", default)
