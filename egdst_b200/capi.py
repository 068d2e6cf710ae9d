"""ctypes binding of the C ABI in include/egdst_b200.h (the same entry points the MEX stubs bind).

No torch types cross this boundary: plain pointers and sizes.  A missing library raises -- there is
no CPU path.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional

import numpy as np

from .quadrature import model_quadrature

ABI_VERSION = 2
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


class EgdstDesc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int),
        ("t0", C.c_int), ("T", C.c_int), ("ngridm", C.c_int), ("ngridmax", C.c_int), ("nthrhmax", C.c_int),
        ("ny", C.c_int), ("nd", C.c_int), ("nnd", C.c_int), ("nst", C.c_int), ("nnst", C.c_int),
        ("mmax", C.c_double), ("a0", C.c_double),
        ("optim_UasD", C.c_int), ("optim_MUnoD", C.c_int), ("optim_UnoD", C.c_int), ("optim_TRPRnoSH", C.c_int),
        ("tolerance", C.c_double), ("zeroconsumption", C.c_double), ("doublepoint_delta", C.c_double),
        ("stm", _dp), ("states", _dp), ("decisions", _dp), ("params", _dp), ("nparam", C.c_int),
        ("quadrature", _dp), ("neq", C.c_int), ("device", C.c_int), ("sigma_eps", C.c_double),
    ]


class EgdstError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(msg)
        self.code = code


class EgdstWarning(UserWarning):
    pass


def _arr(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


def _ptr(a: Optional[np.ndarray]):
    return a.ctypes.data_as(_dp) if a is not None and a.size else None


class Desc:
    """Keeps the numpy buffers alive next to the ctypes struct."""

    def __init__(self, model, device: Optional[int] = None):
        m = model
        self.stm = _arr(m.stm)
        self.states = _arr(np.asfortranarray(m.states).ravel(order="F"))
        self.decisions = _arr(np.asfortranarray(m.decisions).ravel(order="F"))
        self.params = _arr(m.param_vector())
        self.quadrature = _arr(model_quadrature(m.ny)) if m.ny > 1 else None
        d = EgdstDesc()
        d.abi_version = ABI_VERSION
        d.t0, d.T, d.ngridm, d.ngridmax, d.nthrhmax = int(m.t0), int(m.T), int(m.ngridm), int(m.ngridmax), int(m.nthrhmax)
        d.ny, d.nd, d.nnd, d.nst, d.nnst = int(m.ny), int(m.nd), int(m.nnd), int(m.nst), int(m.nnst)
        d.mmax, d.a0 = float(m.mmax), float(m.a0)
        o = m.optim
        d.optim_UasD, d.optim_MUnoD, d.optim_UnoD, d.optim_TRPRnoSH = (int(bool(o["optim_UasD"])), int(bool(o["optim_MUnoD"])),
                                                                      int(bool(o["optim_UnoD"])), int(bool(o["optim_TRPRnoSH"])))
        d.tolerance = float(m.cflags["TOLERANCE"])
        d.zeroconsumption = float(m.cflags["ZEROCONSUMPTION"])
        d.doublepoint_delta = float(m.cflags["DOUBLEPOINT_DELTA"])
        d.stm, d.states, d.decisions, d.params = _ptr(self.stm), _ptr(self.states), _ptr(self.decisions), _ptr(self.params)
        d.nparam = len(m.param)
        d.quadrature = _ptr(self.quadrature)
        d.neq = len(m.eq)
        d.device = int(m.device if device is None else device)
        d.sigma_eps = float(getattr(m, "sigma_eps", 0.0) or 0.0)
        self.c = d


class Solution:
    """Handle of a device-resident solution; ``M``/``D`` are exported lazily as nst x nt nested lists."""

    def __init__(self, lib: "ModelLibrary", handle, model, nvec: int = 1):
        self.lib, self.handle, self.nvec = lib, handle, nvec
        self.nst, self.nt = model.nst, model.nt
        self._cells = None
        self.warning: Optional[str] = None

    def __del__(self):
        try:
            if self.handle:
                self.lib.L.egdst_free_solution(self.handle)
                self.handle = None
        except Exception:
            pass

    def sizes(self):
        n = self.nvec * self.nt * self.nst
        mlen = np.zeros(n, dtype=np.int32)
        thlen = np.zeros(n, dtype=np.int32)
        rc = self.lib.L.egdst_solution_sizes(self.handle, mlen.ctypes.data_as(_ip), thlen.ctypes.data_as(_ip))
        if rc == 2:
            self.lib._raise(rc)
        return mlen, thlen

    def export(self):
        """Returns (mlen, thlen, Mbuf, Dbuf): the packed host copy (saveoutput layouts)."""
        mlen, thlen = self.sizes()
        Mbuf = np.empty(4 * int(mlen.sum()), dtype=np.float64)
        Dbuf = np.empty(2 * int(thlen.sum()), dtype=np.float64)
        rc = self.lib.L.egdst_solution_export(self.handle, Mbuf.ctypes.data_as(_dp), Dbuf.ctypes.data_as(_dp))
        if rc:
            self.lib._raise(rc)
        return mlen, thlen, Mbuf, Dbuf

    def cells(self, ivec: int = 0):
        """(M, D) nested lists [ist][it] of (mlen x 4) / (thlen x 2) arrays for parameter vector ``ivec``."""
        if self._cells is None:
            self._cells = self.export()
        mlen, thlen, Mbuf, Dbuf = self._cells
        moff = np.concatenate([[0], np.cumsum(mlen)]) * 4
        toff = np.concatenate([[0], np.cumsum(thlen)]) * 2
        M = [[None] * self.nt for _ in range(self.nst)]
        D = [[None] * self.nt for _ in range(self.nst)]
        for it in range(self.nt):
            for ist in range(self.nst):
                c = (ivec * self.nt + it) * self.nst + ist
                if mlen[c] > 0:
                    M[ist][it] = Mbuf[moff[c]:moff[c + 1]].reshape((mlen[c], 4), order="F")
                    D[ist][it] = Dbuf[toff[c]:toff[c + 1]].reshape((thlen[c], 2), order="F")
        return M, D

    @property
    def M(self):
        return self.cells(0)[0]

    @property
    def D(self):
        return self.cells(0)[1]

    def choice_cell(self, it: int, ist: int, id: int, ivec: int = 0):
        """Smoothing mode (model.sigma_eps > 0) only: the choice-specific cell of decision ``id`` as an (rows x 4) array
        (M, C, A, V; row 0 = a0, 0, a0, evf_d(a0)), or None where the decision is not available."""
        n = C.c_int(0)
        rc = self.lib.L.egdst_solution_choice_cell(self.handle, ivec, it, ist, id, None, 0, C.byref(n))
        if rc:
            self.lib._raise(rc)
        if n.value == 0:
            return None
        buf = np.empty(4 * n.value, dtype=np.float64)
        rc = self.lib.L.egdst_solution_choice_cell(self.handle, ivec, it, ist, id, buf.ctypes.data_as(_dp), n.value, C.byref(n))
        if rc:
            self.lib._raise(rc)
        return buf.reshape(4, n.value).T.copy()

    def set_choice_draws(self, on: bool):
        """Smoothing mode only: simulations of this solution draw each period's decision from the choice probabilities
        (on) or take the modal choice (off, the default).  See egdst_solution_set_choice_draws in include/egdst_b200.h."""
        rc = self.lib.L.egdst_solution_set_choice_draws(self.handle, 1 if on else 0)
        if rc:
            self.lib._raise(rc)

    def status(self, ivec: int = 0):
        it, ist, idd = C.c_int(0), C.c_int(0), C.c_int(0)
        code = self.lib.L.egdst_solution_status(self.handle, ivec, C.byref(it), C.byref(ist), C.byref(idd))
        return code, it.value, ist.value, idd.value

    def units(self) -> int:
        return int(self.lib.L.egdst_solution_units(self.handle))

    PHASES = ("terminal", "seed", "egm", "resend", "envelope2", "rank", "merge", "tables")

    def phase_ms(self):
        """{phase: ms} of the solve kernel, accumulated over profiled solves of this object (reading resets)."""
        ms = (C.c_double * len(self.PHASES))()
        n = self.lib.L.egdst_solution_phase_ms(self.handle, ms)
        return {self.PHASES[i]: float(ms[i]) for i in range(max(n, 0))}

    def resends(self) -> int:
        """Zero-consumption re-sends after the seed stage that the last solve handled (diagnostic)."""
        return int(self.lib.L.egdst_solution_resends(self.handle))


def observations_from_sims(model, sims, consumption: bool = True, start: bool = False):
    """The live records of a simulation ``sims`` [nsim, nt, nsimout] as observations for ``ModelLibrary.choice_loglik``:
    [nobs, 5 + K] (or [nobs, 4 + K] without ``consumption``) of age t0 + it, state ist + 1, cash, decision id + 1, the
    exact values x_1..x_K of the model's K continuous states (record columns 11 + j, in state order) and consumption,
    agent-major.  Dead and skipped records (NaN) are dropped.  With ``start=True`` returns (obs, start):
    the int32 offsets [nsim + 1] of each agent's rows for ``ModelLibrary.mixture_loglik`` (individual i = agent i; an
    agent without a live record is an empty individual)."""
    s = np.asarray(sims, dtype=np.float64)
    cash, cons, dec, ist = s[:, :, 0], s[:, :, 1], s[:, :, 4], s[:, :, 5]
    live = ~(np.isnan(cash) | np.isnan(dec) | np.isnan(ist))
    ai, ti = np.nonzero(live)
    cols = [model.t0 + ti.astype(np.float64), ist[ai, ti] + 1.0, cash[ai, ti], dec[ai, ti] + 1.0]
    cols += [s[ai, ti, 11 + j] for j, v in enumerate(model.s) if v["continuous"]]
    if consumption:
        cols.append(cons[ai, ti])
    obs = np.column_stack(cols) if ai.size else np.zeros((0, len(cols)))
    if not start:
        return obs
    return obs, np.concatenate([[0], np.cumsum(live.sum(axis=1))]).astype(np.int32)


def _mixture_args(obs, start, tvec, weights):
    """The arrays of a mixture call: (obs column-major, nobs, k, start int32, tvec int32 [nmix, ntypes], weights)."""
    o = np.atleast_2d(np.asarray(obs, dtype=np.float64))
    nobs, k = o.shape
    st = np.ascontiguousarray(np.asarray(start), dtype=np.int32)
    tv = np.ascontiguousarray(np.atleast_2d(np.asarray(tvec)), dtype=np.int32)
    w = _arr(np.atleast_2d(np.asarray(weights, dtype=np.float64)))
    if st.ndim != 1 or st.size < 1:
        raise ValueError("start must be a 1-D array of nind + 1 offsets")
    if tv.ndim != 2 or tv.shape != w.shape:
        raise ValueError("tvec and weights must both be [nmix, ntypes]")
    return _arr(o.ravel(order="F")), nobs, k, st, tv, w


class ModelLibrary:
    """One loaded model image (libegdst_b200_<key>.so)."""

    EXPORTS = ["egdst_abi_version", "egdst_model_key", "egdst_model_nparam", "egdst_model_neq", "egdst_last_error",
               "egdst_set_stream", "egdst_launch_count", "egdst_profile_classes", "egdst_profile_class_name",
               "egdst_profile_enable", "egdst_profile_read", "egdst_solve", "egdst_solve_batch", "egdst_resolve", "egdst_solution_sizes",
               "egdst_solution_export", "egdst_solution_choice_cell", "egdst_solution_set_choice_draws", "egdst_solution_status", "egdst_solution_nvec", "egdst_solution_units", "egdst_solution_resends", "egdst_solution_phase_ms", "egdst_test_envelope2",
               "egdst_test_sim_variant",
               "egdst_free_solution", "egdst_solution_import", "egdst_simulate", "egdst_simulate_philox",
               "egdst_simulate_device", "egdst_sim_moments", "egdst_sim_moments_device", "egdst_choice_loglik",
               "egdst_choice_loglik_device", "egdst_mixture_loglik", "egdst_mixture_loglik_device",
               "egdst_mixture_scores", "egdst_mixture_scores_device", "egdst_call", "egdst_shutdown"]

    def __init__(self, path: str):
        if not os.path.isfile(path):
            raise FileNotFoundError("egdst_b200 model library not found: %s (run model.compile(); there is no CPU path)" % path)
        self.path = path
        self.L = L = C.CDLL(path)
        vp = C.c_void_p
        L.egdst_abi_version.restype = C.c_int
        L.egdst_model_key.restype = C.c_char_p
        L.egdst_last_error.restype = C.c_char_p
        L.egdst_set_stream.argtypes = [vp]
        L.egdst_launch_count.restype = C.c_longlong
        L.egdst_profile_class_name.restype = C.c_char_p
        L.egdst_profile_class_name.argtypes = [C.c_int]
        L.egdst_profile_enable.argtypes = [C.c_int]
        L.egdst_profile_read.argtypes = [_dp, C.POINTER(C.c_longlong)]
        L.egdst_solve.argtypes = [C.POINTER(EgdstDesc), C.POINTER(vp)]
        L.egdst_solve_batch.argtypes = [C.POINTER(EgdstDesc), _dp, C.c_int, C.POINTER(vp)]
        L.egdst_resolve.argtypes = [vp, C.POINTER(EgdstDesc), _dp]
        L.egdst_solution_sizes.argtypes = [vp, _ip, _ip]
        L.egdst_solution_export.argtypes = [vp, _dp, _dp]
        L.egdst_solution_choice_cell.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, _dp, C.c_int, _ip]
        L.egdst_solution_set_choice_draws.argtypes = [vp, C.c_int]
        L.egdst_solution_status.argtypes = [vp, C.c_int, _ip, _ip, _ip]
        L.egdst_solution_nvec.argtypes = [vp]
        L.egdst_solution_units.argtypes = [vp]
        L.egdst_solution_units.restype = C.c_longlong
        L.egdst_solution_phase_ms.argtypes = [vp, _dp]
        L.egdst_solution_resends.argtypes = [vp]
        L.egdst_solution_resends.restype = C.c_longlong
        L.egdst_free_solution.argtypes = [vp]
        L.egdst_free_solution.restype = None
        L.egdst_shutdown.restype = None
        L.egdst_solution_import.argtypes = [C.POINTER(EgdstDesc), _ip, _ip, _dp, _dp, C.POINTER(vp)]
        L.egdst_simulate.argtypes = [C.POINTER(EgdstDesc), vp, C.c_int, _dp, C.c_int, _dp, C.c_longlong, C.c_int, _dp]
        L.egdst_simulate_philox.argtypes = [C.POINTER(EgdstDesc), vp, C.c_int, _dp, C.c_int, C.c_longlong, C.c_ulonglong, _dp, _dp]
        L.egdst_simulate_device.argtypes = [C.POINTER(EgdstDesc), vp, C.c_int, vp, C.c_int, C.c_longlong, C.c_ulonglong,
                                            vp, C.c_int, vp, vp]
        L.egdst_call.argtypes = [C.POINTER(EgdstDesc), vp, C.c_int, _dp, C.c_int, C.c_int, _dp]
        L.egdst_choice_loglik.argtypes = [C.POINTER(EgdstDesc), vp, C.c_int, C.c_int, _dp, C.c_int, C.c_int, C.c_double, _dp, _dp]
        L.egdst_choice_loglik_device.argtypes = [C.POINTER(EgdstDesc), vp, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_double, vp, vp]
        L.egdst_mixture_loglik.argtypes = [C.POINTER(EgdstDesc), vp, C.c_int, C.c_int, _dp, C.c_int, C.c_int, C.c_double, _ip,
                                           C.c_int, C.c_int, C.c_int, _ip, _dp, _dp, _dp, _dp, _dp]
        L.egdst_mixture_loglik_device.argtypes = [C.POINTER(EgdstDesc), vp, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_double,
                                                  vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp]
        L.egdst_mixture_scores.argtypes = [C.POINTER(EgdstDesc), vp, C.c_int, C.c_int, _dp, C.c_int, C.c_int, C.c_double, _ip,
                                           C.c_int, C.c_int, C.c_int, _ip, _dp, C.c_int, _ip, _ip, _dp, _dp, _dp, _dp, _dp]
        L.egdst_mixture_scores_device.argtypes = [C.POINTER(EgdstDesc), vp, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_double,
                                                  vp, C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, vp, vp, vp, vp, vp, vp, vp]
        L.egdst_sim_moments.argtypes = [C.POINTER(EgdstDesc), vp, C.c_int, C.c_int, _dp, C.c_int, C.c_longlong, C.c_ulonglong, _dp]
        L.egdst_sim_moments_device.argtypes = [C.POINTER(EgdstDesc), vp, C.c_int, C.c_int, vp, C.c_int, C.c_longlong, C.c_ulonglong, vp]
        L.egdst_test_sim_variant.argtypes = [C.POINTER(C.c_longlong)]
        L.egdst_test_envelope2.argtypes = [C.POINTER(EgdstDesc), C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, C.c_int, C.c_double,
                                           _dp, _dp, _dp, _ip]
        if L.egdst_abi_version() != ABI_VERSION:
            raise RuntimeError("ABI version mismatch in %s" % path)

    def last_error(self) -> str:
        return self.L.egdst_last_error().decode(errors="replace")

    def _raise(self, rc: int):
        raise EgdstError(rc, self.last_error())

    def set_stream(self, stream_ptr: int):
        self.L.egdst_set_stream(C.c_void_p(stream_ptr))

    def launch_count(self) -> int:
        return int(self.L.egdst_launch_count())

    def profile_enable(self, on: bool):
        self.L.egdst_profile_enable(1 if on else 0)

    def profile_read(self):
        """{class name: (total ms, launches)} accumulated since profile_enable(True)."""
        n = self.L.egdst_profile_classes()
        ms = (C.c_double * n)()
        cnt = (C.c_longlong * n)()
        self.L.egdst_profile_read(ms, cnt)
        return {self.L.egdst_profile_class_name(i).decode(): (float(ms[i]), int(cnt[i])) for i in range(n)}

    def simulate_device(self, model, sol: "Solution", d_init: int, nsim: int, agent0: int, seed: int, d_sims: int = 0,
                        d_moments: int = 0, d_randstream: int = 0, rndtype: int = 0, ivec: int = 0, desc: "Desc" = None):
        """Asynchronous launch on the library stream; all pointers are device addresses (ints)."""
        d = desc or Desc(model)
        rc = self.L.egdst_simulate_device(C.byref(d.c), sol.handle, ivec, C.c_void_p(d_init), nsim, agent0, seed,
                                          C.c_void_p(d_randstream or None), rndtype, C.c_void_p(d_sims or None),
                                          C.c_void_p(d_moments or None))
        if rc:
            self._raise(rc)

    # -- solve
    def solve(self, model, device: Optional[int] = None, strict: bool = False) -> Solution:
        d = Desc(model, device)
        h = C.c_void_p()
        rc = self.L.egdst_solve(C.byref(d.c), C.byref(h))
        if rc == 2 or (rc and strict):
            if h:
                self.L.egdst_free_solution(h)
            self._raise(rc)
        sol = Solution(self, h, model)
        if rc == 1:  # soft error: partial result kept, like mexWarnMsgTxt(err) (egdst_solver.c:237)
            import warnings
            sol.warning = self.last_error()
            warnings.warn(sol.warning, EgdstWarning)
        return sol

    def solve_batch(self, model, params: np.ndarray, device: Optional[int] = None) -> Solution:
        d = Desc(model, device)
        p = _arr(params)
        if p.ndim != 2 or p.shape[1] != len(model.param):
            raise ValueError("params must be [nvec, nparam]")
        h = C.c_void_p()
        rc = self.L.egdst_solve_batch(C.byref(d.c), _ptr(p), p.shape[0], C.byref(h))
        if rc == 2:
            self._raise(rc)
        sol = Solution(self, h, model, nvec=p.shape[0])
        if rc == 1:
            sol.warning = self.last_error()
        return sol

    def resolve(self, sol: Solution, model, params: Optional[np.ndarray] = None, device: Optional[int] = None):
        d = Desc(model, device)
        p = _arr(params) if params is not None else None
        rc = self.L.egdst_resolve(sol.handle, C.byref(d.c), _ptr(p))
        if rc:
            self._raise(rc)
        sol._cells = None

    def import_solution(self, model, M, D, device: Optional[int] = None) -> Solution:
        d = Desc(model, device)
        nst, nt = model.nst, model.nt
        mlen = np.zeros(nt * nst, dtype=np.int32)
        thlen = np.zeros(nt * nst, dtype=np.int32)
        mb: List[np.ndarray] = []
        db: List[np.ndarray] = []
        for it in range(nt):
            for ist in range(nst):
                c = it * nst + ist
                if M[ist][it] is not None and M[ist][it].size:
                    mlen[c] = M[ist][it].shape[0]
                    thlen[c] = D[ist][it].shape[0]
                    mb.append(np.asarray(M[ist][it], dtype=np.float64).ravel(order="F"))
                    db.append(np.asarray(D[ist][it], dtype=np.float64).ravel(order="F"))
        Mbuf = _arr(np.concatenate(mb)) if mb else np.zeros(1)
        Dbuf = _arr(np.concatenate(db)) if db else np.zeros(1)
        h = C.c_void_p()
        rc = self.L.egdst_solution_import(C.byref(d.c), mlen.ctypes.data_as(_ip), thlen.ctypes.data_as(_ip), _ptr(Mbuf), _ptr(Dbuf), C.byref(h))
        if rc:
            self._raise(rc)
        return Solution(self, h, model)

    # -- simulate
    def simulate(self, model, sol: Solution, init, randstream, rndtype: int = 0, ivec: int = 0) -> np.ndarray:
        """[nsim, nt, nsimout] (already permuted as egdstmodel.m:1270 does)."""
        d = Desc(model)
        init = np.atleast_2d(np.asarray(init, dtype=np.float64))
        nsim = init.shape[0]
        initf = _arr(init.ravel(order="F"))
        rs = _arr(np.asarray(randstream, dtype=np.float64).ravel())
        nso, nt = model.nsimout(), model.nt
        sims = np.empty(nso * nt * nsim, dtype=np.float64)
        rc = self.L.egdst_simulate(C.byref(d.c), sol.handle, ivec, _ptr(initf), nsim, _ptr(rs), rs.size, rndtype, _ptr(sims))
        if rc:
            self._raise(rc)
        return np.transpose(sims.reshape((nso, nt, nsim), order="F"), (2, 1, 0))

    def simulate_philox(self, model, sol: Solution, init, seed: int, agent0: int = 0, ivec: int = 0, want_sims=True, want_moments=False):
        d = Desc(model)
        init = np.atleast_2d(np.asarray(init, dtype=np.float64))
        nsim = init.shape[0]
        initf = _arr(init.ravel(order="F"))
        nso, nt = model.nsimout(), model.nt
        sims = np.empty(nso * nt * nsim, dtype=np.float64) if want_sims else None
        mom = np.zeros(3 * nso * nt, dtype=np.float64) if want_moments else None
        rc = self.L.egdst_simulate_philox(C.byref(d.c), sol.handle, ivec, _ptr(initf), nsim, agent0, seed, _ptr(sims), _ptr(mom))
        if rc:
            self._raise(rc)
        out_s = np.transpose(sims.reshape((nso, nt, nsim), order="F"), (2, 1, 0)) if want_sims else None
        out_m = mom.reshape((3, nso, nt), order="F") if want_moments else None
        return out_s, out_m

    def sim_moments(self, model, sol: Solution, init, seed: int, agent0: int = 0, ivec0: int = 0, nvec: Optional[int] = None) -> np.ndarray:
        """Moments [nvec, 3, nsimout, nt] of the same agents under parameter vectors ivec0.. of a batched solution."""
        d = Desc(model)
        init = np.atleast_2d(np.asarray(init, dtype=np.float64))
        nsim = init.shape[0]
        initf = _arr(init.ravel(order="F"))
        nvec = sol.nvec - ivec0 if nvec is None else nvec
        nso, nt = model.nsimout(), model.nt
        mom = np.zeros(nvec * 3 * nso * nt, dtype=np.float64)
        rc = self.L.egdst_sim_moments(C.byref(d.c), sol.handle, ivec0, nvec, _ptr(initf), nsim, agent0, seed, _ptr(mom))
        if rc:
            self._raise(rc)
        # per vector [3, nsimout, nt] column-major == C-order (nt, nsimout, 3): one reshape + transpose, no copies
        return mom.reshape(nvec, nt, nso, 3).transpose(0, 3, 2, 1)

    def sim_moments_device(self, model, sol: Solution, d_init: int, nsim: int, agent0: int, seed: int, d_moments: int,
                           ivec0: int = 0, nvec: Optional[int] = None, desc: "Desc" = None):
        d = desc or Desc(model)
        nvec = sol.nvec - ivec0 if nvec is None else nvec
        rc = self.L.egdst_sim_moments_device(C.byref(d.c), sol.handle, ivec0, nvec, C.c_void_p(d_init), nsim, agent0, seed, C.c_void_p(d_moments))
        if rc:
            self._raise(rc)

    def choice_loglik(self, model, sol: Solution, obs, sigma_c: float = 0.0, ivec0: int = 0, nvec: Optional[int] = None,
                      rows: bool = False):
        """Smoothing mode only: log-likelihood of the observations ``obs`` [nobs, 4 + K or 5 + K] (age, 1-based state,
        cash, 1-based decision, the values of the K continuous states[, consumption]; see ``observations_from_sims``) under parameter vectors ivec0.. of ``sol``.
        Returns the totals [nvec], and with ``rows=True`` also the per-row values [nvec, nobs].  See
        egdst_choice_loglik in include/egdst_b200.h for the formula and the -inf / NaN rules."""
        d = Desc(model)
        o = np.atleast_2d(np.asarray(obs, dtype=np.float64))
        nobs, k = o.shape
        of = _arr(o.ravel(order="F"))
        nvec = sol.nvec - ivec0 if nvec is None else nvec
        tot = np.zeros(max(nvec, 1), dtype=np.float64)
        rowll = np.empty(max(nvec, 1) * nobs, dtype=np.float64) if rows else None
        rc = self.L.egdst_choice_loglik(C.byref(d.c), sol.handle, ivec0, nvec, _ptr(of), nobs, k, float(sigma_c), _ptr(tot), _ptr(rowll))
        if rc:
            self._raise(rc)
        return (tot, rowll.reshape(nvec, nobs)) if rows else tot

    def choice_loglik_device(self, model, sol: Solution, d_obs: int, nobs: int, k: int, d_loglik: int, sigma_c: float = 0.0,
                             d_rowll: int = 0, ivec0: int = 0, nvec: Optional[int] = None, desc: "Desc" = None):
        """Asynchronous launch on the library stream; d_obs [k][nobs], d_loglik [nvec] (accumulated into: the caller
        zeroes it) and d_rowll [nvec][nobs] (optional) are device addresses (ints).  Rows are not checked."""
        d = desc or Desc(model)
        nvec = sol.nvec - ivec0 if nvec is None else nvec
        rc = self.L.egdst_choice_loglik_device(C.byref(d.c), sol.handle, ivec0, nvec, C.c_void_p(d_obs or None), nobs, k,
                                               float(sigma_c), C.c_void_p(d_loglik or None), C.c_void_p(d_rowll or None))
        if rc:
            self._raise(rc)

    def mixture_loglik(self, model, sol: Solution, obs, start, tvec, weights, sigma_c: float = 0.0, ivec0: int = 0,
                       nvec: Optional[int] = None, individuals: bool = False, posterior: bool = False, desc: "Desc" = None):
        """Smoothing mode only: finite-mixture log-likelihood over unobserved types.  ``obs`` [nobs, 4 + K or 5 + K] as for
        ``choice_loglik``, grouped by individual with offsets ``start`` [nind + 1] (``observations_from_sims(...,
        start=True)``); ``tvec`` [nmix, ntypes] the vector of each type relative to ``ivec0``, ``weights`` [nmix,
        ntypes] the type weights (normalised by the library).  A 1-D ``tvec`` / ``weights`` is one mixture.  Returns
        the totals [nmix]; with ``individuals=True`` or ``posterior=True`` a tuple (totals, then indll [nvec, nind] and
        mixll [nmix, nind] if ``individuals``, then post [nmix, ntypes, nind] if ``posterior``).  See
        egdst_mixture_loglik in include/egdst_b200.h for the formula, the edge rules and the determinism contract."""
        d = desc or Desc(model)
        of, nobs, k, st, tv, w = _mixture_args(obs, start, tvec, weights)
        nind, (nmix, ntypes) = st.size - 1, tv.shape
        nvec = sol.nvec - ivec0 if nvec is None else nvec
        tot = np.zeros(max(nmix, 1), dtype=np.float64)
        indll = np.empty(max(nvec, 1) * nind, dtype=np.float64) if individuals else None
        mixll = np.empty(max(nmix, 1) * nind, dtype=np.float64) if individuals else None
        post = np.empty(max(nmix * ntypes, 1) * nind, dtype=np.float64) if posterior else None
        rc = self.L.egdst_mixture_loglik(C.byref(d.c), sol.handle, ivec0, nvec, _ptr(of), nobs, k, float(sigma_c),
                                         st.ctypes.data_as(_ip), nind, ntypes, nmix, tv.ctypes.data_as(_ip), _ptr(w),
                                         _ptr(tot), _ptr(indll), _ptr(mixll), _ptr(post))
        if rc:
            self._raise(rc)
        out = (tot,)
        if individuals:
            out += (indll.reshape(nvec, nind), mixll.reshape(nmix, nind))
        if posterior:
            out += (post.reshape(nmix, ntypes, nind),)
        return out if len(out) > 1 else tot

    def mixture_loglik_device(self, model, sol: Solution, d_obs: int, nobs: int, k: int, d_start: int, nind: int,
                              d_tvec: int, d_w: int, ntypes: int, nmix: int, d_loglik: int, sigma_c: float = 0.0,
                              d_indll: int = 0, d_mixll: int = 0, d_post: int = 0, ivec0: int = 0,
                              nvec: Optional[int] = None, desc: "Desc" = None):
        """Asynchronous launch on the library stream; d_obs [k][nobs], d_start [nind + 1] (int32), d_tvec [nmix][ntypes]
        (int32), d_w [nmix][ntypes], d_loglik [nmix] (accumulated into: the caller zeroes it) and the optional d_indll
        [nvec][nind], d_mixll [nmix][nind] and d_post [nmix][ntypes][nind] are device addresses (ints).  Rows, offsets,
        type vectors and weights are not checked."""
        d = desc or Desc(model)
        nvec = sol.nvec - ivec0 if nvec is None else nvec
        vp = C.c_void_p
        rc = self.L.egdst_mixture_loglik_device(C.byref(d.c), sol.handle, ivec0, nvec, vp(d_obs or None), nobs, k,
                                                float(sigma_c), vp(d_start or None), nind, ntypes, nmix, vp(d_tvec or None),
                                                vp(d_w or None), vp(d_loglik or None), vp(d_indll or None),
                                                vp(d_mixll or None), vp(d_post or None))
        if rc:
            self._raise(rc)

    def mixture_scores(self, model, sol: Solution, obs, start, tvec, weights, mplus, mminus, hinv, sigma_c: float = 0.0,
                       ivec0: int = 0, nvec: Optional[int] = None, scores: bool = False, desc: "Desc" = None):
        """Smoothing mode only: central-difference scores of the mixtures ``tvec`` / ``weights`` (as for
        ``mixture_loglik``).  Component p is the difference of mixtures ``mplus[p]`` and ``mminus[p]`` times ``hinv[p]``
        (1 / the difference of the perturbed values solved); a one-type mixture of weight 1 is the plain likelihood.
        Returns (totals [nmix], grad [npar], opg [npar, npar]), and scores [npar, nind] too with ``scores=True``.  See
        egdst_mixture_scores in include/egdst_b200.h for the NaN rule and the determinism contract."""
        d = desc or Desc(model)
        of, nobs, k, st, tv, w = _mixture_args(obs, start, tvec, weights)
        nind, (nmix, ntypes) = st.size - 1, tv.shape
        mp = np.ascontiguousarray(np.atleast_1d(np.asarray(mplus)), dtype=np.int32)
        mm = np.ascontiguousarray(np.atleast_1d(np.asarray(mminus)), dtype=np.int32)
        h = _arr(np.atleast_1d(np.asarray(hinv, dtype=np.float64)))
        if not (mp.ndim == 1 and mp.shape == mm.shape == h.shape):
            raise ValueError("mplus, mminus and hinv must be 1-D of one length npar")
        npar = mp.size
        nvec = sol.nvec - ivec0 if nvec is None else nvec
        tot = np.zeros(max(nmix, 1), dtype=np.float64)
        grad = np.zeros(max(npar, 1), dtype=np.float64)
        opg = np.zeros(max(npar * npar, 1), dtype=np.float64)
        sc = np.empty(max(npar, 1) * nind, dtype=np.float64) if scores else None
        rc = self.L.egdst_mixture_scores(C.byref(d.c), sol.handle, ivec0, nvec, _ptr(of), nobs, k, float(sigma_c),
                                         st.ctypes.data_as(_ip), nind, ntypes, nmix, tv.ctypes.data_as(_ip), _ptr(w), npar,
                                         mp.ctypes.data_as(_ip), mm.ctypes.data_as(_ip), _ptr(h), _ptr(tot), _ptr(grad),
                                         _ptr(opg), _ptr(sc))
        if rc:
            self._raise(rc)
        out = (tot, grad, opg.reshape(npar, npar))
        return out + (sc.reshape(npar, nind),) if scores else out

    def mixture_scores_device(self, model, sol: Solution, d_obs: int, nobs: int, k: int, d_start: int, nind: int,
                              d_tvec: int, d_w: int, ntypes: int, nmix: int, npar: int, d_mplus: int, d_mminus: int,
                              d_hinv: int, d_loglik: int, d_grad: int, d_opg: int, sigma_c: float = 0.0, d_scores: int = 0,
                              ivec0: int = 0, nvec: Optional[int] = None, desc: "Desc" = None):
        """Asynchronous launch on the library stream; the arguments of ``mixture_loglik_device`` plus d_mplus, d_mminus
        [npar] (int32) and d_hinv [npar]; d_loglik [nmix], d_grad [npar] and d_opg [npar][npar] are accumulated into
        (the caller zeroes them), d_scores [npar][nind] is optional.  Nothing is checked per row, offset, type, weight
        or component: an out-of-range mixture index gives NaN scores."""
        d = desc or Desc(model)
        nvec = sol.nvec - ivec0 if nvec is None else nvec
        vp = C.c_void_p
        rc = self.L.egdst_mixture_scores_device(C.byref(d.c), sol.handle, ivec0, nvec, vp(d_obs or None), nobs, k,
                                                float(sigma_c), vp(d_start or None), nind, ntypes, nmix, vp(d_tvec or None),
                                                vp(d_w or None), npar, vp(d_mplus or None), vp(d_mminus or None),
                                                vp(d_hinv or None), vp(d_loglik or None), vp(d_grad or None),
                                                vp(d_opg or None), vp(d_scores or None))
        if rc:
            self._raise(rc)

    def call(self, model, sol: Solution, sw: int, args: np.ndarray) -> np.ndarray:
        d = Desc(model)
        a = np.atleast_2d(np.asarray(args, dtype=np.float64))
        narg, k = a.shape
        af = _arr(a.ravel(order="F"))
        res = np.full(narg, np.nan, dtype=np.float64)
        rc = self.L.egdst_call(C.byref(d.c), sol.handle, sw, _ptr(af), narg, k, _ptr(res))
        if rc == 2:
            self._raise(rc)
        if rc == 1:  # the reference warns ("Wrong number of arguments") and returns the NaN vector
            import warnings
            warnings.warn(self.last_error(), EgdstWarning)
        return res

    def sim_variant(self):
        """(PHILOX, OUT, HDR, PB, mom_smem) of the egdst_k_simulate launch this thread made last, and the number of
        simulation launches the thread has made (diagnostic, egdst_test_sim_variant)."""
        v = (C.c_longlong * 6)()
        self.L.egdst_test_sim_variant(v)
        return (bool(v[0]), int(v[1]), bool(v[2]), int(v[3]), bool(v[4])), int(v[5])

    def test_envelope2(self, model, it: int, idd: int, X, Cc, V, evfa0: float):
        """Secondary envelope of one decision's EGM points (generation order) by the solve kernel's phases."""
        d = Desc(model)
        X, Cc, V = _arr(X), _arr(Cc), _arr(V)
        cap = int(model.ngridmax) + 8
        oX, oC, oV = np.zeros(cap), np.zeros(cap), np.zeros(cap)
        n = C.c_int(0)
        rc = self.L.egdst_test_envelope2(C.byref(d.c), it, 0, idd, _ptr(X), _ptr(Cc), _ptr(V), X.size, float(evfa0), _ptr(oX), _ptr(oC), _ptr(oV), C.byref(n))
        if rc:
            self._raise(rc)
        return oX[:n.value].copy(), oC[:n.value].copy(), oV[:n.value].copy()

    def shutdown(self):
        """Release the library's cached solution object and this thread's simulation workspace."""
        self.L.egdst_shutdown()
