"""ctypes binding of the CPU oracle (oracle/polymc_oracle.c).

TEST INFRASTRUCTURE ONLY.  Imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / ``--impl reference`` leg; the product (polymer-stats_b200/) never imports it.

PARITY UNPINNED by the reference (it ships no tests or golden data and Julia is not installed
in this image): see the header of polymc_oracle.h for what pins the oracle instead.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libpolymc_oracle.so")

CHAIN_TYPES = {"dielectric": 0, "polar": 1}
ENERGY_TYPES = {"noninteracting": 0, "interacting": 1, "Ising": 2, "cutoff": 3}

AVG_NAMES = ["r1", "r2", "r3", "r1sq", "r2sq", "r3sq", "rsq",
             "p1", "p2", "p3", "p1sq", "p2sq", "p3sq", "psq", "U", "Usq"]


class OrcCase(C.Structure):
    """Mirror of ``orc_case``: one command line of mcmc_eap_chain.jl (:19-153)."""
    _fields_ = [
        ("E0", C.c_double), ("K1", C.c_double), ("K2", C.c_double), ("mu", C.c_double),
        ("kT", C.c_double), ("Fz", C.c_double), ("Fx", C.c_double), ("b", C.c_double),
        ("phi_step", C.c_double), ("theta_step", C.c_double),
        ("adj_lb", C.c_double), ("adj_ub", C.c_double), ("adj_scale", C.c_double),
        ("n", C.c_int64), ("steps_per_adjust", C.c_int64),
        ("chain_type", C.c_int32), ("energy_type", C.c_int32),
        ("do_flips", C.c_int32), ("umbrella", C.c_int32),
        ("omega_compat", C.c_int32), ("_pad", C.c_int32),
        # clustering driver (mcmc_clustering_eap_chain.jl:19-153)
        ("kappa", C.c_double), ("psi0", C.c_double), ("cutoff_radius", C.c_double), ("cluster_prob", C.c_double),
        ("clustering", C.c_int32), ("alpha_carry", C.c_int32), ("cutoff_full", C.c_int32), ("planar", C.c_int32),
    ]


def make_case(n=100, E0=0.0, K1=1.0, K2=0.0, mu=1e-2, kT=1.0, Fz=0.0, Fx=0.0, b=1.0,
              chain_type="dielectric", energy_type="noninteracting",
              phi_step=3 * math.pi / 8, theta_step=3 * math.pi / 16,
              adj_lb=0.15, adj_ub=0.55, adj_scale=1.1, steps_per_adjust=2500,
              do_flips=False, umbrella=False, omega_compat=False,
              kappa=0.0, psi0=0.0, cutoff_radius=7.5, cluster_prob=0.5, clustering=False, alpha_carry=True,
              cutoff_full=False, planar=False) -> OrcCase:
    """Defaults are the ArgParse defaults of mcmc_eap_chain.jl:19-153 (and, for the clustering fields,
    of mcmc_clustering_eap_chain.jl:36-51,87-90; note that driver's own defaults for --energy-type (Ising)
    and --step-adjust-ub (0.40) differ and are set by its host)."""
    return OrcCase(E0, K1, K2, mu, kT, Fz, Fx, b, phi_step, theta_step, adj_lb, adj_ub, adj_scale,
                   n, steps_per_adjust, CHAIN_TYPES[chain_type], ENERGY_TYPES[energy_type],
                   int(do_flips), int(umbrella), int(omega_compat), 0,
                   kappa, psi0, cutoff_radius, cluster_prob, int(clustering), int(alpha_carry), int(cutoff_full),
                   int(planar))


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "polymc_oracle.c")
    hdr = os.path.join(_HERE, "polymc_oracle.h")
    stale = (not os.path.exists(_LIB_PATH)) or any(
        os.path.exists(s) and os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in (src, hdr))
    if force or stale:
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B"])
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(_LIB_PATH)
    dp = C.POINTER(C.c_double)
    vp = C.c_void_p
    cp = C.POINTER(OrcCase)
    L.orc_philox4x32_10.argtypes = [C.POINTER(C.c_uint32)] * 3
    L.orc_draw_init.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_int64, dp, dp]
    L.orc_draw_step.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_int64, C.c_int64,
                                C.POINTER(C.c_int64), dp, C.POINTER(C.c_int32), dp, dp]
    L.orc_draw_reinit_eps.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32]
    L.orc_draw_reinit_eps.restype = C.c_double
    L.orc_chain_new.argtypes = [cp, dp, dp]
    L.orc_chain_new.restype = vp
    L.orc_chain_new_random.argtypes = [cp, C.c_uint64, C.c_uint32, C.c_uint32]
    L.orc_chain_new_random.restype = vp
    L.orc_chain_copy.argtypes = [vp]
    L.orc_chain_copy.restype = vp
    L.orc_chain_free.argtypes = [vp]
    L.orc_chain_energy.argtypes = [vp, dp]
    L.orc_chain_abs_pair_sum.argtypes = [vp]
    L.orc_chain_abs_pair_sum.restype = C.c_double
    for f in (L.orc_chain_r, L.orc_chain_p, L.orc_chain_xs, L.orc_chain_mus):
        f.argtypes = [vp, dp]
    L.orc_chain_state.argtypes = [vp, dp, dp]
    L.orc_chain_move.argtypes = [vp, C.c_int64, C.c_double, C.c_double]
    L.orc_chain_delta_u.argtypes = [vp, C.c_int64, C.c_double, C.c_double, dp]
    L.orc_chain_energy_ex.argtypes = [vp, dp]
    L.orc_chain_new_x0.argtypes = [cp, C.c_uint64, C.c_uint32, C.c_uint32, dp, C.c_int64, dp]
    L.orc_chain_new_x0.restype = vp
    L.orc_draw_cluster.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_int64, C.c_int32, C.c_int64]
    L.orc_draw_cluster.restype = C.c_double
    L.orc_draw_cluster_gate.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_int64]
    L.orc_draw_cluster_gate.restype = C.c_double
    L.orc_chain_delta_segment.argtypes = [vp, C.c_int64, C.c_double, C.c_double, C.c_int32, C.c_int64, C.c_int64, dp]
    L.orc_chain_move_segment.argtypes = [vp, C.c_int64, C.c_double, C.c_double, C.c_int32, C.c_int64, C.c_int64]
    L.orc_chain_link_prob.argtypes = [vp, C.c_int64]
    L.orc_chain_link_prob.restype = C.c_double
    L.orc_run_begin_stage.argtypes = [vp, C.c_double]
    L.orc_run_init_x0.argtypes = [vp, dp, C.c_int64, dp]
    L.orc_run_extra_averages.argtypes = [vp, dp]
    L.orc_run_steps_ex.argtypes = [vp, C.c_int64, C.c_int64, dp, dp, dp]
    L.orc_run_cluster_stats.argtypes = [vp, dp]
    L.orc_run_new.argtypes = [cp, C.c_uint64, C.c_uint32, C.c_int32]
    L.orc_run_new.restype = vp
    L.orc_run_new_tape.argtypes = [cp, C.c_int32, dp, C.c_int64, C.c_int32]
    L.orc_run_new_tape.restype = vp
    L.orc_run_tape_pos.argtypes = [vp]
    L.orc_run_tape_pos.restype = C.c_int64
    L.orc_run_set_state.argtypes = [vp, dp, dp]
    L.orc_run_steps.argtypes = [vp, C.c_int64, C.c_int64, dp, dp]
    L.orc_run_reinit.argtypes = [vp, C.c_int32]
    L.orc_run_reinit.restype = C.c_int32
    L.orc_run_averages.argtypes = [vp, dp, dp, dp]
    L.orc_run_diag.argtypes = [vp, dp]
    L.orc_run_chain.argtypes = [vp]
    L.orc_run_chain.restype = vp
    L.orc_run_free.argtypes = [vp]
    L.orc_bench.argtypes = [cp, C.c_uint64, C.c_int32, C.c_int32, C.c_int64, C.c_int32]
    L.orc_bench.restype = C.c_double
    _lib = L
    return L


def _dp(a: np.ndarray):
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.POINTER(C.c_double))


def philox(ctr, key):
    c = (C.c_uint32 * 4)(*ctr)
    k = (C.c_uint32 * 2)(*key)
    o = (C.c_uint32 * 4)()
    lib().orc_philox4x32_10(c, k, o)
    return list(o)


def draw_init(seed, chain_id, init, n):
    phi = np.empty(n)
    theta = np.empty(n)
    a, b = C.c_double(), C.c_double()
    for k in range(n):
        lib().orc_draw_init(seed, chain_id, init, k, C.byref(a), C.byref(b))
        phi[k], theta[k] = a.value, b.value
    return phi, theta


def draw_step(seed, chain_id, init, step, n):
    idx = C.c_int64()
    flip = C.c_int32()
    up, ut, eps = C.c_double(), C.c_double(), C.c_double()
    lib().orc_draw_step(seed, chain_id, init, step, n, C.byref(idx), C.byref(up), C.byref(flip),
                        C.byref(ut), C.byref(eps))
    return idx.value, up.value, flip.value, ut.value, eps.value


class Chain:
    """EAPChain (inc/eap_chain.jl:12-36) restated on the CPU."""

    def __init__(self, case: OrcCase, phi=None, theta=None, *, seed=None, chain_id=0, init=0, _ptr=None):
        self.case = case
        self.n = int(case.n)
        if _ptr is not None:
            self._p = _ptr
            self._own = False
            return
        self._own = True
        if phi is None:
            self._p = lib().orc_chain_new_random(C.byref(case), seed, chain_id, init)
        else:
            phi = np.ascontiguousarray(phi, dtype=np.float64)
            theta = np.ascontiguousarray(theta, dtype=np.float64)
            assert phi.shape == (self.n,) and theta.shape == (self.n,)
            self._p = lib().orc_chain_new(C.byref(case), _dp(phi), _dp(theta))

    def __del__(self):
        if getattr(self, "_own", False) and self._p:
            lib().orc_chain_free(self._p)
            self._p = None

    def energy(self):
        """-> dict(U, su, Udd, Omega): energy.jl:7-23 pieces."""
        o = np.empty(4)
        lib().orc_chain_energy(self._p, _dp(o))
        return {"U": o[0], "su": o[1], "Udd": o[2], "Omega": o[3]}

    def abs_pair_sum(self):
        return lib().orc_chain_abs_pair_sum(self._p)

    def energy_ex(self):
        """-> dict(U, su (incl. bending), Udd, Omega, Ubend, psi, cos2, abs_pair_sum)."""
        o = np.empty(8)
        lib().orc_chain_energy_ex(self._p, _dp(o))
        return dict(zip(["U", "su", "Udd", "Omega", "Ubend", "psi", "cos2", "abs_pair_sum"], o))

    def link_prob(self, i0):
        """pflip_linear(n̂_i·n̂_{i+1}) (eap_chain.jl:267,290)."""
        return lib().orc_chain_link_prob(self._p, i0)

    def delta_segment(self, idx0, dphi, dtheta, reflect, lo0, hi0):
        """Changed-term ΔU of move!(idx) followed by refl_n! on [lo,hi]; non-mutating."""
        o = np.empty(12)
        lib().orc_chain_delta_segment(self._p, idx0, dphi, dtheta, int(reflect), lo0, hi0, _dp(o))
        return dict(zip(["dU", "dOmega", "abs_sum", "du", "drF", "dpair", "dbend", "dpsi", "dcos2",
                         "dp1", "dp2", "dp3"], o))

    def move_segment(self, idx0, dphi, dtheta, reflect, lo0, hi0):
        """The same composite trial done literally (move! + refl_n! per monomer, full recomputes); mutates."""
        lib().orc_chain_move_segment(self._p, idx0, dphi, dtheta, int(reflect), lo0, hi0)

    def r(self):
        o = np.empty(3)
        lib().orc_chain_r(self._p, _dp(o))
        return o

    def p(self):
        o = np.empty(3)
        lib().orc_chain_p(self._p, _dp(o))
        return o

    def state(self):
        phi, theta = np.empty(self.n), np.empty(self.n)
        lib().orc_chain_state(self._p, _dp(phi), _dp(theta))
        return phi, theta

    def xs(self):
        o = np.empty(3 * self.n)
        lib().orc_chain_xs(self._p, _dp(o))
        return o.reshape(self.n, 3)

    def mus(self):
        o = np.empty(3 * self.n)
        lib().orc_chain_mus(self._p, _dp(o))
        return o.reshape(self.n, 3)

    def move(self, idx0, dphi, dtheta):
        """move! (eap_chain.jl:230-257), 0-based idx; mutates, full energy recompute."""
        lib().orc_chain_move(self._p, idx0, dphi, dtheta)

    def delta_u(self, idx0, dphi, dtheta):
        """Changed-pair ΔU, non-mutating -> dict(dU, dOmega, abs_sum, du, drF, dpair)."""
        o = np.empty(6)
        lib().orc_chain_delta_u(self._p, idx0, dphi, dtheta, _dp(o))
        return dict(zip(["dU", "dOmega", "abs_sum", "du", "drF", "dpair"], o))

    def copy(self):
        c = Chain(self.case, _ptr=lib().orc_chain_copy(self._p))
        c._own = True
        return c


class Run:
    """The mcmc() loop of mcmc_eap_chain.jl:171-376 for one chain.  algo 0 = the reference
    algorithm (deep copy + full recompute per trial), algo 1 = the changed-pair ΔU formulation."""

    def __init__(self, case: OrcCase, seed: int, chain_id: int = 0, algo: int = 0, tape=None, reinit_stale=False):
        """tape: an array of uniforms consumed in the reference's rand() call order instead of the Philox stream
        (polymc_oracle.h `orc_run_new_tape`); reinit_stale: the reference's literal stale acceptor after a re-init."""
        self.case = case
        if tape is None:
            self._p = lib().orc_run_new(C.byref(case), seed, chain_id, algo)
        else:
            self._tape = np.ascontiguousarray(tape, dtype=np.float64)   # must outlive the run
            self._p = lib().orc_run_new_tape(C.byref(case), algo, _dp(self._tape), self._tape.size, int(reinit_stale))

    def tape_pos(self) -> int:
        return int(lib().orc_run_tape_pos(self._p))

    def __del__(self):
        if getattr(self, "_p", None):
            lib().orc_run_free(self._p)
            self._p = None

    def set_state(self, phi, theta):
        phi = np.ascontiguousarray(phi, dtype=np.float64)
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        lib().orc_run_set_state(self._p, _dp(phi), _dp(theta))

    def steps(self, nsteps, stepout=0):
        rows = nsteps // stepout if stepout else 0
        traj = np.zeros((rows, 8))
        roll = np.zeros((rows, 17))
        lib().orc_run_steps(self._p, nsteps, stepout, _dp(traj) if rows else None, _dp(roll) if rows else None)
        return traj, roll

    def reinit(self, force=False):
        return bool(lib().orc_run_reinit(self._p, int(force)))

    # ---- clustering driver (mcmc_clustering_eap_chain.jl) ----
    def begin_stage(self, kT):
        """A fresh mcmc(nsteps, pargs, chain) call on the current chain at temperature kT (:171-265)."""
        lib().orc_run_begin_stage(self._p, float(kT))

    def init_x0(self, x0, dx0):
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        dx0 = np.ascontiguousarray(dx0, dtype=np.float64)
        lib().orc_run_init_x0(self._p, _dp(x0), x0.size, _dp(dx0))

    def steps_ex(self, nsteps, stepout=0, want_state=False):
        """-> traj [rows][8], roll [rows][19], state [rows][2n] (phi,theta interleaved) or None."""
        rows = nsteps // stepout if stepout else 0
        traj = np.zeros((rows, 8))
        roll = np.zeros((rows, 19))
        state = np.zeros((rows, 2 * int(self.case.n))) if want_state else None
        lib().orc_run_steps_ex(self._p, nsteps, stepout, _dp(traj) if rows else None, _dp(roll) if rows else None,
                               _dp(state) if (want_state and rows) else None)
        return traj, roll, state

    def extra_averages(self):
        o = np.empty(2)
        lib().orc_run_extra_averages(self._p, _dp(o))
        return o

    def cluster_stats(self):
        o = np.empty(3)
        lib().orc_run_cluster_stats(self._p, _dp(o))
        return dict(zip(["ncluster", "cluster_sum", "cluster_max"], o))

    def averages(self):
        avg = np.empty(16)
        ar, nrm = C.c_double(), C.c_double()
        lib().orc_run_averages(self._p, _dp(avg), C.byref(ar), C.byref(nrm))
        return avg, ar.value, nrm.value

    def diag(self):
        o = np.empty(8)
        lib().orc_run_diag(self._p, _dp(o))
        return dict(zip(["phi_step", "theta_step", "nacc", "natt", "nacc_total", "steps_total", "U", "Omega"], o))

    def chain(self) -> Chain:
        return Chain(self.case, _ptr=lib().orc_run_chain(self._p))


_native = None


def native_lib():
    """The `-O3 -march=native` build of the same source, compiled on THIS machine (timing only; bench.py).  Returns
    (library, flags text); falls back to the portable build when the host has no compiler.  Built in a temporary
    directory (the tree may be read-only) that is removed once the library is loaded."""
    global _native
    if _native is not None:
        return _native
    try:
        with tempfile.TemporaryDirectory(prefix="polymc_oracle_native_") as tmp:
            path = os.path.join(tmp, "libpolymc_oracle_native.so")
            subprocess.check_call(["make", "-C", _HERE, "-s", "native", f"NATIVE_OUT={path}"],
                                  stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            L = C.CDLL(path)
        L.orc_bench.argtypes = [C.POINTER(OrcCase), C.c_uint64, C.c_int32, C.c_int32, C.c_int64, C.c_int32]
        L.orc_bench.restype = C.c_double
        _native = (L, "gcc -O3 -march=native, built on the timed host")
    except Exception:
        _native = (lib(), "gcc -O3 -march=x86-64-v3 -ffp-contract=off (portable build; no compiler on the timed host)")
    return _native


def bench(case: OrcCase, seed: int, algo: int, nchains: int, nsteps: int, nthreads: int, native: bool = False) -> float:
    """Seconds to run nchains independent chains for nsteps trials each on nthreads pthreads."""
    L = native_lib()[0] if native else lib()
    return L.orc_bench(C.byref(case), seed, algo, nchains, nsteps, nthreads)
