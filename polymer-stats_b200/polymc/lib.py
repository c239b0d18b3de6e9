"""ctypes binding of libpolymc_b200.so (include/polymc.h) — the only compute path of this package.

There is deliberately no CPU fallback: if the shared library is missing, or no CUDA device is
present, every compute call raises `PolymcError`.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import subprocess

import numpy as np

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG_DIR)                      # polymer-stats_b200/
# PMC_LIB_PATH: an experiment build of the same library (tools/tune_*.py A/B runs); never a different implementation
LIB_PATH = os.environ.get("PMC_LIB_PATH") or os.path.join(_ROOT, "libpolymc_b200.so")
CSRC_DIR = os.path.join(_ROOT, "csrc")

CHAIN_TYPES = {"dielectric": 0, "polar": 1}
ENERGY_TYPES = {"noninteracting": 0, "interacting": 1, "Ising": 2, "cutoff": 3}
PAIR_PRECISIONS = {"fp64": 0, "fp32": 1}

AVG_NAMES = ["r1", "r2", "r3", "r1sq", "r2sq", "r3sq", "rsq",
             "p1", "p2", "p3", "p1sq", "p2sq", "p3sq", "psq", "U", "Usq"]

EXPORTS = [
    "pmc_abi_version", "pmc_last_error", "pmc_device_count", "pmc_create", "pmc_destroy",
    "pmc_num_chains", "pmc_num_monomers", "pmc_set_stream", "pmc_set_ensemble_hint", "pmc_set_pair_precision", "pmc_pair_precision", "pmc_block_threads", "pmc_set_state", "pmc_get_state",
    "pmc_set_state_all", "pmc_get_state_all", "pmc_energy", "pmc_energy_all", "pmc_observables",
    "pmc_delta_u", "pmc_run", "pmc_rows_for", "pmc_last_run_ms", "pmc_reinit", "pmc_averages",
    "pmc_accumulators", "pmc_diagnostics", "pmc_fp64_peak_probe", "pmc_launch_count",
    # ABI v2: the clustering driver (mcmc_clustering_eap_chain.jl)
    "pmc_energy_ex", "pmc_delta_segment", "pmc_run_ex", "pmc_begin_stage", "pmc_init_x0",
    "pmc_extra_averages", "pmc_extra_accumulators", "pmc_cluster_stats",
    # ABI v3: kernel name, checkpoints, double-double accumulators, one ensemble over several GPUs
    "pmc_kernel_name", "pmc_checkpoint_bytes", "pmc_checkpoint_save", "pmc_checkpoint_load", "pmc_accumulators_dd",
    "pmc_multi_create", "pmc_multi_destroy", "pmc_multi_num_devices", "pmc_multi_num_chains",
    "pmc_multi_gather_backend", "pmc_multi_shard", "pmc_multi_set_ensemble_hint", "pmc_multi_set_pair_precision", "pmc_multi_begin_stage",
    "pmc_multi_set_state_all", "pmc_multi_get_state_all", "pmc_multi_rows_for", "pmc_multi_run", "pmc_multi_run_ex",
    "pmc_multi_run_async", "pmc_multi_wait", "pmc_multi_gather", "pmc_multi_last_run_ms", "pmc_multi_launch_count",
    "pmc_release_cached_memory",
    # replica exchange across kT / force ladders of one handle
    "pmc_set_ladders", "pmc_exchange", "pmc_run_tempering", "pmc_run_tempering_ex", "pmc_exchange_stats",
    # conformation sampling: gyration tensor, bond-orientation correlation, orientation profile, extension histogram
    "pmc_set_conformation", "pmc_conformation_cols", "pmc_sample_conformation", "pmc_run_sampled", "pmc_run_sampled_ex",
    "pmc_conformation_sums",
]
RESULT_COLS = 24
RESULT_NAMES = AVG_NAMES + ["acc_rate", "normalizer", "phi_step", "theta_step", "trials", "U_running", "Ealign", "psi"]


class PolymcError(RuntimeError):
    """Raised for any non-zero pmc_status (mirrors the reference's `error(...)` convention,
    mcmc_eap_chain.jl:184,195)."""

    def __init__(self, code, msg):
        super().__init__(f"libpolymc_b200 error {code}: {msg}")
        self.code = code


class PmcCase(C.Structure):
    """Mirror of `pmc_case` (include/polymc.h): one command line of mcmc_eap_chain.jl:19-153."""
    _fields_ = [
        ("E0", C.c_double), ("K1", C.c_double), ("K2", C.c_double), ("mu", C.c_double),
        ("kT", C.c_double), ("Fz", C.c_double), ("Fx", C.c_double), ("b", C.c_double),
        ("phi_step", C.c_double), ("theta_step", C.c_double),
        ("adj_lb", C.c_double), ("adj_ub", C.c_double), ("adj_scale", C.c_double),
        ("n", C.c_int64), ("steps_per_adjust", C.c_int64),
        ("chain_type", C.c_int32), ("energy_type", C.c_int32),
        ("do_flips", C.c_int32), ("umbrella", C.c_int32),
        ("force_init", C.c_int32), ("accum_mode", C.c_int32),
        # mcmc_clustering_eap_chain.jl:36-51,87-90
        ("kappa", C.c_double), ("psi0", C.c_double), ("cutoff_radius", C.c_double), ("cluster_prob", C.c_double),
        ("clustering", C.c_int32), ("alpha_carry", C.c_int32), ("cutoff_full", C.c_int32), ("planar", C.c_int32),
    ]


def make_case(n=100, E0=0.0, K1=1.0, K2=0.0, mu=1e-2, kT=1.0, Fz=0.0, Fx=0.0, b=1.0,
              chain_type="dielectric", energy_type="noninteracting",
              phi_step=3 * math.pi / 8, theta_step=3 * math.pi / 16,
              adj_lb=0.15, adj_ub=0.55, adj_scale=1.1, steps_per_adjust=2500,
              do_flips=False, umbrella=False, force_init=False, accum_mode=0,
              kappa=0.0, psi0=0.0, cutoff_radius=7.5, cluster_prob=0.5, clustering=False, alpha_carry=True,
              cutoff_full=False, planar=False) -> PmcCase:
    """Defaults are the ArgParse defaults of mcmc_eap_chain.jl:19-153; the clustering fields default to
    "off" (kappa 0, clustering False) with the option defaults of mcmc_clustering_eap_chain.jl:48-51,87-90."""
    if chain_type not in CHAIN_TYPES:
        raise PolymcError(-1, "chain-type is not understood.")      # eap_chain.jl:86
    if energy_type not in ENERGY_TYPES:
        raise PolymcError(-1, "energy-type is not understood.")     # eap_chain.jl:104
    return PmcCase(E0, K1, K2, mu, kT, Fz, Fx, b, phi_step, theta_step, adj_lb, adj_ub, adj_scale,
                   n, steps_per_adjust, CHAIN_TYPES[chain_type], ENERGY_TYPES[energy_type],
                   int(do_flips), int(umbrella), int(force_init), int(accum_mode),
                   kappa, psi0, cutoff_radius, cluster_prob, int(clustering), int(alpha_carry), int(cutoff_full),
                   int(planar))


class CaseTable:
    """A contiguous array of `pmc_case` records — the form `pmc_create` takes, so handles are created from slices of it
    without copying, and the (n, energy_type) bucketing of a large sweep is vectorised.  Behaves like a read-only
    sequence of PmcCase; built once from a list (a phase-diagram grid has tens of thousands of cases)."""

    def __init__(self, cases=None, _rec=None):
        if _rec is not None:
            self.rec = _rec
        elif isinstance(cases, CaseTable):
            self.rec = cases.rec
        else:
            cases = [cases] if isinstance(cases, PmcCase) else list(cases)
            arr = (PmcCase * len(cases))(*cases)
            self.rec = np.frombuffer(arr, dtype=np.dtype(PmcCase)).copy() if cases else np.zeros(0, np.dtype(PmcCase))

    def __len__(self):
        return int(self.rec.shape[0])

    def __getitem__(self, i):
        if isinstance(i, slice):
            return CaseTable(_rec=self.rec[i])
        return PmcCase.from_buffer_copy(self.rec[i].tobytes())

    def __iter__(self):
        return (self[i] for i in range(len(self)))

    def column(self, name):
        return self.rec[name]

    def pointer(self):
        rec = self.rec if self.rec.flags["C_CONTIGUOUS"] else np.ascontiguousarray(self.rec)
        self._keep = rec
        return C.cast(rec.ctypes.data, C.POINTER(PmcCase))


def build(force: bool = False) -> str:
    """Compile libpolymc_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC_DIR, f) for f in os.listdir(CSRC_DIR) if f.endswith((".cu", ".cuh"))]
    srcs.append(os.path.join(os.path.dirname(_ROOT), "include", "polymc.h"))
    stale = (not os.path.exists(LIB_PATH)) or any(
        os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs if os.path.exists(s))
    if force or stale:
        subprocess.check_call(["make", "-C", CSRC_DIR, "-s"] + (["-B"] if force else []))
    return LIB_PATH


_lib = None


def load():
    """dlopen the library and declare the prototypes.  Fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PolymcError(-2, f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    dp = C.POINTER(C.c_double)
    hp = C.c_void_p
    L.pmc_abi_version.restype = C.c_int32
    L.pmc_last_error.restype = C.c_char_p
    L.pmc_device_count.argtypes = [C.POINTER(C.c_int32)]
    L.pmc_create.argtypes = [C.POINTER(PmcCase), C.c_int64, C.c_int32, C.c_uint64, C.c_int32, C.c_uint32,
                             C.POINTER(hp)]
    L.pmc_destroy.argtypes = [hp]
    L.pmc_destroy.restype = None
    L.pmc_set_pair_precision.argtypes = [hp, C.c_int32]
    L.pmc_pair_precision.argtypes = [hp]
    L.pmc_num_chains.argtypes = [hp]
    L.pmc_num_chains.restype = C.c_int64
    L.pmc_num_monomers.argtypes = [hp]
    L.pmc_num_monomers.restype = C.c_int64
    L.pmc_set_stream.argtypes = [hp, C.c_void_p]
    L.pmc_set_ensemble_hint.argtypes = [hp, C.c_int64]
    L.pmc_block_threads.argtypes = [hp]
    L.pmc_block_threads.restype = C.c_int32
    L.pmc_set_state.argtypes = [hp, C.c_int64, dp, dp]
    L.pmc_get_state.argtypes = [hp, C.c_int64, dp, dp]
    L.pmc_set_state_all.argtypes = [hp, dp, dp]
    L.pmc_get_state_all.argtypes = [hp, dp, dp]
    L.pmc_energy.argtypes = [hp, C.c_int64, dp]
    L.pmc_energy_all.argtypes = [hp, dp]
    L.pmc_observables.argtypes = [hp, C.c_int64, dp]
    L.pmc_delta_u.argtypes = [hp, C.c_int64, C.c_int64, C.c_double, C.c_double, dp]
    L.pmc_run.argtypes = [hp, C.c_int64, C.c_int64, dp, dp]
    L.pmc_rows_for.argtypes = [hp, C.c_int64, C.c_int64]
    L.pmc_rows_for.restype = C.c_int64
    L.pmc_last_run_ms.argtypes = [hp, C.POINTER(C.c_float)]
    L.pmc_launch_count.argtypes = [hp]
    L.pmc_launch_count.restype = C.c_int64
    L.pmc_reinit.argtypes = [hp, C.POINTER(C.c_int32)]
    L.pmc_averages.argtypes = [hp, dp, dp, dp]
    L.pmc_accumulators.argtypes = [hp, dp]
    L.pmc_diagnostics.argtypes = [hp, dp]
    L.pmc_fp64_peak_probe.argtypes = [C.c_int32, C.c_int32, dp, C.POINTER(C.c_float)]
    L.pmc_energy_ex.argtypes = [hp, C.c_int64, dp]
    L.pmc_delta_segment.argtypes = [hp, C.c_int64, C.c_int64, C.c_double, C.c_double, C.c_int32, C.c_int64,
                                    C.c_int64, dp]
    L.pmc_run_ex.argtypes = [hp, C.c_int64, C.c_int64, dp, dp, dp]
    L.pmc_begin_stage.argtypes = [hp, C.c_double]
    L.pmc_init_x0.argtypes = [hp, dp, C.c_int64, dp]
    L.pmc_extra_averages.argtypes = [hp, dp]
    L.pmc_extra_accumulators.argtypes = [hp, dp]
    L.pmc_cluster_stats.argtypes = [hp, dp]
    L.pmc_kernel_name.argtypes = [hp, C.c_char_p, C.c_int32]
    L.pmc_checkpoint_bytes.argtypes = [hp]
    L.pmc_checkpoint_bytes.restype = C.c_int64
    L.pmc_checkpoint_save.argtypes = [hp, C.c_void_p, C.c_int64]
    L.pmc_checkpoint_load.argtypes = [hp, C.c_void_p, C.c_int64]
    L.pmc_accumulators_dd.argtypes = [hp, dp, dp]
    L.pmc_multi_create.argtypes = [C.POINTER(PmcCase), C.c_int64, C.c_int32, C.c_uint64, C.POINTER(C.c_int32),
                                   C.c_int32, C.POINTER(hp)]
    L.pmc_multi_destroy.argtypes = [hp]
    L.pmc_multi_destroy.restype = None
    L.pmc_multi_num_devices.argtypes = [hp]
    L.pmc_multi_num_devices.restype = C.c_int32
    L.pmc_multi_num_chains.argtypes = [hp]
    L.pmc_multi_num_chains.restype = C.c_int64
    L.pmc_multi_gather_backend.argtypes = [hp]
    L.pmc_multi_gather_backend.restype = C.c_char_p
    L.pmc_multi_shard.argtypes = [hp, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.pmc_multi_shard.restype = C.c_void_p
    L.pmc_multi_set_ensemble_hint.argtypes = [hp, C.c_int64]
    L.pmc_multi_set_pair_precision.argtypes = [hp, C.c_int32]
    L.pmc_multi_begin_stage.argtypes = [hp, C.c_double]
    L.pmc_multi_set_state_all.argtypes = [hp, dp, dp]
    L.pmc_multi_get_state_all.argtypes = [hp, dp, dp]
    L.pmc_multi_rows_for.argtypes = [hp, C.c_int64, C.c_int64]
    L.pmc_multi_rows_for.restype = C.c_int64
    L.pmc_multi_run.argtypes = [hp, C.c_int64, C.c_int64, dp, dp]
    L.pmc_multi_run_ex.argtypes = [hp, C.c_int64, C.c_int64, dp, dp, dp]
    L.pmc_multi_run_async.argtypes = [hp, C.c_int64, C.c_int64, dp, dp]
    L.pmc_multi_wait.argtypes = [hp]
    L.pmc_multi_gather.argtypes = [hp, dp]
    L.pmc_multi_last_run_ms.argtypes = [hp, C.POINTER(C.c_float)]
    L.pmc_multi_launch_count.argtypes = [hp]
    L.pmc_multi_launch_count.restype = C.c_int64
    i64p = C.POINTER(C.c_int64)
    L.pmc_set_ladders.argtypes = [hp, C.POINTER(C.c_int32), C.c_int64]
    L.pmc_exchange.argtypes = [hp, C.POINTER(C.c_int32)]
    L.pmc_run_tempering.argtypes = [hp, C.c_int64, C.c_int64, C.c_int64, dp, dp]
    L.pmc_run_tempering_ex.argtypes = [hp, C.c_int64, C.c_int64, C.c_int64, dp, dp, dp]
    L.pmc_exchange_stats.argtypes = [hp, dp, i64p, i64p]
    L.pmc_set_conformation.argtypes = [hp, C.c_int32, C.c_int32]
    L.pmc_conformation_cols.argtypes = [hp]
    L.pmc_conformation_cols.restype = C.c_int64
    L.pmc_sample_conformation.argtypes = [hp]
    L.pmc_run_sampled.argtypes = [hp, C.c_int64, C.c_int64, C.c_int64, dp, dp]
    L.pmc_run_sampled_ex.argtypes = [hp, C.c_int64, C.c_int64, C.c_int64, dp, dp, dp]
    L.pmc_conformation_sums.argtypes = [hp, dp]
    for name in EXPORTS:
        f = getattr(L, name)
        if f.restype is C.c_int:  # default restype: every status-returning entry point
            f.restype = C.c_int32
    if L.pmc_abi_version() != 4:
        raise PolymcError(-1, "ABI version mismatch")
    _lib = L
    return L


def _check(rc):
    if rc != 0:
        raise PolymcError(rc, load().pmc_last_error().decode("utf-8", "replace"))


def _dp(a):
    if a is None:
        return None
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.POINTER(C.c_double))


def device_count() -> int:
    n = C.c_int32(0)
    rc = load().pmc_device_count(C.byref(n))
    return n.value if rc == 0 else 0


def release_cached_memory():
    """Return the library's cache of device blocks (kept across handles) to the driver."""
    _check(load().pmc_release_cached_memory())


def fp64_peak_probe(device=0, iters=1 << 17):
    t = C.c_double()
    ms = C.c_float()
    _check(load().pmc_fp64_peak_probe(device, iters, C.byref(t), C.byref(ms)))
    return t.value, ms.value


def conformation_averages(sums, n: int, bins: int) -> dict:
    """Averages of conformation sums [chains][8 + 3n + B] (pmc_conformation_sums, or rows of one case added up):
    S [chains][6] (S_xx S_yy S_zz S_xy S_xz S_yz), Rg2 = ⟨tr S⟩, Rg4 = ⟨(tr S)²⟩, bondcorr [chains][n] = ⟨C_s⟩/(n−s),
    nz, nz2 [chains][n] = ⟨n̂z_i⟩, ⟨n̂z_i²⟩, hist [chains][B] = the fraction of samples in each ζ bin, samples [chains]."""
    sums = np.asarray(sums, dtype=np.float64)
    if sums.shape[-1] != 8 + 3 * n + bins:
        raise PolymcError(-1, f"conformation rows have 8 + 3n + B = {8 + 3 * n + bins} columns, not {sums.shape[-1]}")
    k = sums[..., 0:1]
    S = sums[..., 1:7] / k
    return {"samples": sums[..., 0].copy(), "S": S, "Rg2": S[..., 0] + S[..., 1] + S[..., 2], "Rg4": sums[..., 7] / k[..., 0],
            "bondcorr": sums[..., 8:8 + n] / k / np.arange(n, 0, -1), "nz": sums[..., 8 + n:8 + 2 * n] / k,
            "nz2": sums[..., 8 + 2 * n:8 + 3 * n] / k, "hist": sums[..., 8 + 3 * n:] / k}


class Ensemble:
    """A batch of independent chains on one GPU: ncases × replicas, uniform n and energy type.

    The methods map 1:1 onto the C ABI; docstrings there cite the reference seams."""

    def __init__(self, cases, replicas=1, seed=0, device=0, chain_id_base=0, ensemble_chains=0):
        if isinstance(cases, PmcCase):
            cases = [cases]
        self.cases = cases if isinstance(cases, CaseTable) else list(cases)
        self.replicas = int(replicas)
        arr = self.cases.pointer() if isinstance(cases, CaseTable) else (PmcCase * len(self.cases))(*self.cases)
        h = C.c_void_p()
        _check(load().pmc_create(arr, len(self.cases), self.replicas, seed, device, chain_id_base, C.byref(h)))
        self._h = h
        self.nchains = int(load().pmc_num_chains(h))
        self.n = int(load().pmc_num_monomers(h))
        if ensemble_chains:
            self.set_ensemble_hint(ensemble_chains)

    def set_ensemble_hint(self, ensemble_chains: int):
        """Choose the launch shape for an ensemble of `ensemble_chains` chains (a shard passes the unsharded
        count so that results do not depend on the sharding, bit for bit); 0 = this handle's own count."""
        _check(load().pmc_set_ensemble_hint(self._h, int(ensemble_chains)))

    def set_pair_precision(self, precision: str):
        """"fp64" (default) or "fp32": the rectangle of a single-monomer trial in FP32 with the tolerance stated in
        include/polymc.h (pmc_set_pair_precision); launches without an FP32 kernel stay FP64."""
        if precision not in PAIR_PRECISIONS:
            raise PolymcError(-1, "pair-precision is not understood.")
        _check(load().pmc_set_pair_precision(self._h, PAIR_PRECISIONS[precision]))

    def pair_precision(self) -> str:
        """What the next run uses: "fp32" only where the FP32 kernel serves this handle."""
        return {v: k for k, v in PAIR_PRECISIONS.items()}[int(load().pmc_pair_precision(self._h))]

    def block_threads(self) -> int:
        return int(load().pmc_block_threads(self._h))

    def close(self):
        if getattr(self, "_h", None):
            load().pmc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_stream(self, cuda_stream_ptr: int):
        _check(load().pmc_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def set_state(self, chain, phi, theta):
        phi = np.ascontiguousarray(phi, dtype=np.float64)
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        if phi.shape != (self.n,) or theta.shape != (self.n,):
            raise PolymcError(-1, "state arrays must have num-monomers entries")
        _check(load().pmc_set_state(self._h, chain, _dp(phi), _dp(theta)))

    def get_state(self, chain):
        phi, theta = np.empty(self.n), np.empty(self.n)
        _check(load().pmc_get_state(self._h, chain, _dp(phi), _dp(theta)))
        return phi, theta

    def set_state_all(self, phi, theta):
        phi = np.ascontiguousarray(phi, dtype=np.float64)
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        if phi.shape != (self.nchains, self.n) or theta.shape != (self.nchains, self.n):
            raise PolymcError(-1, "state arrays must be [chains][num-monomers]")
        _check(load().pmc_set_state_all(self._h, _dp(phi), _dp(theta)))

    def get_state_all(self):
        phi, theta = np.empty((self.nchains, self.n)), np.empty((self.nchains, self.n))
        _check(load().pmc_get_state_all(self._h, _dp(phi), _dp(theta)))
        return phi, theta

    def energy(self, chain):
        o = np.empty(4)
        _check(load().pmc_energy(self._h, chain, _dp(o)))
        return {"U": o[0], "su": o[1], "Udd": o[2], "Omega": o[3]}

    def energy_all(self):
        o = np.empty((self.nchains, 4))
        _check(load().pmc_energy_all(self._h, _dp(o)))
        return o

    def observables(self, chain):
        o = np.empty(6)
        _check(load().pmc_observables(self._h, chain, _dp(o)))
        return o[:3].copy(), o[3:].copy()

    def delta_u(self, chain, idx0, dphi, dtheta):
        o = np.empty(3)
        _check(load().pmc_delta_u(self._h, chain, idx0, dphi, dtheta, _dp(o)))
        return {"dU": o[0], "dOmega": o[1], "clamped": bool(o[2])}

    def rows_for(self, nsteps, stepout):
        return int(load().pmc_rows_for(self._h, nsteps, stepout))

    def run(self, nsteps, stepout=0, fetch_rows=True, traj=None, roll=None):
        """The hot loop for every chain.  Returns (traj [chains][rows][8], roll [chains][rows][17])
        or (None, None) when fetch_rows is False (rows stay on the device)."""
        rows = self.rows_for(nsteps, stepout)
        if fetch_rows and rows > 0:
            if traj is None:
                traj = np.empty((self.nchains, rows, 8))
            if roll is None:
                roll = np.empty((self.nchains, rows, 17))
        else:
            traj = roll = None
        _check(load().pmc_run(self._h, nsteps, stepout, _dp(traj), _dp(roll)))
        return traj, roll

    def last_run_ms(self) -> float:
        ms = C.c_float()
        _check(load().pmc_last_run_ms(self._h, C.byref(ms)))
        return ms.value

    def launch_count(self) -> int:
        return int(load().pmc_launch_count(self._h))

    def kernel_name(self) -> str:
        """The MCMC kernel `run` launches for this handle as it is now (the library's own decision)."""
        buf = C.create_string_buffer(96)
        _check(load().pmc_kernel_name(self._h, buf, len(buf)))
        return buf.value.decode()

    def checkpoint(self) -> bytes:
        """Everything needed to continue this run in a later process (pmc_checkpoint_save)."""
        nb = int(load().pmc_checkpoint_bytes(self._h))
        buf = C.create_string_buffer(nb)
        _check(load().pmc_checkpoint_save(self._h, buf, nb))
        return buf.raw

    def restore(self, blob: bytes):
        buf = C.create_string_buffer(blob, len(blob))
        _check(load().pmc_checkpoint_load(self._h, buf, len(blob)))

    def accumulators_dd(self):
        """(hi, lo) [chains][19]: the double-double sums behind --numeric-type float128|dec128|big."""
        hi, lo = np.empty((self.nchains, 19)), np.empty((self.nchains, 19))
        _check(load().pmc_accumulators_dd(self._h, _dp(hi), _dp(lo)))
        return hi, lo

    def reinit(self):
        flags = (C.c_int32 * self.nchains)()
        _check(load().pmc_reinit(self._h, flags))
        return np.frombuffer(flags, dtype=np.int32).copy()

    def averages(self):
        avg = np.empty((self.nchains, 16))
        ar = np.empty(self.nchains)
        nrm = np.empty(self.nchains)
        _check(load().pmc_averages(self._h, _dp(avg), _dp(ar), _dp(nrm)))
        return avg, ar, nrm

    def accumulators(self):
        s = np.empty((self.nchains, 17))
        _check(load().pmc_accumulators(self._h, _dp(s)))
        return s

    def diagnostics(self):
        d = np.empty((self.nchains, 8))
        _check(load().pmc_diagnostics(self._h, _dp(d)))
        return d

    # ---- clustering driver (mcmc_clustering_eap_chain.jl), ABI v2 ----
    def energy_ex(self, chain):
        o = np.empty(8)
        _check(load().pmc_energy_ex(self._h, chain, _dp(o)))
        return {"U": o[0], "su": o[1], "Udd": o[2], "Omega": o[3], "Ubend": o[4], "psi": o[5], "cos2": o[6]}

    def delta_segment(self, chain, idx0, dphi, dtheta, reflect, lo0, hi0):
        o = np.empty(12)
        _check(load().pmc_delta_segment(self._h, chain, idx0, dphi, dtheta, int(reflect), lo0, hi0, _dp(o)))
        return dict(zip(["dU", "dOmega", "dpair", "du", "drF", "dbend", "dpsi", "dcos2", "dp1", "dp2", "dp3",
                         "log_alpha"], o))

    def run_ex(self, nsteps, stepout=0, fetch_rows=True, want_state=False):
        """The clustering driver's loop.  Returns (traj [chains][rows][8], roll [chains][rows][19],
        state [chains][rows][2n] or None)."""
        rows = self.rows_for(nsteps, stepout)
        traj = roll = state = None
        if fetch_rows and rows > 0:
            traj = np.empty((self.nchains, rows, 8))
            roll = np.empty((self.nchains, rows, 19))
            if want_state:
                state = np.empty((self.nchains, rows, 2 * self.n))
        _check(load().pmc_run_ex(self._h, nsteps, stepout, _dp(traj), _dp(roll), _dp(state)))
        return traj, roll, state

    def begin_stage(self, kT_scale=1.0):
        _check(load().pmc_begin_stage(self._h, float(kT_scale)))

    def init_x0(self, x0, dx0):
        x0 = np.ascontiguousarray(x0, dtype=np.float64).ravel()
        dx0 = np.ascontiguousarray(dx0, dtype=np.float64).ravel()
        if dx0.size != 2:
            raise PolymcError(-1, "Invalid input for 'dx0'")
        _check(load().pmc_init_x0(self._h, _dp(x0), x0.size, _dp(dx0)))

    def extra_averages(self):
        o = np.empty((self.nchains, 2))
        _check(load().pmc_extra_averages(self._h, _dp(o)))
        return o

    def extra_accumulators(self):
        o = np.empty((self.nchains, 2))
        _check(load().pmc_extra_accumulators(self._h, _dp(o)))
        return o

    def cluster_stats(self):
        o = np.empty((self.nchains, 3))
        _check(load().pmc_cluster_stats(self._h, _dp(o)))
        return o

    # ---- replica exchange across kT / force ladders (include/polymc.h, DESIGN.md §12) ----
    def set_ladders(self, ladders):
        """ladders: a list of lists of case indices, each in rung order (e.g. by increasing kT); [] clears.  Resets
        the round counter and the exchange diagnostics."""
        flat = []
        for lad in ladders:
            flat += [int(c) for c in lad] + [-1]
        arr = (C.c_int32 * max(1, len(flat)))(*flat)
        _check(load().pmc_set_ladders(self._h, arr, len(flat)))

    def exchange(self):
        """One exchange round; returns accepted [chains] (1 at the lower slot of every accepted pair)."""
        flags = (C.c_int32 * self.nchains)()
        _check(load().pmc_exchange(self._h, flags))
        return np.frombuffer(flags, dtype=np.int32).copy()

    def _tempering_rows(self, nsteps, exchange_every, stepout, fetch_rows, cols, want_state):
        if exchange_every < 1 or nsteps % exchange_every:
            raise PolymcError(-1, "exchange_every must divide nsteps")
        rows = self.rows_for(nsteps, stepout)
        if not (fetch_rows and rows > 0):
            return None, None, None
        return (np.empty((self.nchains, rows, 8)), np.empty((self.nchains, rows, cols)),
                np.empty((self.nchains, rows, 2 * self.n)) if want_state else None)

    def run_tempering(self, nsteps, exchange_every, stepout=0, fetch_rows=True):
        """run(exchange_every) followed by exchange(), nsteps / exchange_every times, on the device without host
        synchronisation between the chunks.  Returns (traj [chains][rows][8], roll [chains][rows][17]) as run()."""
        traj, roll, _ = self._tempering_rows(nsteps, exchange_every, stepout, fetch_rows, 17, False)
        _check(load().pmc_run_tempering(self._h, nsteps, exchange_every, stepout, _dp(traj), _dp(roll)))
        return traj, roll

    def run_tempering_ex(self, nsteps, exchange_every, stepout=0, fetch_rows=True, want_state=False):
        """The clustering driver's run_ex(exchange_every) followed by exchange(), repeated; rows as run_ex()."""
        traj, roll, state = self._tempering_rows(nsteps, exchange_every, stepout, fetch_rows, 19, want_state)
        _check(load().pmc_run_tempering_ex(self._h, nsteps, exchange_every, stepout, _dp(traj), _dp(roll), _dp(state)))
        return traj, roll, state

    def exchange_stats(self):
        """-> dict(attempts [ncases], accepts [ncases]: with the next rung, summed over replicas; walker [chains]:
        global chain id of the initial configuration each slot holds; round_trips [chains]: by walker)."""
        ncases = len(self.cases)
        if ncases * self.replicas != self.nchains:
            raise PolymcError(-1, "exchange_stats needs the handle's case list (a MultiEnsemble shard has none)")
        ps = np.empty((ncases, 2))
        walker = np.empty(self.nchains, dtype=np.int64)
        trips = np.empty(self.nchains, dtype=np.int64)
        i64p = C.POINTER(C.c_int64)
        _check(load().pmc_exchange_stats(self._h, _dp(ps), walker.ctypes.data_as(i64p), trips.ctypes.data_as(i64p)))
        return {"attempts": ps[:, 0].astype(np.int64), "accepts": ps[:, 1].astype(np.int64), "walker": walker,
                "round_trips": trips}

    # ---- conformation sampling (include/polymc.h, DESIGN.md §13) ----
    def set_conformation(self, hist_bins=0, enable=True):
        """Enable sampling of the chains' shape with an extension histogram of `hist_bins` bins (0: none) and zero the
        sums; enable=False disables it."""
        _check(load().pmc_set_conformation(self._h, int(bool(enable)), int(hist_bins)))

    def conformation_cols(self) -> int:
        return int(load().pmc_conformation_cols(self._h))

    def sample_conformation(self):
        """One sample of every chain's current configuration."""
        _check(load().pmc_sample_conformation(self._h))

    def _sampled_rows(self, nsteps, sample_every, stepout, fetch_rows, cols, want_state):
        if sample_every < 1 or nsteps % sample_every:
            raise PolymcError(-1, "sample_every must divide nsteps")
        return self._tempering_rows(nsteps, sample_every, stepout, fetch_rows, cols, want_state)

    def run_sampled(self, nsteps, sample_every, stepout=0, fetch_rows=True):
        """run(sample_every) followed by sample_conformation(), nsteps / sample_every times, on the device without host
        synchronisation between the chunks.  Returns (traj, roll) as run()."""
        traj, roll, _ = self._sampled_rows(nsteps, sample_every, stepout, fetch_rows, 17, False)
        _check(load().pmc_run_sampled(self._h, nsteps, sample_every, stepout, _dp(traj), _dp(roll)))
        return traj, roll

    def run_sampled_ex(self, nsteps, sample_every, stepout=0, fetch_rows=True, want_state=False):
        """The clustering driver's run_ex(sample_every) followed by sample_conformation(), repeated; rows as run_ex()."""
        traj, roll, state = self._sampled_rows(nsteps, sample_every, stepout, fetch_rows, 19, want_state)
        _check(load().pmc_run_sampled_ex(self._h, nsteps, sample_every, stepout, _dp(traj), _dp(roll), _dp(state)))
        return traj, roll, state

    def conformation_sums(self):
        """[chains][8 + 3n + B] running sums (include/polymc.h)."""
        cols = self.conformation_cols()
        if cols == 0:
            raise PolymcError(-1, "conformation sampling is not enabled (set_conformation)")
        s = np.empty((self.nchains, cols))
        _check(load().pmc_conformation_sums(self._h, _dp(s)))
        return s

    def conformation(self):
        """Per-chain averages of the samples (conformation_averages)."""
        s = self.conformation_sums()
        return conformation_averages(s, self.n, s.shape[1] - 8 - 3 * self.n)


class _Shard(Ensemble):
    """The single-device handle behind one slot of a MultiEnsemble (owned by it: close() is a no-op)."""

    def __init__(self, h, device, first, count, n):
        self._h = h
        self.device, self.first, self.nchains, self.n = device, first, count, n
        self.cases, self.replicas = [], 1

    def close(self):
        self._h = None


class MultiEnsemble:
    """One ensemble over several GPUs of one box through pmc_multi_*: contiguous blocks of global chain ids, one
    internal host thread per device, no data-path collective, one final NCCL all-gather of the result rows
    (replaces `julia -p N run/interacting_dielectric_study.jl`, :37-47)."""

    def __init__(self, cases, replicas=1, seed=0, devices=None, ndevices=0):
        if isinstance(cases, PmcCase):
            cases = [cases]
        self.cases = list(cases)
        self.replicas = int(replicas)
        arr = (PmcCase * len(self.cases))(*self.cases)
        dv = None
        if devices is not None:
            devices = list(devices)
            dv = (C.c_int32 * len(devices))(*devices)
            ndevices = len(devices)
        h = C.c_void_p()
        _check(load().pmc_multi_create(arr, len(self.cases), self.replicas, seed, dv, int(ndevices), C.byref(h)))
        self._h = h
        self.nchains = int(load().pmc_multi_num_chains(h))
        self.ndevices = int(load().pmc_multi_num_devices(h))
        self.n = int(self.cases[0].n)

    def close(self):
        if getattr(self, "_h", None):
            load().pmc_multi_destroy(self._h)
            self._h = None

    __del__ = Ensemble.__del__
    __enter__ = Ensemble.__enter__
    __exit__ = Ensemble.__exit__

    def gather_backend(self) -> str:
        return load().pmc_multi_gather_backend(self._h).decode()

    def shard(self, slot) -> _Shard:
        dev, first, cnt = C.c_int32(), C.c_int64(), C.c_int64()
        h = load().pmc_multi_shard(self._h, slot, C.byref(dev), C.byref(first), C.byref(cnt))
        if not h:
            _check(-1)
        return _Shard(C.c_void_p(h), dev.value, first.value, cnt.value, self.n)

    def set_ensemble_hint(self, chains):
        _check(load().pmc_multi_set_ensemble_hint(self._h, int(chains)))

    def set_pair_precision(self, precision: str):
        if precision not in PAIR_PRECISIONS:
            raise PolymcError(-1, "pair-precision is not understood.")
        _check(load().pmc_multi_set_pair_precision(self._h, PAIR_PRECISIONS[precision]))

    def begin_stage(self, kT_scale=1.0):
        _check(load().pmc_multi_begin_stage(self._h, float(kT_scale)))

    def set_state_all(self, phi, theta):
        phi = np.ascontiguousarray(phi, dtype=np.float64)
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        if phi.shape != (self.nchains, self.n) or theta.shape != (self.nchains, self.n):
            raise PolymcError(-1, "state arrays must be [chains][num-monomers]")
        _check(load().pmc_multi_set_state_all(self._h, _dp(phi), _dp(theta)))

    def get_state_all(self):
        phi, theta = np.empty((self.nchains, self.n)), np.empty((self.nchains, self.n))
        _check(load().pmc_multi_get_state_all(self._h, _dp(phi), _dp(theta)))
        return phi, theta

    def rows_for(self, nsteps, stepout):
        return int(load().pmc_multi_rows_for(self._h, nsteps, stepout))

    def _rows(self, nsteps, stepout, fetch_rows, traj, roll, cols):
        rows = self.rows_for(nsteps, stepout)
        if fetch_rows and rows > 0:
            if traj is None:
                traj = np.empty((self.nchains, rows, 8))
            if roll is None:
                roll = np.empty((self.nchains, rows, cols))
            return rows, traj, roll
        return rows, None, None

    def run(self, nsteps, stepout=0, fetch_rows=True, traj=None, roll=None):
        rows, traj, roll = self._rows(nsteps, stepout, fetch_rows, traj, roll, 17)
        _check(load().pmc_multi_run(self._h, nsteps, stepout, _dp(traj), _dp(roll)))
        return traj, roll

    def run_async(self, nsteps, stepout=0, fetch_rows=True, traj=None, roll=None):
        """Returns at once; the buffers are filled when wait() returns."""
        rows, traj, roll = self._rows(nsteps, stepout, fetch_rows, traj, roll, 17)
        _check(load().pmc_multi_run_async(self._h, nsteps, stepout, _dp(traj), _dp(roll)))
        return traj, roll

    def wait(self):
        _check(load().pmc_multi_wait(self._h))

    def run_ex(self, nsteps, stepout=0, fetch_rows=True, want_state=False):
        rows, traj, roll = self._rows(nsteps, stepout, fetch_rows, None, None, 19)
        state = np.empty((self.nchains, rows, 2 * self.n)) if (want_state and traj is not None) else None
        _check(load().pmc_multi_run_ex(self._h, nsteps, stepout, _dp(traj), _dp(roll), _dp(state)))
        return traj, roll, state

    def gather(self):
        """[chains][24] result rows (RESULT_NAMES), gathered device-to-device (NCCL) and read from the first device."""
        t = np.empty((self.nchains, RESULT_COLS))
        _check(load().pmc_multi_gather(self._h, _dp(t)))
        return t

    def averages(self):
        t = self.gather()
        return t[:, :16].copy(), t[:, 16].copy(), t[:, 17].copy()

    def last_run_ms(self) -> float:
        ms = C.c_float()
        _check(load().pmc_multi_last_run_ms(self._h, C.byref(ms)))
        return ms.value

    def launch_count(self) -> int:
        return int(load().pmc_multi_launch_count(self._h))
