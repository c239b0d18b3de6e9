/*
 * polymc.h — C ABI of libpolymc_b200.so: the B200 (sm_100a) fixed-force-ensemble MCMC hot path
 * of grasingerm/polymer-stats, i.e. everything inside `mcmc(nsteps, pargs)` of
 * mcmc_eap_chain.jl:171-376 for thousands of independent chains at once — and, since ABI version 2,
 * inside `mcmc(nsteps, pargs, chain)` of its clustering twin mcmc_clustering_eap_chain.jl:171-352
 * (cluster_flip!, bending energy, cut-off pair sum, burn-in stages; SURVEY.md §8f ranks 1-2).  ABI version 3
 * adds the multi-GPU ensemble (pmc_multi_*: one host thread per device, one final NCCL all-gather — the
 * fan-out of run/interacting_dielectric_study.jl:37-47), checkpoints and pmc_kernel_name.
 *
 * The reference has no FFI of its own (pure Julia).  The seams this ABI replaces are ordinary
 * Julia functions; each entry point below cites the one it stands in for.  A Julia host binds
 * these with `ccall` (see INTEGRATION.md and polymer-stats_b200/julia/mcmc_eap_chain.jl); the
 * Python host in polymer-stats_b200/polymc/ binds them with ctypes.
 *
 * Conventions
 *   - plain C, POD only; the caller owns every host buffer and passes pointer + implied length;
 *     the library owns all device memory behind the opaque handle.
 *   - every function returns 0 on success or a negative pmc_status; the message for the calling
 *     thread is available from pmc_last_error().  No exception or exit() crosses the boundary.
 *   - calls are synchronous (they return after the stream work has completed) and a handle is
 *     not re-entrant, like the single-threaded reference (`julia -t 1`).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     PMC_ERR_NO_DEVICE.
 *   - monomer indices are 0-based at this boundary (the Julia host passes idx-1).
 *   - one handle holds chains of ONE chain length n and ONE energy type (they select the
 *     kernel); all other parameters may differ per case.  Hosts bucket mixed sweeps by (n, energy).
 */
#ifndef POLYMC_H
#define POLYMC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PMC_ABI_VERSION 4

typedef enum pmc_status {
  PMC_OK = 0,
  PMC_ERR_INVALID = -1,    /* bad argument / unsupported option combination        */
  PMC_ERR_NO_DEVICE = -2,  /* no CUDA device, or device index out of range         */
  PMC_ERR_CUDA = -3,       /* a CUDA runtime call or kernel failed                 */
  PMC_ERR_NOMEM = -4,      /* host or device allocation failed                     */
  PMC_ERR_UNSUPPORTED = -5 /* chain too long for one CTA's shared memory, etc.     */
} pmc_status;

/* --chain-type (mcmc_eap_chain.jl:25-28; inc/eap_chain.jl:81-87) */
enum { PMC_CHAIN_DIELECTRIC = 0, PMC_CHAIN_POLAR = 1 };
/* --energy-type (mcmc_eap_chain.jl:41-44; inc/eap_chain.jl:95-105; "Ising" is accepted by the ctor) */
enum { PMC_ENERGY_NONINTERACTING = 0, PMC_ENERGY_INTERACTING = 1, PMC_ENERGY_ISING = 2,
       PMC_ENERGY_CUTOFF = 3 /* UCutoff, inc/eap_chain.jl:102,165-192; mcmc_clustering_eap_chain.jl:44-51 */ };

/* One case = one command line of mcmc_eap_chain.jl (ArgParse table :19-153). */
typedef struct pmc_case {
  double E0, K1, K2, mu, kT, Fz, Fx, b;   /* --E0 --K1 --K2 --mu --kT --Fz --Fx --mlen            */
  double phi_step, theta_step;            /* --phi-step --theta-step                              */
  double adj_lb, adj_ub, adj_scale;       /* --step-adjust-lb/-ub/-scale (scale 1.0 disables)     */
  int64_t n;                              /* --num-monomers                                       */
  int64_t steps_per_adjust;               /* --steps-per-adjust                                   */
  int32_t chain_type;                     /* PMC_CHAIN_*                                          */
  int32_t energy_type;                    /* PMC_ENERGY_*                                         */
  int32_t do_flips;                       /* --do-flips                                           */
  int32_t umbrella;                       /* --umbrella-sampling                                  */
  int32_t force_init;                     /* --force-init                                         */
  int32_t accum_mode;                     /* --numeric-type: 0 = float64 (plain sums, the reference default),
                                             1 = float128|dec128|big → Neumaier-compensated FP64 sums      */
  /* ---- mcmc_clustering_eap_chain.jl (ABI v2); all zero = the plain driver ---------------------- */
  double kappa, psi0;                     /* --bend-mod --bend-angle (:36-43; inc/eap_chain.jl:54-58,91-92)  */
  double cutoff_radius;                   /* --cutoff-radius, monomer lengths (:48-51; inc/eap_chain.jl:102)  */
  double cluster_prob;                    /* --cluster-prob (:87-90): cluster_flip! returns early (no flip)
                                             iff rand() <= cluster_prob (inc/eap_chain.jl:273)               */
  int32_t clustering;                     /* 1: the trial is move! + cluster_flip! with α in the acceptor
                                             (mcmc_clustering_eap_chain.jl:267-279) and the two extra
                                             averagers <Σcos²θ>, <Σψ/(n-1)> (:243-244) are recorded           */
  int32_t alpha_carry;                    /* 1 = reference: the acceptor stores logπ+log α as logπ_prev
                                             (inc/acceptance.jl:30-33); 0 = stores logπ (plain M-H)           */
  int32_t cutoff_full;                    /* 0 = reference: the UCutoff functor is the bare pair sum, without
                                             Σu and −r·F (inc/eap_chain.jl:171-192 vs inc/energy.jl:13-16);
                                             1 = Σu + U_cut − r·F                                             */
  int32_t planar;                         /* 1: the 2-D tree (2D/mcmc_clustering_eap_chain.jl, 2D/inc/eap_chain.jl): the state
                                             is phi only, n = (cos phi, sin phi) in the x-z plane (field along z),
                                             no solid-angle term, flip_n! = phi + pi, the cluster gate flips WITH
                                             probability cluster_prob (2D/inc/eap_chain.jl:233), and every stage starts
                                             from a NEW random chain (2D/mcmc_clustering_eap_chain.jl:151).  theta arrays
                                             at this boundary are ignored (read back as 0).  Requires clustering = 1.   */
} pmc_case;

typedef struct pmc_handle pmc_handle;

/* ---- library / device ------------------------------------------------------------------ */
int32_t pmc_abi_version(void);
const char* pmc_last_error(void);                 /* replaces Julia `error(...)` text, mcmc_eap_chain.jl:184,195 */
int32_t pmc_device_count(int32_t* count);

/* ---- life cycle ------------------------------------------------------------------------- */
/* Builds ncases*replicas_per_case chains on CUDA device `device` and draws their random initial
 * state (phi~U(0,2pi), theta~U(0,pi)) — replaces `EAPChain(pargs)`, inc/eap_chain.jl:60-135, and
 * the set-up half of mcmc(), mcmc_eap_chain.jl:171-265.  Chain c belongs to case c/replicas_per_case.
 * Its Philox stream is keyed by (seed, chain_id_base + c), so results do not depend on how a sweep
 * is sharded over GPUs. */
int32_t pmc_create(const pmc_case* cases, int64_t ncases, int32_t replicas_per_case, uint64_t seed,
                   int32_t device, uint32_t chain_id_base, pmc_handle** out);
void pmc_destroy(pmc_handle* h);
int64_t pmc_num_chains(const pmc_handle* h);
int64_t pmc_num_monomers(const pmc_handle* h);
/* Launch shape.  The block size of the CTA-per-chain kernels is chosen from the chain length AND the ensemble
 * size: a small ensemble leaves SMs idle, so each chain gets more warps (same Markov chain, same Philox stream;
 * only the order of the pair-sum reduction changes, i.e. results agree to rounding).  A sharded sweep passes the
 * UNSHARDED chain count of the ensemble here so that its results stay bit-identical however it is sharded
 * (polymc.sweep does); 0 = this handle's own chain count (the default).  No counterpart in the reference (its
 * launchers run one single-threaded process per case, run/K1_Fz_long.jl:45). */
int32_t pmc_set_ensemble_hint(pmc_handle* h, int64_t ensemble_chains);
/* Precision of the dipole–dipole pair sums of a single-monomer trial (ABI v4).  PMC_PAIR_FP64 (the default) evaluates
 * every changed pair in FP64 — the reference's Float64 (inc/eap_chain.jl:196-211).  PMC_PAIR_FP32 evaluates the
 * RECTANGLE of a trial — the idx·(n−1−idx) pairs (i < idx < j) whose dipoles are unchanged and whose separation
 * changes by the rigid translation of the tail — in FP32 from positions mirrored relative to the rotated monomer, and
 * everything else (the row {idx}×rest, state, running energy, acceptance test, accumulators) in FP64 as before.
 * Stated tolerance (tests/test_gpu_fp32.py): every pair term of the rectangle carries an error of at most
 * 2e-6 · (1 + a) · m, m = (|μi·μj| + 3|μi·r̂||μj·r̂|) / (4π r³) the magnitude of its two parts, a = (|r| + |D|) / |r − D|
 * for the new term (a ≲ 2 unless the trial brings the two monomers much closer than they were — then the new term is
 * huge and decides the trial by itself) and a = 0 for the old one, i.e.
 * |ΔU_fp32 − ΔU_fp64| ≤ 2e-6 · Σ_pairs (m_old + (1 + a) m_new): a few 1e-6 of the pair-term magnitudes of the trial.
 * Use it while that is small against kT — extended or coiled chains.  Chains that have collapsed onto themselves
 * (|U| of 1e5 kT and more, where point dipoles without excluded volume end up at low temperature) need FP64; the
 * library re-synchronises the running energy with an FP64 evaluation after every FP32 launch and pmc_diagnostics
 * column 7 reports the largest drift it found, a direct measure of the accumulated error.  Averages agree with the FP64
 * path within 3σ and a few hundred trials reproduce its decisions (same test); long trajectories are not
 * decision-identical.  Served by the windowed CTA-per-chain kernel of interacting chains of the plain
 * driver on one SM per chain (n ≤ 768 in a full ensemble); every other launch ignores the setting and stays FP64.  pmc_pair_precision returns what the
 * next pmc_run will use.  No counterpart in the reference. */
#define PMC_PAIR_FP64 0
#define PMC_PAIR_FP32 1
int32_t pmc_set_pair_precision(pmc_handle* h, int32_t mode);
int32_t pmc_pair_precision(const pmc_handle* h);
int32_t pmc_block_threads(const pmc_handle* h);   /* the block size in use (diagnostics) */
/* Work is enqueued on `cuda_stream` (a cudaStream_t; NULL = the legacy default stream). */
int32_t pmc_set_stream(pmc_handle* h, void* cuda_stream);

/* ---- state ------------------------------------------------------------------------------ */
/* Overwrite / read the independent state (phi, theta), n doubles each — the fields `ϕs`, `θs` of
 * EAPChain (inc/eap_chain.jl:22,25); all caches are rebuilt on device.  *_all: [chains][n]. */
int32_t pmc_set_state(pmc_handle* h, int64_t chain, const double* phi, const double* theta);
int32_t pmc_get_state(pmc_handle* h, int64_t chain, double* phi, double* theta);
int32_t pmc_set_state_all(pmc_handle* h, const double* phi, const double* theta);
int32_t pmc_get_state_all(pmc_handle* h, double* phi, double* theta);

/* ---- energies (parity seams) ------------------------------------------------------------ */
/* out[4] = {U, sum(us), U_dipole_dipole, Omega}: `U(chain)` inc/eap_chain.jl:411 → inc/energy.jl:7-23
 * with U_interaction :196-211 / U_Ising :215-228; Omega = Σ log sin θ (fix of :117, see DESIGN.md). */
int32_t pmc_energy(pmc_handle* h, int64_t chain, double out[4]);
int32_t pmc_energy_all(pmc_handle* h, double* out /* [chains][4] */);
/* Observables of the current state: out[6] = {r1,r2,r3,p1,p2,p3} — end_to_end :405, chain_μ :408. */
int32_t pmc_observables(pmc_handle* h, int64_t chain, double out[6]);
/* Energy change of the single-monomer trial `move!(trial, idx, dphi, dtheta)` (inc/eap_chain.jl:230-257)
 * WITHOUT mutating the chain: out[3] = {dU, dOmega, theta_was_clamped}.  Same device code as pmc_run. */
int32_t pmc_delta_u(pmc_handle* h, int64_t chain, int64_t idx0, double dphi, double dtheta, double out[3]);

/* out[8] = {U, sum(us) incl. bending, U_dipole_dipole, Omega, U_bend, sum(psi)/(n-1), sum(cos^2 theta), 0}:
 * the pieces of `U(chain)` with `ubend` (inc/eap_chain.jl:54-58,130) and UCutoff (:171-192), and the
 * accessors of the two extra averagers (mcmc_clustering_eap_chain.jl:243-244). */
int32_t pmc_energy_ex(pmc_handle* h, int64_t chain, double out[8]);
/* The composite trial of the clustering driver WITHOUT mutating the chain — `move!(trial, idx, dphi,
 * dtheta)` followed, if reflect, by `refl_n!(trial, i)` for i in [lo0,hi0] (inc/eap_chain.jl:263-265,
 * 311-315; lo0 <= idx0 <= hi0, 0-based): out[12] = {dU, dOmega, dU_pairs, du_self, -dr·F, dU_bend,
 * d sum(psi), d sum(cos^2 theta), dp1, dp2, dp3, log(alpha)} with alpha of inc/eap_chain.jl:317-330.
 * Same device code as pmc_run on a clustering handle. */
int32_t pmc_delta_segment(pmc_handle* h, int64_t chain, int64_t idx0, double dphi, double dtheta, int32_t reflect,
                          int64_t lo0, int64_t hi0, double out[12]);

/* ---- the hot loop ------------------------------------------------------------------------ */
/* Runs `nsteps` Metropolis trials on every chain — the `for step=1:nsteps` loop,
 * mcmc_eap_chain.jl:276-350: proposal :277-280, ΔU (replacing the deep copy + full recompute
 * :281-283), Metropolis inc/acceptance.jl:29-37, step adaptation :301-322, the 8 averagers
 * :327-328 (inc/average.jl:40-48, umbrella :63-97) and, every `stepout` steps, one trajectory row
 * (step,r1..3,p1..3,U) :330-333 and one rolling row (step + 16 running averages) :334-346.
 * traj: [chains][rows][8], roll: [chains][rows][17], rows = number of multiples of stepout in
 * (step0, step0+nsteps]; either may be NULL (rows are then left on the device).  stepout<=0: no rows.
 * The step counter continues across calls within one init. */
int32_t pmc_run(pmc_handle* h, int64_t nsteps, int64_t stepout, double* traj, double* roll);
int64_t pmc_rows_for(const pmc_handle* h, int64_t nsteps, int64_t stepout);
/* The loop of the clustering driver, mcmc_clustering_eap_chain.jl:267-336 (handles whose cases set
 * clustering, kappa or PMC_ENERGY_CUTOFF): roll19 [chains][rows][19] = step + 16 averages + Ealign + psi
 * (:259,:334-346); state [chains][rows][2n] = phi1,theta1,phi2,theta2,… of each trajectory row (:317; the
 * mu columns :318 are a function of these and are filled in by the host).  Any pointer may be NULL.
 * pmc_run on such a handle runs the same loop and returns the first 17 rolling columns. */
int32_t pmc_run_ex(pmc_handle* h, int64_t nsteps, int64_t stepout, double* traj, double* roll19, double* state);
/* A fresh `mcmc(nsteps, pargs, chain)` call on the chains as they are (mcmc_clustering_eap_chain.jl:171-265,
 * the burn-in ladder :365-386): kT = kT_case * kT_scale, chain.U = U(chain), new weight function, acceptor,
 * averagers, counters; step sizes restart from --phi-step/--theta-step (burnargs is a copy of pargs, :368);
 * the step counter restarts and a fresh random stream is used. */
int32_t pmc_begin_stage(pmc_handle* h, double kT_scale);
/* `EAPChain(pargs)` with --x0/--dx0 (inc/eap_chain.jl:63-78): phi = phi0 + U(0,dx0[0]), theta = theta0 +
 * U(0,dx0[1]); x0 holds {phi0, theta0} (x0_len 2) or 2n interleaved values. */
int32_t pmc_init_x0(pmc_handle* h, const double* x0, int64_t x0_len, const double dx0[2]);
/* Device time of the last pmc_run's MCMC kernel, CUDA events on the handle's stream. */
int32_t pmc_last_run_ms(const pmc_handle* h, float* ms);
/* Number of CUDA kernels this handle has launched so far (bench.py's `gpu_launches`). */
int64_t pmc_launch_count(const pmc_handle* h);
/* Name of the MCMC kernel pmc_run / pmc_run_ex launches for this handle as it is now (driver, energy type, chain
 * length, ensemble size and hint select it), e.g. "k_run_cta_win<128,4,2>".  The library's own launch decision,
 * taken without launching anything. */
int32_t pmc_kernel_name(pmc_handle* h, char* buf, int32_t buflen);

/* Re-initialisation between inits, mcmc_eap_chain.jl:352-361 (metropolis_acc, inc/acceptance.jl:1-3):
 * draws a fresh random chain per chain and swaps it in iff force_init or
 * eps <= exp(-dU/kT) Π sinθ_new / Π sinθ_old.  replaced: [chains] 0/1, may be NULL.  Restarts the
 * step counter; accumulators keep accumulating. */
int32_t pmc_reinit(pmc_handle* h, int32_t* replaced);

/* ---- results ----------------------------------------------------------------------------- */
/* get_avg of the 8 averagers (inc/average.jl:38): avg [chains][16] in rolling.csv column order
 * (r1,r2,r3,r1sq,r2sq,r3sq,rsq,p1,p2,p3,p1sq,p2sq,p3sq,psq,U,Usq); acc_rate [chains] = nacc_total /
 * trials (mcmc_eap_chain.jl:365); normalizer [chains] = Σ of averaging weights (trial count unless
 * umbrella).  Any pointer may be NULL. */
int32_t pmc_averages(pmc_handle* h, double* avg, double* acc_rate, double* normalizer);
/* Raw accumulators for pooling replicas exactly: sums [chains][17] (16 sums + normaliser). */
int32_t pmc_accumulators(pmc_handle* h, double* sums);
/* The two extra averagers of the clustering driver (mcmc_clustering_eap_chain.jl:243-244, printed :398-399):
 * ex [chains][2] = {<sum cos^2 theta>, <sum(psi)/(n-1)>}; raw sums for pooling: sums [chains][2]. */
int32_t pmc_extra_averages(pmc_handle* h, double* ex);
int32_t pmc_extra_accumulators(pmc_handle* h, double* sums);
/* out [chains][3] = {trials with a cluster flip, sum of cluster sizes, largest cluster} of the current stage. */
int32_t pmc_cluster_stats(pmc_handle* h, double* out);
/* diag [chains][8] = {phi_step, theta_step, nacc, natt, nacc_total, trials, U_running, max |U_running -
 * U_recomputed| seen at re-synchronisation}. */
int32_t pmc_diagnostics(pmc_handle* h, double* diag);

/* ---- checkpoint / resume ------------------------------------------------------------------ */
/* Everything a later process needs to continue the run exactly where it stopped: the chain records (phi, theta
 * and caches), the running scalars, step sizes, counters, the 17+2 accumulators (both parts of the compensated
 * sums), the init / stage number and the stage temperature.  The reference has no checkpointing (a killed
 * `julia mcmc_eap_chain.jl` starts over); its closest seam is --x0 (inc/eap_chain.jl:63-78), which restores
 * angles only.  Load into a handle created with the same cases, replicas, seed and chain_id_base; continuing
 * with pmc_run then gives bit-identical results to an uninterrupted run. */
int64_t pmc_checkpoint_bytes(const pmc_handle* h);
int32_t pmc_checkpoint_save(pmc_handle* h, void* buf, int64_t bytes);
int32_t pmc_checkpoint_load(pmc_handle* h, const void* buf, int64_t bytes);

/* Both parts of the error-free-transformation sums: value = hi + lo with |lo| <= ulp(hi), i.e. double-double
 * accumulators — what `--numeric-type float128|dec128|big` asks of the averagers (mcmc_eap_chain.jl:186-197,
 * inc/average.jl:8-48).  hi, lo: [chains][19] = the 16 sums, the normaliser, and the two extra sums of the
 * clustering driver. */
int32_t pmc_accumulators_dd(pmc_handle* h, double* hi, double* lo);

/* ---- replica exchange (parallel tempering) across kT and force ladders of one handle --------- */
/* A new capability: the reference has no exchange, and a handle without ladders runs exactly as before.
 *
 * Ladder.  An ordered list of case indices of this handle, the rungs.  Replica r of rung k pairs with replica r of
 * rung k+1, so R replicas per case hold R independent copies of every ladder.  A case is in at most one ladder; cases
 * outside every ladder run as usual.  The rungs of a ladder agree on every field that enters the energy or the target
 * density (E0, K1, K2, mu, b, n, chain_type, energy_type, kappa, psi0, cutoff_radius, cutoff_full, clustering, planar)
 * and may differ in kT, Fz, Fx and the proposal / protocol fields (step sizes, adj_*, steps_per_adjust, do_flips,
 * cluster_prob, accum_mode, alpha_carry, force_init).  PMC_ERR_INVALID, with a message, for umbrella = 1 (its weight
 * function depends on kT and F), for rungs whose Fz / Fx differ under PMC_ENERGY_CUTOFF with cutoff_full = 0 (F is then
 * not part of the energy), for a case index out of range or repeated, for a ladder of fewer than two rungs and for any
 * mismatch in the fields above.  Ladders are a single-handle feature: pmc_multi_* has no exchange, and on a
 * pmc_multi_shard handle the rungs are that shard's own case indices.
 *
 * Exchange rule.  Slot s samples π_s(x) ∝ exp(−U_s(x)/kT_s)·Ω(x), U_s the running energy of the run kernels
 * (U_s(x) = U₀(x) − r(x)·F_s when F enters the energy).  A swap of slots a and b is accepted iff Δ ≥ 0 (no draw) or
 * ε < exp(Δ), Δ = β_a [U_a(x_a) − U_a(x_b)] + β_b [U_b(x_b) − U_b(x_a)], U_a(x_b) = U_b(x_b) + r_b·(F_b − F_a),
 * β = 1/kT of the stage (pmc_begin_stage's scale included).  Ω and the bending energy cancel.
 *
 * Pairing.  Round k (counted per handle from 0) attempts the pairs (rung i, rung i+1) with i ≡ k (mod 2) in every
 * ladder and replica column.  ε comes from Philox stream 7 at position k of the lower-rung chain (DESIGN.md §4); the
 * trial streams are untouched, a slot keeps drawing its own stream whatever configuration it holds.
 *
 * What moves.  With the configuration: the monomer records, Ω, Σu, r, p, the clustering driver's Σψ and Σcos²θ, and
 * U (re-expressed for the new slot by the formula above).  With the slot (its temperature or force): accumulators,
 * step sizes, counters, drift_max and cluster statistics, so the averages of a case are the averages of its rung.
 * The acceptor is re-bound to the slot's new configuration (α carry 0, the rule for alpha_carry = 1), as
 * pmc_begin_stage does.  pmc_reinit and pmc_begin_stage leave ladders, labels and statistics as they are.
 *
 * pmc_set_ladders: rungs = case indices in rung order, ladders separated by -1 (a trailing -1 is allowed); len 0
 * clears.  Resets the round counter and the diagnostics.
 * pmc_exchange: one round.  accepted [chains] (may be NULL): 1 at the lower slot of each accepted pair, else 0.
 * pmc_run_tempering / _ex: pmc_run / pmc_run_ex (exchange_every) followed by pmc_exchange, nsteps / exchange_every
 * times, bit-identical to that loop, rows included, without host synchronisation between the chunks.  exchange_every
 * must divide nsteps and stepout must divide exchange_every (or be <= 0: no rows).  Rows as pmc_run / pmc_run_ex over
 * all nsteps.
 * pmc_exchange_stats, any pointer may be NULL: pair_stats [ncases][2] = attempts, accepts of (case, its next rung),
 * summed over replicas (0 for top rungs and cases outside ladders); walker [chains] = the global chain id whose initial
 * configuration the slot now holds (a permutation within every ladder column); round_trips [chains], by walker (index =
 * label − chain_id_base) = completed bottom → top → bottom trips.
 * With ladders set, pmc_checkpoint_save appends the ladders, the round counter, the statistics and the walker labels
 * and round-trip state; pmc_checkpoint_load requires the same ladders.  Without ladders checkpoints are unchanged. */
int32_t pmc_set_ladders(pmc_handle* h, const int32_t* rungs, int64_t len);
int32_t pmc_exchange(pmc_handle* h, int32_t* accepted);
int32_t pmc_run_tempering(pmc_handle* h, int64_t nsteps, int64_t exchange_every, int64_t stepout, double* traj, double* roll);
int32_t pmc_run_tempering_ex(pmc_handle* h, int64_t nsteps, int64_t exchange_every, int64_t stepout,
                             double* traj, double* roll19, double* state);
int32_t pmc_exchange_stats(pmc_handle* h, double* pair_stats, int64_t* walker, int64_t* round_trips);

/* ---- conformation sampling: the shape of every chain, sampled on the device (DESIGN.md §13) ---- */
/* A new capability: the reference measures only whole-chain scalars, and a handle without sampling runs as before.
 * Per chain the device keeps plain FP64 running sums over samples, cols = 8 + 3n + B doubles (x_i = monomer centres,
 * n̂_i the record's direction; averages = sums / col 0; replicas of one case pool by adding rows):
 *   0: 1 (the sample count) · 1–6: S_xx S_yy S_zz S_xy S_xz S_yz of the gyration tensor S = (1/n) Σ_i (x_i − x̄)(x_i − x̄)ᵀ
 *   7: (tr S)² · 8 + s, s = 0 … n−1: C_s = Σ_{i=0}^{n−1−s} n̂_i·n̂_{i+s} · 8 + n + i: n̂z_i · 8 + 2n + i: n̂z_i²
 *   8 + 3n + k, k < B: histogram of ζ = r_z / (n b) on [−1, 1], bin k = min(B−1, max(0, ⌊(ζ+1)·B/2⌋)), r_z as
 *   pmc_observables computes it.
 * pmc_set_conformation: enable != 0 enables sampling with B = hist_bins (0: no histogram, at most 65536) and zeroes the
 * sums; enable = 0 disables it and frees the sums.  PMC_ERR_INVALID for any umbrella case in the handle (its samples
 * would need the umbrella weights) and for hist_bins out of range.
 * pmc_conformation_cols: 8 + 3n + B, or 0 when disabled.
 * pmc_sample_conformation: one sample of every chain's current configuration.
 * pmc_run_sampled / _ex: pmc_run / pmc_run_ex (sample_every) followed by pmc_sample_conformation, nsteps / sample_every
 * times, bit-identical to that loop, rows included, without host synchronisation between the chunks; preconditions and
 * rows as pmc_run_tempering*.  With sampling enabled, pmc_run_tempering* also samples after every exchange round
 * (pmc_run; pmc_exchange; pmc_sample_conformation, repeated).  pmc_run / pmc_run_ex never sample.
 * pmc_conformation_sums: sums [chains][cols].
 * pmc_begin_stage zeroes the sums; pmc_reinit keeps them; pmc_exchange leaves them with the slot (a case's averages are
 * those of its rung).  With sampling enabled pmc_checkpoint_save appends B and the sums after the ladder block, and
 * pmc_checkpoint_load requires the same setting; without it checkpoints are unchanged.  pmc_multi_* has no sampling
 * of its own: enable it on each shard (pmc_multi_shard). */
int32_t pmc_set_conformation(pmc_handle* h, int32_t enable, int32_t hist_bins);
int64_t pmc_conformation_cols(const pmc_handle* h);
int32_t pmc_sample_conformation(pmc_handle* h);
int32_t pmc_run_sampled(pmc_handle* h, int64_t nsteps, int64_t sample_every, int64_t stepout, double* traj, double* roll);
int32_t pmc_run_sampled_ex(pmc_handle* h, int64_t nsteps, int64_t sample_every, int64_t stepout,
                           double* traj, double* roll19, double* state);
int32_t pmc_conformation_sums(pmc_handle* h, double* sums);

/* ---- one ensemble over several GPUs of one box (ABI v3) ------------------------------------ */
/* Replaces the fan-out of the reference's launchers — `julia -p N run/interacting_dielectric_study.jl workdir`,
 * run/interacting_dielectric_study.jl:37-47 (pmap over cases, one single-threaded process per case).  The
 * ncases*replicas_per_case chains are split into contiguous blocks of global chain ids, one per device (device g
 * owns [g·R/G, (g+1)·R/G)); Philox streams are keyed by the global id, so results do not depend on the number of
 * devices.  Every device is driven from its own internal host thread; there is no data-path collective.  The only
 * exchange is pmc_multi_gather: the final per-chain result rows, one ncclAllGather over NVLink (libnccl.so.2 is
 * opened with dlopen; without it the rows travel by device-to-device copies).
 * All cases must share n, the energy type and the driver (plain / composite trials / 2-D) — PMC_ERR_INVALID otherwise —
 * so that the kernel a case runs on does not depend on which other cases share its device.
 * devices = NULL: devices 0..ndevices-1; ndevices <= 0: every device of the box. */
typedef struct pmc_multi pmc_multi;
#define PMC_RESULT_COLS 24 /* one gathered row: 16 averages (rolling.csv order), acc_rate, normalizer, phi_step,
                              theta_step, trials, U_running, <sum cos^2 theta>, <sum(psi)/(n-1)>               */
int32_t pmc_multi_create(const pmc_case* cases, int64_t ncases, int32_t replicas_per_case, uint64_t seed,
                         const int32_t* devices, int32_t ndevices, pmc_multi** out);
void pmc_multi_destroy(pmc_multi* m);
int32_t pmc_multi_num_devices(const pmc_multi* m);
int64_t pmc_multi_num_chains(const pmc_multi* m);
const char* pmc_multi_gather_backend(const pmc_multi* m);   /* "nccl", "peer" or "none" (one device) */
/* The single-device handle behind slot `slot` (for the per-chain seams: pmc_set_state, pmc_energy, pmc_delta_u,
 * pmc_reinit, pmc_checkpoint_*, ...), the device it lives on and its block of global chain ids. */
pmc_handle* pmc_multi_shard(pmc_multi* m, int32_t slot, int32_t* device, int64_t* first_chain, int64_t* nchains);
int32_t pmc_multi_set_ensemble_hint(pmc_multi* m, int64_t ensemble_chains);
int32_t pmc_multi_set_pair_precision(pmc_multi* m, int32_t mode);   /* pmc_set_pair_precision on every device handle */
int32_t pmc_multi_begin_stage(pmc_multi* m, double kT_scale);
int32_t pmc_multi_set_state_all(pmc_multi* m, const double* phi, const double* theta);   /* [chains][n] */
int32_t pmc_multi_get_state_all(pmc_multi* m, double* phi, double* theta);
int64_t pmc_multi_rows_for(const pmc_multi* m, int64_t nsteps, int64_t stepout);
/* pmc_run / pmc_run_ex on every device at once; traj/roll/state are [chains][rows][...] over the WHOLE ensemble
 * and every device fills its own slice.  _async returns at once (the host may format the previous interval's
 * rows meanwhile); pmc_multi_wait joins and reports the first error. */
int32_t pmc_multi_run(pmc_multi* m, int64_t nsteps, int64_t stepout, double* traj, double* roll);
int32_t pmc_multi_run_ex(pmc_multi* m, int64_t nsteps, int64_t stepout, double* traj, double* roll19, double* state);
int32_t pmc_multi_run_async(pmc_multi* m, int64_t nsteps, int64_t stepout, double* traj, double* roll);
int32_t pmc_multi_wait(pmc_multi* m);
/* table [chains][PMC_RESULT_COLS]: packed on each device, gathered device-to-device, read from the first device. */
int32_t pmc_multi_gather(pmc_multi* m, double* table);
int32_t pmc_multi_last_run_ms(const pmc_multi* m, float* ms_max);   /* slowest device's MCMC kernel time */
int64_t pmc_multi_launch_count(const pmc_multi* m);

/* Device memory of destroyed handles is kept in a per-process cache and reused by the next pmc_create (a study
 * creates one handle per bucket per call); this returns the cached blocks to the driver.  No reference counterpart. */
int32_t pmc_release_cached_memory(void);

/* ---- measurement helper ------------------------------------------------------------------ */
/* Dependent-free DFMA loop on all SMs of `device`; returns achieved FP64 TFLOP/s (2 flop per DFMA)
 * and the device time in ms.  Used by bench.py as the measured FP64 roofline denominator. */
int32_t pmc_fp64_peak_probe(int32_t device, int32_t iters, double* tflops, float* ms);

#ifdef __cplusplus
}
#endif
#endif /* POLYMC_H */
