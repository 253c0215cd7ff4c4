/* afesp_gpu.h -- C ABI of the B200-native coupled-cluster engine (libafesp_gpu.so).
 *
 * Drop-in boundary for the coupled-cluster hot path of AFESP (brianz98/A-Fortran-Electronic-Structure-Programme).
 * The reference has no FFI today; the boundary sits at the call sites of src/main.F90 that enter the hot path
 * (do_mp2_spatial :60/:98, do_ccsd_spinorb :67, do_ccsd_spatial :105, do_ccsd_t_spinorb[_acc] :75-79,
 * do_ccsd_t_spatial :112) and follows the only precedent in the reference for handing plain arrays to an
 * accelerator routine, do_ccsd_t_spinorb_acc (src/ccsd.f90:1924-1938; selected by `#ifdef OPENACC`, main.F90:74).
 * shim/afesp_gpu.f90 holds the ISO_C_BINDING interfaces and INTEGRATION.md the edited call sites.
 *
 * Conventions (what a Fortran caller needs):
 *   - every function returns an int status: 0 = ok, non-zero = failure (1 bad argument/state, 2 CUDA error,
 *     3 linear solve failed, 4 NCCL error, 5 the reference's own run-time assertion on the integrals failed); afesp_gpu_last_error() gives the text.  The shim maps a non-zero
 *     status to `call error('afesp_gpu::<fn>', msg)` -> stderr + stop 999 (src/error_handling.f90:7-20).
 *   - scalars by value; arrays are caller-owned, contiguous, column-major real(c_double), never retained after the
 *     call returns; a NULL output pointer means "do not copy back".
 *   - the library prints nothing: the host program keeps every line of els.out.
 *   - one handle = one CUDA device; all state between calls (integrals, amplitudes, intermediates, DIIS history)
 *     stays on that device.  Calls on one handle must not overlap (the caller is single-threaded, main.F90).
 *     At most ONE open handle per device and process (a second afesp_gpu_open on the same device fails until the first
 *     is closed); handles on different devices of one process are independent.  The kernel-selection and measurement
 *     options ("gemm_use_tma", "gemm_force_config", "gemm_tma_edge", "gemm_timing") are process-wide.
 *   - there is no CPU fallback: without a usable CUDA device afesp_gpu_open fails.
 *
 * Packed two-electron integrals use the reference's 8-fold canonical order (src/integrals.f90:196-210):
 *   pair(i,j) = i(i-1)/2 + j (1-based, i >= j);  eri[pair(pair(i,j), pair(k,l))] = (ij|kl); length npair(npair+1)/2.
 */
#ifndef AFESP_GPU_H
#define AFESP_GPU_H

#ifdef __cplusplus
extern "C" {
#endif

typedef void* afesp_handle;

/* Context ------------------------------------------------------------------------------------------------------ */
int afesp_gpu_open(int device, afesp_handle* h);
int afesp_gpu_close(afesp_handle h);
const char* afesp_gpu_last_error(afesp_handle h); /* h may be NULL: error of the last failed afesp_gpu_open */
/* Parity switches (SURVEY.md App. B), all default to the reference's as-coded behaviour (value 1):
 *   "q1_transposed_foo"        spin-orbital F_mi dgemm term lands transposed (src/ccsd.f90:793-795)
 *   "q3a_truncated_e"          `do e = 1, nocc` over a virtual index in I_ooov_pp (src/ccsd.f90:2535)
 *   "q3b_stale_intermediates"  CR intermediates use I_vo/asym_t2 of the last iteration's input (src/ccsd.f90:2377)
 *   "triples_ijk_symmetry"     (T) over unique i<=j<=k with multiplicities (1) or all o^3 ordered triples (0)
 *   "triples_batch_bytes"      work-buffer budget of the (T) batches, bytes
 * Measurement switches (default 0):
 *   "finalize_keep_ccsd"       afesp_gpu_ccsd_finalize keeps the DIIS history and intermediates (benchmark loops)
 *   "gemm_timing"              bracket every DMMA GEMM launch with CUDA events (see afesp_gpu_gemm_time)
 * Kernel selection:
 *   "gemm_use_tma"             0 = cp.async kernels only; 1 = the TMA-staged kernel for the gathered (T) batches only;
 *                              2 (default) = also for every other aligned GEMM the 64x64 tile is chosen for.  With a
 *                              value > 0 a consistency check against the cp.async kernel runs once per process
 *                              (at afesp_gpu_open / when switched on); if it fails the path is off (afesp_gpu_tma_status)
 *   "gemm_force_config"        tile menu entry (tuning aid), -1 = automatic
 *   "gemm_tma_edge"            1 (default): the TMA kernel multiplies only ceil(M/8) row fragments (ragged last m-tile shared
 *                              evenly by the warps) and two instead of four DMMA groups for a K tail of <= 8; 0: pad (A/B tests)
 *   "spinorb_symmetry_tol"     abort threshold of the spin-orbital symmetry self-check (default 1e-12, see ccsd_init_info)
 * Model:
 *   "frozen_core"              number k of frozen doubly occupied spatial orbitals (default 0): MP2, CCSD and the triples
 *                              correlate orbitals k..nbasis-1 only -- the same calculation as on the active-orbital
 *                              integrals (orbitals k.., eps[k:], nocc-k occupied), since the canonical RHF Fock operator is
 *                              diagonal.  Read by afesp_gpu_mp2_energy and afesp_gpu_ccsd_init when they are called;
 *                              ccsd_init keeps it with the CC state, so finalize, the CR intermediates and the triples of
 *                              that state use it whatever the option says later.  A negative or non-integer value is
 *                              refused here (status 1); k >= nocc is refused by mp2_energy / ccsd_init (status 1).  With a
 *                              communicator attached every rank sets the same value.
 *   "dist_ccsd", "dist_min_flops"   see the multi-GPU section below */
int afesp_gpu_set_option(afesp_handle h, const char* key, double value);
/* State of the TMA-staged GEMM path: *scope = value of "gemm_use_tma" in force; *selftest = 1 when the start-up
 * consistency check against the cp.async kernel passed on this device, -1 when it failed (the TMA path is then off for
 * the process and cannot be switched on), 0 when it has not run (TMA never requested). */
int afesp_gpu_tma_status(afesp_handle h, int* scope, int* selftest);
/* Kernel launches and executed DMMA flop (2*M*N*K per GEMM) since the handle was opened. */
int afesp_gpu_counters(afesp_handle h, long long* launches, double* gemm_flops);

/* AO->MO transform + MP2: replaces the body of do_mp2_spatial (src/mp2.f90:261-449) ---------------------------- */
/* eri_ao[npacked], coeff(n,n) = C(mo,ao) (sys%canon_coeff, src/hf.f90:102,127) -> eri_mo[npacked] (host, optional).
 * Passing eri_ao == NULL and coeff == NULL repeats the transform on the copies already resident on the device. */
int afesp_gpu_ao2mo(afesp_handle h, int nbasis, const double* eri_ao, const double* coeff, double* eri_mo);
/* Synthetic workload input (SURVEY.md §8d-ii / §8f-3): build the packed AO integrals on the device from a low-rank
 * factor, eri[(ij|kl)] = sum_P B(ij,P) B(kl,P), B = factors(npair, naux) column-major in pair order, and upload
 * coeff(n,n); afterwards afesp_gpu_ao2mo(h, n, NULL, NULL, ...) transforms the resident copy.  (A text eri.dat at
 * nbf=400 would be ~3e9 lines.) */
int afesp_gpu_synth_eri_ao(afesp_handle h, int nbasis, int naux, const double* factors, const double* coeff);
/* Copy the device-resident packed MO integrals to the host (npacked doubles). */
int afesp_gpu_get_eri_mo(afesp_handle h, double* eri_mo);
/* Free device memory the next stage does not need: what = "eri_ao" | "eri_mo" | "scratch". */
int afesp_gpu_release(afesp_handle h, const char* what);
/* Load packed MO integrals directly (a host that already holds int_store%eri_mo).  With a communicator attached the
 * call is collective.  If EVERY rank passes the array (replicated host copies, or one copy per node in shared memory)
 * each rank uploads 1/nranks of it over its own PCIe link and the shares are exchanged over NVLink; if only some do,
 * rank 0 must be one of them: it uploads the whole array and the other ranks (which may pass NULL) receive it over NVLink. */
int afesp_gpu_set_eri_mo(afesp_handle h, int nbasis, const double* eri_mo);
/* MP2 correlation energy from the device-resident MO integrals (src/mp2.f90:418-438); eps = sys%canon_levels(n). */
int afesp_gpu_mp2_energy(afesp_handle h, int nocc, const double* eps, double* e_mp2);

/* CCSD: replaces do_ccsd_spatial (src/ccsd.f90:279-402) / do_ccsd_spinorb (src/ccsd.f90:71-277) ----------------- */
/* init_cc + init_diis_cc_t + the first update_cc_energy: returns the "MP1" line (energy, sum dT2^2).
 * nocc = number of doubly occupied spatial orbitals (sys%nel/2) in both formulations, frozen core included.  diis_n_errmat = sys%ccsd_diis_n_errmat,
 * 0..64 (< 2 switches DIIS off as src/ccsd.f90:593-595 does; the history costs 2 x diis_n_errmat amplitude-sized arrays). */
int afesp_gpu_ccsd_init(afesp_handle h, int nocc, int restricted, const double* eps, int diis_n_errmat,
                        double* e_mp1, double* rmst2);
/* Spin-orbital integral preparation inside afesp_gpu_ccsd_init (restricted == 0), src/ccsd.f90:106-202: the nine
 * slices of <pq||rs> are gathered from the packed MO integrals, then the reference's permutational-symmetry self-check
 * (:150-167) runs on the device over the same index set.  If its error exceeds depsilon = 1e-12 (src/const.F90:19;
 * option "spinorb_symmetry_tol") afesp_gpu_ccsd_init returns status 5 with the reference's message
 * "Permutational symmetry of antisymmetrised integrals does not hold" (the host prints the
 * 'Permutational symmetry error:' line from info[0] and stops through error('ccsd::do_ccsd', ...), :161-164).
 * info[0] = the accumulated error, info[1] = device seconds of the slice gather, info[2] = device seconds of the
 * check, info[3] = 0 (reserved).  Valid after afesp_gpu_ccsd_init returned 0 or 5. */
int afesp_gpu_ccsd_init_info(afesp_handle h, double info[4]);
/* One pass of the iteration body up to and including update_cc_energy (src/ccsd.f90:340-359 / 230-246):
 * stash amplitudes for DIIS, intermediates, amplitude equations, energy.  rmst2 is the squared norm the reference
 * prints (src/ccsd.f90:1806); the host applies the convergence test of :1805. */
int afesp_gpu_ccsd_iterate(afesp_handle h, double* e_cc, double* rmst2);
/* update_diis_cc (src/ccsd.f90:617-676): extrapolate the amplitudes in place. */
int afesp_gpu_ccsd_diis(afesp_handle h);
/* After convergence (src/ccsd.f90:366-393 / 252-269): T1 diagnostic (spin-free: sqrt(sum t1^2)/sqrt(nel), nel = 2(nocc-k)
 * correlated electrons with k = "frozen_core"), the CR intermediates when want_cr != 0, optional copies of t1(o,v) and
 * t2(o,o,v,v) over the active orbitals: o = nocc-k, v = nbasis-nocc (spin-free) or o = 2(nocc-k), v = 2(nbasis-nocc)
 * (spin-orbital).  Amplitudes and the integral slices (T) needs stay on the device (the int_store_cc hand-over of the
 * reference). */
int afesp_gpu_ccsd_finalize(afesp_handle h, int want_cr, double* t1_diagnostic, double* t1, double* t2);

/* Triples: replaces do_ccsd_t_spatial (src/ccsd.f90:2018-2293) / do_ccsd_t_spinorb (src/ccsd.f90:1812-1922) ------ */
/* sums[6] = e_T, e_TT, D_T, D_TT, e_CR, e_CRT as accumulated by the (i,j,k) loop (src/ccsd.f90:2218-2233), summed
 * over all ranks of the communicator when one is attached; denominator_constant = 1 + 2 sum t1^2 + sum asym_t2*c
 * (src/ccsd.f90:2243).  The host assembles the printed energies exactly as src/ccsd.f90:2239-2276. */
int afesp_gpu_ccsd_t_spatial(afesp_handle h, int paren, int renorm, int comp_renorm, double sums[6],
                             double* denominator_constant);
/* e_T of src/ccsd.f90:1910 (host adds sys%e_ccsd). */
int afesp_gpu_ccsd_t_spinorb(afesp_handle h, double* e_T);

/* Multi-GPU: one process (or handle) per device.  (T) triples are dealt round-robin over ranks and the six sums are
 * combined with one ncclAllReduce.  With a communicator attached the CCSD state stays replicated but the heavy GEMMs
 * (ladder, rings, AO->MO half transforms) are sharded over output columns -- each rank keeps only its column slab of
 * the (+/-)-symmetrised <ef|ab> ladder integrals -- and the computed slabs are exchanged over NVLink (grouped
 * ncclBroadcast; ncclSend/ncclRecv all-to-all between the two AO->MO half transforms).  Every call that touches the
 * communicator (ao2mo, ccsd_init, ccsd_iterate, ccsd_finalize, ccsd_t_*) is collective: all ranks make it with the
 * same arguments.  Options: "dist_ccsd" (1/0, default 1), "dist_min_flops" (GEMMs below stay replicated),
 * "dist_allgather" (-1 default: one in-place ncclAllGather of padded equal slabs from 8 ranks on, grouped broadcasts
 * below; 0 / 1 force) and "dist_overlap_chunks" (default 1: serial compute / exchange).
 * The 128-byte id comes from rank 0 and is broadcast by the host (MPI, torchrun...). */
int afesp_gpu_comm_unique_id(char id[128]);
int afesp_gpu_comm_init(afesp_handle h, int rank, int nranks, const char id[128]);
/* Page-lock (and release) a host array the caller owns, e.g. int_store%eri_mo or a shared-memory mapping of it, so that
 * the H2D / D2H copies of afesp_gpu_set_eri_mo / afesp_gpu_ccsd_finalize run at full PCIe speed.  Status 2 = the driver
 * refused (the array then simply stays pageable); no handle needed, the calling thread's current device is used. */
int afesp_gpu_host_register(void* ptr, long long bytes);
int afesp_gpu_host_unregister(void* ptr);
/* Without NCCL: give the handle a (rank, nranks) share only; the caller sums the partial results itself. */
int afesp_gpu_set_partition(afesp_handle h, int rank, int nranks);
/* Host-only: number of (i,j,k) work units per rank (no device needed). */
int afesp_gpu_triples_partition(int nocc_active, int symmetric, int strict, int nranks, long long* counts);
/* Host-only: contiguous column range [lo[r], hi[r]) of `ncols` columns owned by rank r (multiples of `granularity`),
 * the split used by the sharded GEMMs (granularity 64) and the AO->MO pair blocks (granularity 16). */
int afesp_gpu_column_partition(long long ncols, int nranks, int granularity, long long* lo, long long* hi);

/* Operators of src/linalg.fpp on host arrays (used by the parity tests; the CC drivers call the same kernels) ---- */
/* dgemm_wrapper (src/linalg.fpp:58-89): C(MxN) = alpha*op(A)(MxK)*op(B)(KxN) + beta*C, leading dimensions inferred
 * exactly as the reference does (LDA = K if transA=='T' else M; LDB = N if transB=='T' else K; LDC = M). */
int afesp_gpu_dgemm_wrapper(afesp_handle h, char transA, char transB, int outer_row, int outer_col, int inner_dim,
                            const double* A, const double* B, double* C, double alpha, double beta);
/* omp_reshape (src/linalg.fpp:99-156): out(perm(i,j,k,l)) = beta*out + in(i,j,k,l); arr_order e.g. "2341" means
 * out(j,k,l,i) = in(i,j,k,l).  has_beta == 0 reproduces the absent optional argument (out is overwritten). */
int afesp_gpu_omp_reshape(afesp_handle h, double* out_arr, const double* in_arr, const int in_dims[4],
                          const char arr_order[4], int has_beta, double beta);
/* Synthetic-workload helper (bench): time `reps` back-to-back device-resident dgemms, returns milliseconds/gemm. */
int afesp_gpu_bench_dgemm(afesp_handle h, char transA, char transB, int M, int N, int K, double beta, int reps,
                          double* ms);
/* HBM-bound kernels of the path timed device-resident at the shape of an (o,o,v,v) amplitude array:
 * what = "permute:<order>" (omp_reshape order, e.g. "permute:3412"; 16 B/element), "permute_acc:<order>" (24 B),
 * "divide" (T2 = X / D_ijab, 16 B), "energy" (E_CC + sum dT2^2 in one pass, 24 B), "axpby" (24 B).
 * Returns milliseconds per launch and the algorithmic bytes per launch (SURVEY.md section 8d). */
int afesp_gpu_bench_hbm(afesp_handle h, const char* what, int nocc, int nvirt, int reps, double* ms, double* bytes);
/* Soak aid: the TMA-staged GEMM kernel against the cp.async kernel on one (optionally strided-batched) problem with
 * pseudo-random operands -- the cp.async result once, the TMA kernel `reps` times, each compared on the device.
 * Returns the number of differing elements (tolerance 1e-12 on O(1e-2) data) and the mean milliseconds per launch. */
int afesp_gpu_gemm_crosscheck(afesp_handle h, char transA, char transB, int M, int N, int K, int nbatch, double beta,
                              int reps, long long* mismatches, double* ms_tma, double* ms_cpasync);
/* Raw DMMA issue-rate probe: register-resident mma.sync loop on all SMs; returns TFLOP/s (the FP64 tensor peak the
 * roofline fractions are quoted against; MEASURED_PEAKS.json has no FP64 entry). */
int afesp_gpu_dmma_peak(afesp_handle h, double* tflops);
/* Device time (CUDA events on the engine's stream) of the last stage call on this handle, milliseconds. */
int afesp_gpu_last_stage_ms(afesp_handle h, double* ms);
/* Stopwatch on the engine's stream: stop == 0 records the start event; stop != 0 records the end event, waits for it
 * and returns the device milliseconds between the two (spans any number of stage calls, idle gaps included). */
int afesp_gpu_timer(afesp_handle h, int stop, double* ms);
/* With option "gemm_timing" on: accumulated device milliseconds and executed flop of all DMMA GEMM launches since the
 * option was switched on or since the previous call (synchronises the stream). */
int afesp_gpu_gemm_time(afesp_handle h, double* ms, double* flops);
/* Same, plus the number of GEMM launches bracketed (per-launch averages for the roofline line of bench.py). */
int afesp_gpu_gemm_stats(afesp_handle h, double* ms, double* flops, long long* launches);

#ifdef __cplusplus
}
#endif
#endif /* AFESP_GPU_H */
