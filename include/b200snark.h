/* libb200snark — C ABI of the B200-native Groth16 / Pinocchio prove path.
 *
 * The reference (arnaucube/go-snark-study) has no FFI: its boundary is the
 * exported Go package API.  Each entry point below names the Go function(s)
 * whose body a cgo shim replaces (file:line in the upstream tree); the shim
 * itself is shown in INTEGRATION.md.  Conventions:
 *
 *   - field elements / scalars: 4 little-endian uint64 limbs, STANDARD form
 *     (not Montgomery), canonical (< modulus) — i.e. big.Int.Bits() on amd64,
 *     zero-padded.  Scalars must be reduced mod r (the shim sends |e| mod r:
 *     the reference's MulScalar consumes |e|, fields/fq.go:138-140, SURVEY H7).
 *   - G1 point  = [3]*big.Int  Jacobian (X, Y, Z)            -> 12 uint64
 *     G2 point  = [3][2]*big.Int Jacobian (X.c0, X.c1, Y.., Z..) -> 24 uint64
 *     Z == 0 (e.g. the (0,0,0) entries of Pk.BACDelta, groth16.go:177-180) is
 *     the point at infinity.  Outputs are normalised: (x, y, 1), infinity as
 *     all-zero — valid inputs to every reference function (SURVEY H1).
 *   - every function returns 0 (B200_OK) or a negative B200_E* code; no
 *     exceptions or panics cross the ABI; b200_last_error() gives the text.
 *   - all pointers are HOST pointers unless the name ends in _device.
 *   - thread-safety: calls are serialised per process by an internal mutex
 *     (cgo may migrate goroutines between OS threads).
 *   - there is NO CPU fallback: without a CUDA device every call fails with
 *     B200_ENODEVICE.
 */
#ifndef B200SNARK_H
#define B200SNARK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK 0
#define B200_ENODEVICE (-1) /* no CUDA device / init failed                         */
#define B200_ECUDA (-2)     /* CUDA runtime error (see b200_last_error)              */
#define B200_EINVAL (-3)    /* bad argument (null pointer, size mismatch, handle)    */
#define B200_ERANGE (-4)    /* a field element >= modulus or a scalar >= r           */
#define B200_EDIVZERO (-5)  /* polynomial division by a zero leading coefficient     */
#define B200_ENOMEM (-6)
#define B200_ECOMM (-7)     /* NCCL: library not found, or a collective failed       */

typedef uint64_t b200_bases_t; /* device-resident, window-precomputed base-point set */
typedef uint64_t b200_pk_t;    /* device-resident proving key                        */
typedef uint64_t b200_r1cs_t;  /* device-resident sparse R1CS (CSR + CSC)            */

/* ---- context ------------------------------------------------------------ */
int b200_init(int device);        /* idempotent; selects the CUDA device of this process */
int b200_shutdown(void);
const char* b200_last_error(void);
int b200_version(void);
/* Process-wide options for objects created AFTERWARDS.  B200_CFG_ACC_MODE: bucket-accumulation kernel of base sets and
 * proving keys — 0 auto (batched affine where bucket population and shard size amortise its rounds, else XYZZ mixed
 * adds), 1 batched affine, 2 XYZZ.  Same results either way; the parity tests run every MSM size under both.          */
#define B200_CFG_ACC_MODE 1
/* B200_CFG_TMA_STAGING: the batched-affine backward pass with its operands staged into shared memory — TMA bulk
 * copies (cp.async.bulk + per-warp mbarrier) in the contiguous rounds, cp.async gathers in round 1.  0 (default) the
 * register-load kernel: measured FASTER (18.92 vs 20.17 ms per 2^20 proof, profiles/r2_notes.md: the kernel is bound by
 * the multiply pipe, not by the fetch); 1 staged in every round, 2 staged in rounds >= 2 only.  Same results.          */
#define B200_CFG_TMA_STAGING 2
/* B200_CFG_PK_CONTEXT: prove context (0 or 1) of proving keys loaded AFTERWARDS.  The two contexts own separate side
 * streams and polynomial workspaces, so a device-resident proof on a context-1 key (b200_groth16_prove_device on the
 * caller's second stream) may be in flight beside one on a context-0 key: a prover that keeps two proofs in flight hides
 * the latency-bound sort / bucket-tail / blinding-product chains of one behind the accumulation of the other (bench.py
 * `proofs_in_flight`; the keys are independent objects, each with its own tables and scratch).                       */
#define B200_CFG_PK_CONTEXT 4
/* B200_CFG_PAIRING_KERNEL: b200_pairing_batch with one THREAD per pairing (1: the step-by-step restatement of
 * bn128.go:179-421, ~10 ms of dependent multiplications per pairing) or one WARP per pairing (2: F_q^12 in shared
 * memory, 27 F_q^2 products of a tower multiplication on 27 lanes; csrc/pairing_warp.cuh: 3.4 ms); 0 = auto: a warp per
 * pairing up to 2048 pairings per call (latency), a thread per pairing above (462 k vs 204 k pairings/s at 2^16).
 * Bit-identical F_q^12 values.  b200_groth16_verify always runs four warps (4.2 ms per verification, was 20).          */
#define B200_CFG_PAIRING_KERNEL 5
/* Partition tuning of SHARDED proving keys loaded afterwards (defaults = the measured best for one proof at a time,
 * profiles/r2_notes.md section 8): cost weight x100 of an A / B1 term (10) and of a G2 term (11) in C||PTD terms, and the
 * smallest per-rank set that still takes the batched-affine tree, in G1 (12) / G2 (13) terms — below it the set runs
 * the XYZZ kernel, whose single launch has the shorter latency chain.  With two proofs in flight (B200_CFG_PK_CONTEXT)
 * that latency is hidden and the affine tree's 6 multiplications per add win at every shard size: set 12 and 13 to 1. */
#define B200_CFG_SHARD_W_AB 10
#define B200_CFG_SHARD_W_G2 11
#define B200_CFG_SHARD_AFFINE_MIN_G1 12
#define B200_CFG_SHARD_AFFINE_MIN_G2 13
int b200_config(int key, int value);

/* ---- base-point sets (the CRS arrays of groth16.Pk / snark.Pk) ---------- */
/* Upload n Jacobian points, normalise to affine Montgomery form on the device
 * and precompute 2^(c*w) * P for every window w (the CRS is static, so all
 * windows of one MSM share a single bucket set; see DESIGN.md §3).
 * window_bits = 0 picks c from n.  Replaces nothing in the reference (its Pk
 * is consumed directly); this is the "load proving key once" step of H9.     */
int b200_g1_bases_load(const uint64_t* points_jac, size_t n, int window_bits, b200_bases_t* out);
int b200_g2_bases_load(const uint64_t* points_jac, size_t n, int window_bits, b200_bases_t* out);
int b200_bases_free(b200_bases_t h);
int b200_bases_info(b200_bases_t h, size_t* n, int* group, int* window_bits, int* n_windows);
/* which bucket-accumulation kernel the set was built for: 1 batched affine, 2 XYZZ (see b200_config) */
int b200_bases_acc_mode(b200_bases_t h, int* mode);

/* ---- multi-scalar multiplication ---------------------------------------- */
/* out = sum_i scalars[i] * P_i over the first n bases of the set.
 * Replaces the hot loops  acc = G1.Add(acc, G1.MulScalar(P_i, w_i))  of
 * groth16/groth16.go:243-250,269-271 and snark.go:265-286 (G1: bn128/g1.go:32-155;
 * G2: bn128/g2.go:32-181).                                                    */
int b200_g1_msm(b200_bases_t h, const uint64_t* scalars, size_t n, uint64_t out_jac[12]);
int b200_g2_msm(b200_bases_t h, const uint64_t* scalars, size_t n, uint64_t out_jac[24]);

/* Same, scalars already resident in device memory (n * 32 bytes, standard form,
 * or Montgomery form when scalars_mont != 0), result left on the device as an
 * XYZZ record (4 field elements, Montgomery form; 128 B for G1, 256 B for G2)
 * on `stream` (a cudaStream_t, may be NULL).  No host synchronisation.  Used by
 * the prove pipeline, by bench.py's device-resident timing and by the
 * multi-GPU path (each rank's partial record is what the NCCL gather moves).  */
int b200_msm_device(b200_bases_t h, const void* d_scalars, size_t n, int scalars_mont,
                    void* d_out_xyzz, void* stream);
/* Sum `count` XYZZ partial records (device memory, e.g. the gathered per-rank
 * partials) and normalise: out_jac = (x, y, 1) in standard form on the host.  */
int b200_g1_sum_partials(const void* d_xyzz, size_t count, uint64_t out_jac[12], void* stream);
int b200_g2_sum_partials(const void* d_xyzz, size_t count, uint64_t out_jac[24], void* stream);

/* ---- batch scalar multiplication, reference operation order -------------- */
/* out[i] = MulScalar(points[i], scalars[i]) with the reference's MSB-first
 * double-and-add and its add-2007-bl / dbl-2009-l formulas, one thread per
 * term: X,Y,Z-exact drop-in for bn128.G1.MulScalar (bn128/g1.go:140-155) and
 * bn128.G2.MulScalar (bn128/g2.go:142-181).  Also mints CRSs on the GPU
 * (groth16/groth16.go:139-219: every Pk/Vk entry is G.MulScalar(g, k)).       */
int b200_g1_mul_batch(const uint64_t* points_jac, const uint64_t* scalars, size_t n, uint64_t* out_jac);
int b200_g2_mul_batch(const uint64_t* points_jac, const uint64_t* scalars, size_t n, uint64_t* out_jac);
/* points_jac may hold a single point broadcast to all scalars when n_points == 1 */
int b200_g1_mul_batch_bcast(const uint64_t* point_jac, const uint64_t* scalars, size_t n, uint64_t* out_jac);
int b200_g2_mul_batch_bcast(const uint64_t* point_jac, const uint64_t* scalars, size_t n, uint64_t* out_jac);

/* ---- proving keys and the prove path -------------------------------------- */
/* Upload a Groth16 proving key (groth16.Pk, groth16/groth16.go:15-32) once:
 *   at        = Pk.G1.At[0..m)            b1 = Pk.G1.BACGamma[0..m)   (G1, 12 u64 each)
 *   b2        = Pk.G2.BACGamma[0..m)      (G2, 24 u64 each)
 *   bacdelta  = Pk.BACDelta[0..m)         (entries 0..npublic are ignored, as in groth16.go:248)
 *   ptd       = Pk.PowersTauDelta[0..n_ptd)
 *   z         = Pk.Z[0..nz) coefficients  alpha1/beta1/delta1 = Pk.G1.{Alpha,Beta,Delta}
 *   beta2/delta2 = Pk.G2.{Beta,Delta}     npublic = circuit.NPublic, m = circuit.NVars
 * The blinding points are appended to the MSM base sets so that
 * A = sum w_i At_i + alpha + r*delta etc. are single MSMs (DESIGN.md §4).          */
int b200_groth16_pk_load(const uint64_t* at, const uint64_t* b1, const uint64_t* b2, const uint64_t* bacdelta,
                         size_t m, const uint64_t* ptd, size_t n_ptd, const uint64_t* z, size_t nz,
                         const uint64_t alpha1[12], const uint64_t beta1[12], const uint64_t delta1[12],
                         const uint64_t beta2[24], const uint64_t delta2[24], size_t npublic, int window_bits,
                         b200_pk_t* out);
/* groth16.GenerateProofs (groth16/groth16.go:225-278) with the randomness r, s
 * supplied by the caller (the Go shim draws them with Fq.Rand, fields/fq.go:116-132,
 * exactly as the reference does at groth16.go:231-238).  w: nw = NVars witness
 * scalars (|w_i| mod r); px: npx coefficients.  Outputs are Jacobian points (Z != 1
 * in general, like the reference's own), standard form.  Like DivisorPolynomial
 * (r1csqap.go:213-216: quotient kept, remainder dropped) the proof depends only on the
 * top npx - len(Z) + 1 coefficients of px; only those are read from the host buffer. */
int b200_groth16_prove(b200_pk_t pk, const uint64_t* w, size_t nw, const uint64_t* px, size_t npx,
                       const uint64_t r[4], const uint64_t s[4], uint64_t pi_a[12], uint64_t pi_b[24],
                       uint64_t pi_c[12]);
/* Same with the witness and px already resident in DEVICE memory (standard form)
 * and the 48-u64 result (PiA | PiC | PiB) left in device memory on `stream`; no
 * host synchronisation.  This is the region bench.py times as `value`.            */
int b200_groth16_prove_device(b200_pk_t pk, const void* d_w, size_t nw, const void* d_px, size_t npx,
                              const uint64_t r[4], const uint64_t s[4], void* d_out, void* stream);
/* Multi-GPU (one process per GPU): rank `rank` of `world` keeps the contiguous
 * index slice [m*rank/world, m*(rank+1)/world) of every CRS array (and the same
 * fraction of PowersTauDelta); the blinding points ride on rank 0.  With such a key
 * b200_groth16_prove_device leaves a 1024-byte PARTIAL record (XYZZ sums A | B1 |
 * B2 | CH) in d_out instead of a proof WHEN NO COMMUNICATOR IS ACTIVE (b200_comm_init):
 * the caller then all-gathers the records of all ranks itself and calls
 * b200_groth16_finalize_device, which adds them and applies groth16.go:272-275 (this is
 * how the one-GPU tests emulate N ranks).  With a communicator the gather + finalize run
 * inside the call and d_out receives the proof.  No EC-point reduction exists in NCCL,
 * hence gather-then-add (SURVEY §5).                                               */
int b200_groth16_pk_load_shard(const uint64_t* at, const uint64_t* b1, const uint64_t* b2, const uint64_t* bacdelta,
                               size_t m, const uint64_t* ptd, size_t n_ptd, const uint64_t* z, size_t nz,
                               const uint64_t alpha1[12], const uint64_t beta1[12], const uint64_t delta1[12],
                               const uint64_t beta2[24], const uint64_t delta2[24], size_t npublic, int window_bits,
                               int rank, int world, b200_pk_t* out);
/* ---- multi-GPU inside the library (one process per GPU) -------------------------------------------------
 * b200_comm_unique_id (on one rank) mints an NCCL id; the caller distributes the 128 bytes by whatever means it has
 * (a file, a socket, MPI, torch.distributed) and every rank calls b200_comm_init(id, rank, world) after b200_init.
 * With a communicator, b200_groth16_prove / b200_groth16_prove_device on a key loaded with
 * b200_groth16_pk_load_shard(.., rank, world) return the FINAL proof on every rank: each rank computes its partial
 * sums, the 1 KB records are all-gathered over NVLink (ncclAllGather on the library's stream) and added.  All ranks
 * must make the same call with the same witness, px, r and s (SPMD), as N copies of a Go process calling
 * groth16.GenerateProofs (groth16/groth16.go:225) would.  libnccl.so.2 is dlopen'ed; absent -> B200_ECOMM.           */
int b200_comm_unique_id(uint8_t out[128]);
int b200_comm_init(const uint8_t id[128], int rank, int world);
int b200_comm_destroy(void);
/* What a sharded key reads: out = { A lo, hi, B1 lo, hi, B2 lo, hi (witness index ranges), C-part witness
 * range lo, hi, needs_px (0/1), rank, world, NVars }.  A caller that stages inputs per proof only has to upload
 * those witness ranges, and px only when needs_px is set.                                                        */
int b200_groth16_shard_info(b200_pk_t pk, uint64_t out[12]);
int b200_groth16_finalize_device(b200_pk_t pk, const void* d_parts, int nparts, const uint64_t r[4],
                                 const uint64_t s[4], void* d_out, void* stream);
/* Pinocchio proving key (snark.Pk, snark.go:16-26): A, Ap, Bp, C, Cp, Kp in G1 and
 * B in G2, each m points; G1T n_g1t points; Z.                                     */
int b200_pinocchio_pk_load(const uint64_t* a, const uint64_t* ap, const uint64_t* b2, const uint64_t* bp,
                           const uint64_t* c, const uint64_t* cp, const uint64_t* kp, size_t m,
                           const uint64_t* g1t, size_t n_g1t, const uint64_t* z, size_t nz, size_t npublic,
                           int window_bits, b200_pk_t* out);
/* snark.GenerateProofs (snark.go:254-289).  out_g1 = 7 Jacobian G1 points in the
 * order PiA, PiAp, PiBp, PiC, PiCp, PiH, PiKp (84 u64); pi_b = PiB (G2).           */
int b200_pinocchio_prove(b200_pk_t pk, const uint64_t* w, size_t nw, const uint64_t* px, size_t npx,
                         uint64_t* out_g1, uint64_t pi_b[24]);
/* Multi-GPU Pinocchio: the eight MSMs of snark.GenerateProofs are independent, so rank `rank` of `world` keeps WHOLE MSMs
 * (dealt greedily by cost, identically on every rank; no MSM is split).  With a communicator (b200_comm_init)
 * b200_pinocchio_prove on such a key computes the rank's MSMs, all-gathers the 2 KB result records and returns the whole
 * proof on every rank.  Without one, b200_pinocchio_prove_record_device leaves the rank's record (8 XYZZ slots, 256 B
 * each, device memory) to the caller and b200_pinocchio_finalize_records sums `world` gathered records — how the
 * one-GPU tests emulate N ranks.                                                                                      */
int b200_pinocchio_pk_load_shard(const uint64_t* a, const uint64_t* ap, const uint64_t* b2, const uint64_t* bp,
                                 const uint64_t* c, const uint64_t* cp, const uint64_t* kp, size_t m,
                                 const uint64_t* g1t, size_t n_g1t, const uint64_t* z, size_t nz, size_t npublic,
                                 int window_bits, int rank, int world, b200_pk_t* out);
int b200_pinocchio_prove_record_device(b200_pk_t pk, const uint64_t* w, size_t nw, const uint64_t* px, size_t npx,
                                       void* d_record);
int b200_pinocchio_finalize_records(const void* d_records, int world, uint64_t* out_g1, uint64_t pi_b[24]);
int b200_pk_free(b200_pk_t pk);

/* ---- instrumentation (bench.py) -------------------------------------------- */
/* b200_profile(flags): bit 0 brackets every bucket-accumulation phase (the dominant
 * kernels) with CUDA events on its stream; bit 1 additionally issues all MSMs of a
 * proof on the caller's stream instead of overlapping them on side streams, so that
 * those event times are exclusive (measurement mode, slower).  b200_profile_read synchronises and returns
 * out = { G1 ms total, G1 launches, G1 terms total, G2 ms total, G2 launches,
 *         G2 terms total, kernel launches since the last read, 0 } and resets.      */
int b200_profile(int enable);
int b200_profile_read(double out[8]);

/* ---- polynomials over F_r (coefficient arrays, index = power of x) -------- */
/* out[0..na+nb-1) = a * b.   Replaces PolynomialField.Mul (r1csqap/r1csqap.go:57-67). */
int b200_poly_mul(const uint64_t* a, size_t na, const uint64_t* b, size_t nb, uint64_t* out);
/* q[0..na-nb+1) = a div b, rem[0..nb-1) = a mod b (rem may be NULL).
 * Replaces PolynomialField.Div / DivisorPolynomial (r1csqap/r1csqap.go:70-84,213-216).
 * b[nb-1] must be non-zero (B200_EDIVZERO; the reference panics on ModInverse(0)).
 * na < nb: quotient is empty and rem = a (na coefficients), as in the reference. */
int b200_poly_div(const uint64_t* a, size_t na, const uint64_t* b, size_t nb, uint64_t* q, uint64_t* rem);

int b200_poly_add(const uint64_t* a, size_t na, const uint64_t* b, size_t nb, uint64_t* out); /* r1csqap.go:94-103, max(na,nb) out */
int b200_poly_sub(const uint64_t* a, size_t na, const uint64_t* b, size_t nb, uint64_t* out); /* r1csqap.go:106-115 */
int b200_poly_eval(const uint64_t* v, size_t n, const uint64_t x[4], uint64_t out[4]);        /* r1csqap.go:118-126 */

/* out[i] = Eval(polys[i], x) for m polynomials of n coefficients each (row-major): the At/Bt/Ct loops of
 * GenerateTrustedSetup (groth16/groth16.go:164-205, snark.go:181-218).                                        */
int b200_poly_eval_batch(const uint64_t* polys, size_t m, size_t n, const uint64_t x[4], uint64_t* out);
/* out[0..n] = coefficients of prod_{i=1}^{n} (x - i): the "z pol" of groth16.go:122-132 / snark.go:221-232; n <= 2^26. */
int b200_zero_poly(size_t n, uint64_t* out);

/* ---- verifier side (SURVEY §8f row 2) ------------------------------------------------------------------ */
/* out[i] = Bn128.Pairing(g1[i], g2[i]) (bn128/bn128.go:179-186): optimal-ate Miller loop + the reference's plain
 * final exponentiation, one GPU thread per pairing; 48 uint64 per result in the reference's [2][3][2]*big.Int order.
 * Bit-identical to the reference (golden: externalVerif/circom-test/verification_key.json vk_alfabeta_12).
 * A G2 point at infinity returns B200_EINVAL where the reference panics "q1[2] != Fq2.One()" (bn128.go:238-241);
 * a G1 point at infinity is processed like the reference does (Affine -> (0,0)).                                    */
int b200_pairing_batch(const uint64_t* g1_jac, const uint64_t* g2_jac, size_t n, uint64_t* out);
/* out[i] = a[i] * b[i] in F_q^12 (fields/fq12.go:72-84; 48 uint64 per element, same order as b200_pairing_batch):
 * the product step of the verification equations (snark.go:338-341,357; groth16.go:297-301).                      */
int b200_fq12_mul_batch(const uint64_t* a, const uint64_t* b, size_t n, uint64_t* out);
/* groth16.VerifyProof (groth16/groth16.go:281-305): *ok = 1 iff e(A,B) == e(alpha,beta) * (e(icPubl,gamma) * e(C,delta)),
 * icPubl = IC[0] + sum publicSignals[i] * IC[i+1].  The four pairings run concurrently.                              */
int b200_groth16_verify(const uint64_t* ic, size_t n_ic, const uint64_t alpha1[12], const uint64_t beta2[24],
                        const uint64_t gamma2[24], const uint64_t delta2[24], const uint64_t pi_a[12],
                        const uint64_t pi_b[24], const uint64_t pi_c[12], const uint64_t* public_signals, size_t n_public,
                        int* ok);
/* Verify nproofs Groth16 proofs under ONE verification key (groth16.VerifyProof, groth16/groth16.go:281-305, per proof).
 * pi_a: nproofs x 12 u64, pi_b: nproofs x 24, pi_c: nproofs x 12, public_signals: nproofs x n_public x 4 (row-major),
 * rho: nproofs x 2 u64 — the caller's secret, uniformly random, non-zero 128-bit batching scalars (like r, s of the prove
 * calls, drawn by the caller; a prover who knows them can make invalid proofs cancel).  ok[i] = 1 / 0, or the negative
 * code b200_groth16_verify would return for proof i alone.  stats (may be NULL) = { proofs in the aggregated check,
 * proofs verified one by one, aggregated checks run, Miller loops run }.
 * The proofs that pair bilinearly are checked together: prod e(rho_i A_i, B_i) * e(-(sum rho_i) alpha, beta) *
 * e(-sum rho_i icPubl_i, gamma) * e(-sum rho_i C_i, delta) == 1, N + 3 Miller loops and one final exponentiation (a false
 * accept has probability <= 2^-128 over rho).  A, C or icPubl at infinity, A or C off the curve, B off the twist or outside
 * G2 are verified one by one, as is every proof of a batch whose aggregated check fails.  Call-level errors, ok[] untouched:
 * null pointers, nproofs == 0, n_ic < n_public + 1, a rho_i == 0 (B200_EINVAL); a verification-key coordinate >= q
 * (B200_ERANGE) or G2 point at infinity (B200_EINVAL); alpha at infinity, a vk point off the curve or outside G2 (EINVAL). */
int b200_groth16_verify_batch(const uint64_t* ic, size_t n_ic, const uint64_t alpha1[12], const uint64_t beta2[24],
                              const uint64_t gamma2[24], const uint64_t delta2[24], size_t nproofs,
                              const uint64_t* pi_a, const uint64_t* pi_b, const uint64_t* pi_c,
                              const uint64_t* public_signals, size_t n_public, const uint64_t* rho,
                              int* ok, uint64_t stats[4]);
/* snark.VerifyProof (snark.go:292-372) for one proof.  vk_g1 = Vkb | G1Kbg (2 x 12 u64), vk_g2 = Vka | Vkc | Vkz | G2Kbg |
 * G2Kg (5 x 24 u64), proof_g1 = PiA, PiAp, PiBp, PiC, PiCp, PiH, PiKp (84 u64: the out_g1 order of b200_pinocchio_prove),
 * pi_b = PiB.  *ok = 1 / 0; *failed_check (may be NULL) = 0, or 1..5 for the first of the reference's five checks that
 * fails.  vkx = IC[0] + sum publicSignals[j] * IC[j+1], VkxA = vkx + PiA and VkxAC = VkxA + PiC use the reference's Add
 * (Add(P, P) is infinity); a G1 point at infinity is paired as (0, 0), as the reference does.  The twelve pairings run
 * concurrently.  Errors: null pointers or n_ic < n_public + 1 (B200_EINVAL); PiB or a vk G2 point at infinity (B200_EINVAL:
 * the reference panics, bn128.go:238-241); otherwise a coordinate >= q or a public signal >= r (B200_ERANGE).  So when a
 * G2 point at infinity and an out-of-range value occur together, B200_EINVAL wins.                                    */
int b200_pinocchio_verify(const uint64_t* ic, size_t n_ic, const uint64_t vk_g1[24], const uint64_t vk_g2[120],
                          const uint64_t proof_g1[84], const uint64_t pi_b[24], const uint64_t* public_signals,
                          size_t n_public, int* ok, int* failed_check);
/* Verify nproofs Pinocchio proofs under ONE verification key (b200_pinocchio_verify per proof).  proofs_g1: nproofs x 84
 * u64, pi_b: nproofs x 24, public_signals: nproofs x n_public x 4, rho: nproofs x 5 x 2 u64 — the caller's secret,
 * uniformly random, non-zero 128-bit batching scalars, one per check of each proof.  ok[i] = 1 / 0, or the negative code
 * b200_pinocchio_verify would return for proof i alone.  stats (may be NULL) = { proofs in the aggregated check, proofs
 * verified one by one, aggregated checks run, Miller loops run (12 per proof verified one by one) }.
 * Check k of proof i is raised to rho_ik and the product of all of them is grouped by G2 point: one Miller loop per PiB_i
 * (G1 side rho2 Vkb + rho4 VkxA_i + rho5 G1Kbg) and six for g2, Vka, Vkc, Vkz, G2Kbg, G2Kg — N + 6 Miller loops and one
 * final exponentiation (a false accept has probability <= 2^-128 over rho).  A G1 point, VkxA or VkxAC at infinity, a G1
 * point off the curve, PiB off the twist or outside G2 are verified one by one, as is every proof of a batch whose
 * aggregated check fails.  Call-level errors, ok[] untouched: null pointers, nproofs == 0 or > 2^26, n_ic < n_public + 1,
 * a rho == 0 (B200_EINVAL); a vk G2 point at infinity (B200_EINVAL) or else a vk coordinate >= q (B200_ERANGE); Vkb or
 * G1Kbg at infinity or off the curve, an IC point off the curve, a vk G2 point off the twist or outside G2 (B200_EINVAL). */
int b200_pinocchio_verify_batch(const uint64_t* ic, size_t n_ic, const uint64_t vk_g1[24], const uint64_t vk_g2[120],
                                size_t nproofs, const uint64_t* proofs_g1, const uint64_t* pi_b,
                                const uint64_t* public_signals, size_t n_public, const uint64_t* rho, int* ok,
                                uint64_t stats[4]);

/* ---- dense QAP API upstream of GenerateProofs (small n; the prove path consumes px) ---- */
/* PolynomialField.R1CSToQAP (r1csqap/r1csqap.go:161-188).  a, b, c: n x m row-major R1CS matrices (coefficients
 * reduced mod r).  alphas/betas/gammas: m x n (row i = coefficients of signal i's polynomial over the domain {1..n});
 * z: m-1 coefficients of prod_{i=1}^{m-2}(x-i).  Exact big-integer Lagrange denominators: identical to the reference
 * for n <= 21, and the mathematically intended result where the reference's native-int factorial overflows
 * (r1csqap.go:130-136, SURVEY E3).  1 <= n <= 8191.                                                                   */
int b200_r1cs_to_qap(const uint64_t* a, const uint64_t* b, const uint64_t* c, size_t n, size_t m, uint64_t* alphas,
                     uint64_t* betas, uint64_t* gammas, uint64_t* z);
/* PolynomialField.CombinePolynomials (r1csqap/r1csqap.go:191-210): ax = sum r_i*ap[i] (likewise bx, cx; n coefficients
 * each, ap/bp/cp m x n row-major) and px = ax*bx - cx (2n-1 coefficients).                                            */
int b200_combine_polynomials(const uint64_t* r, size_t m, const uint64_t* ap, const uint64_t* bp, const uint64_t* cp,
                             size_t n, uint64_t* ax, uint64_t* bx, uint64_t* cx, uint64_t* px);

/* ---- sparse QAP front end (any n): the same mathematics without the dense m x n polynomial matrices -------- */
/* A sparse R1CS, n constraints x m signals, three CSR matrices (rowptr n+1 entries, col/val nnz entries; val = 4-limb
 * coefficients reduced mod r, negative coefficients of circuitcompiler (circuit.go:78) sent as r - |v|).  Stays on
 * the device; also stored transposed for the trusted setup.  Replaces the dense a, b, c [][]*big.Int arguments of
 * PolynomialField.R1CSToQAP (r1csqap/r1csqap.go:161) where m*n coefficients cannot exist (137 GB per matrix at
 * n = 2^16, SURVEY H4).                                                                                              */
int b200_r1cs_load(size_t n, size_t m, const uint32_t* a_rowptr, const uint32_t* a_col, const uint64_t* a_val,
                   const uint32_t* b_rowptr, const uint32_t* b_col, const uint64_t* b_val, const uint32_t* c_rowptr,
                   const uint32_t* c_col, const uint64_t* c_val, b200_r1cs_t* out);
int b200_r1cs_free(b200_r1cs_t h);
/* CombinePolynomials(w, R1CSToQAP(a, b, c)) (r1csqap/r1csqap.go:161-210) fused: ax, bx, cx (n coefficients each, any
 * may be NULL) and px = ax*bx - cx (2n-1 coefficients).  ax is the unique polynomial of degree < n with
 * ax(j+1) = (A w)_j: one sparse mat-vec and one O(n log^2 n) interpolation over {1..n} per matrix.  Field-exact, so
 * equal to the reference's coefficients wherever the reference can run (n <= 21, SURVEY E3).                          */
int b200_qap_px(b200_r1cs_t h, const uint64_t* w, size_t nw, uint64_t* ax, uint64_t* bx, uint64_t* cx, uint64_t* px);
/* at[i] = Eval(alphas[i], tau), bt[i], ct[i] for every signal i < m — the loops of GenerateTrustedSetup
 * (groth16/groth16.go:164-205, snark.go:171-189) — as A^T l(tau) with l the Lagrange basis of {1..n} at tau, and
 * zt = prod_{i=1..nz} (tau - i) (groth16.go:122-136 with nz = len(alphas) - 2).  tau must not be one of 1..n.          */
int b200_qap_eval_at(b200_r1cs_t h, const uint64_t tau[4], size_t nz, uint64_t* at, uint64_t* bt, uint64_t* ct,
                     uint64_t zt[4]);
/* PolynomialField.LagrangeInterpolation over x = 1..n (r1csqap/r1csqap.go:150-158) at any n <= 2^26: n values ->
 * n coefficients.                                                                                                    */
int b200_interpolate(const uint64_t* values, size_t n, uint64_t* coeffs);
/* groth16.GenerateProofs fed from the witness: px is computed on the device from the resident R1CS (b200_qap_px) and
 * never leaves HBM; otherwise identical to b200_groth16_prove (groth16/groth16.go:225-278 after the caller's
 * CombinePolynomials step, cli/main.go:339-349).                                                                     */
int b200_groth16_prove_witness(b200_pk_t pk, b200_r1cs_t r1cs, const uint64_t* w, size_t nw, const uint64_t r[4],
                               const uint64_t s[4], uint64_t pi_a[12], uint64_t pi_b[24], uint64_t pi_c[12]);

/* ---- element-wise group operations, reference formulas (X,Y,Z-exact) ------------------- */
/* bn128.G1.Add / Double / Neg / Affine (bn128/g1.go:32-170) and the G2 twins (bn128/g2.go:32-200), n independent
 * operations per call.  Affine writes (x, y) per point, infinity as (0, 0) like G1.Affine.                            */
int b200_g1_add_batch(const uint64_t* p, const uint64_t* q, size_t n, uint64_t* out);
int b200_g1_double_batch(const uint64_t* p, size_t n, uint64_t* out);
int b200_g1_neg_batch(const uint64_t* p, size_t n, uint64_t* out);
int b200_g1_affine_batch(const uint64_t* p, size_t n, uint64_t* out_xy);
int b200_g2_add_batch(const uint64_t* p, const uint64_t* q, size_t n, uint64_t* out);
int b200_g2_double_batch(const uint64_t* p, size_t n, uint64_t* out);
int b200_g2_neg_batch(const uint64_t* p, size_t n, uint64_t* out);
int b200_g2_affine_batch(const uint64_t* p, size_t n, uint64_t* out_xy);

#ifdef __cplusplus
}
#endif
#endif /* B200SNARK_H */
