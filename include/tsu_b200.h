/*
 * tsu_b200.h - C-ABI of libtsu_b200.so: B200 (sm_100a) kernels for the data-parallel hot path
 * of tsu-emulator (heat-bath Gibbs spin updates over Ising models, batched Langevin steps).
 *
 * The reference (Arsham-001/tsu-emulator) is pure Python/NumPy and has no FFI of its own; the
 * boundary it exposes is its Python class API.  Each entry point below names the reference
 * interface (file:line under /root/reference) whose inner loop it replaces.  The Python host
 * layer (tsu_emulator_b200/*.py) binds these with ctypes and mirrors the reference classes;
 * INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every d_* pointer is DEVICE memory owned by the caller
 *     (torch allocates it), h_* pointers are host memory; `stream` is a cudaStream_t passed as
 *     uintptr_t (0 = default stream).  Nothing is allocated or freed behind the caller's back
 *     and no call synchronises the device.
 *   - return value: 0 = ok; negative = TSU_ERR_* (invalid argument, ...); positive = the
 *     cudaError_t of the launch.  Nothing throws.
 *   - spins are stored as bits: bit 1 <=> s = +1 (tsu/models/ising.py:119-125).
 *   - all randomness is counter-based Philox4x32-10 keyed by (seed, coordinates); it replaces the
 *     global numpy stream (tsu/gibbs.py:126,157,201; tsu/core.py:78,143).
 */
#ifndef TSU_B200_H
#define TSU_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TSU_OK 0
#define TSU_ERR_INVALID_ARG (-1)
#define TSU_ERR_UNSUPPORTED (-2)
#define TSU_ERR_NO_DEVICE (-3)

#define TSU_B200_ABI_VERSION 2

int tsu_version(void);
const char* tsu_error_string(int code);
/* number of SMs / compute capability of the current device; TSU_ERR_NO_DEVICE without a GPU */
int tsu_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------ Philox4x32-10 ---- */
/* host-side single block (known-answer tests; same code as the device generator) */
void tsu_philox4x32_10_host(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
/* d_out[i] = word (i&3) of Philox(counter=(i>>2 lo, i>>2 hi, offset lo, 'FILL'), key=seed) */
int tsu_philox_fill_u32(uint32_t* d_out, uint64_t n, uint64_t seed, uint32_t offset, uintptr_t stream);

/* ------------------------------------------------------------------ peer-mapped buffers */
/* Device buffers that other processes of the same box can map (CUDA IPC over NVLink): the halo rows of the
 * row-slab driver are written straight into the neighbour's buffer.  tsu_peer_alloc is the one place where the
 * library allocates device memory (zero-filled cudaMalloc: pooled / virtual-memory allocations cannot be exported);
 * the owner frees it with tsu_peer_free after every peer has closed its mapping. */
int tsu_peer_alloc(void** d_ptr, size_t bytes);
int tsu_peer_free(void* d_ptr);
int tsu_peer_get_handle(void* d_ptr, unsigned char handle[64]);
int tsu_peer_open_handle(const unsigned char handle[64], void** d_ptr);
int tsu_peer_close_handle(void* d_ptr);
/* one word of such a buffer to the host (synchronising copy; status words) */
int tsu_peer_read_u32(const void* d_ptr, uint32_t* h_out);

/* ------------------------------------------------------------------ 2-D lattice ------- */
/* The lattice kernels read their tuning knobs (TSU_LATTICE_STRIP, TSU_LATTICE_W, TSU_LATTICE_RESIDENT,
 * TSU_LATTICE_OPEN_GENERIC, TSU_LATTICE_OBS_GENERIC, TSU_JIT_W, TSU_JIT_MINB, TSU_JIT_UNROLL: launch shapes and
 * kernel choice, never results) from the environment once, when the library is loaded; this reads them again. */
void tsu_ising2d_reload_tuning(void);
/*
 * Replaces the inner loop of GibbsSampler.gibbs_sweep / sample_conditional
 * (tsu/gibbs.py:102-162) for the nearest-neighbour lattice that IsingGrid wires up
 * (tsu/models/ising.py:320-361), and README's IsingModel2D.gibbs_update (README.md:116-131).
 *
 * State layout (uint32 words): state[replica][colour][row][wpr]
 *   colour = (row_global + col) & 1 (0 = "black", updated first); within a row the sites of one
 *   colour are compressed: col = 2k + ((row_global + colour) & 1); word w holds k in [32w,32w+32),
 *   lane b = k & 31.  wpr = tsu_ising2d_words_per_row(cols) (padded to 4 words = 16 bytes);
 *   padding bits are always 0.
 *
 * Threshold table `lut` (uint32[32] per table): lut[d*5+u] = ceil(p * 2^32) for a site with d
 *   existing neighbours of which u are up, p = sigmoid(h_bit/T) computed by the HOST in float64
 *   with the reference's formula (tsu/gibbs.py:61-77,124-125); lut[25] bit (d*5+u) set means
 *   p == 1.0 (always accept).  New bit = 1 iff uniform_u32 < threshold, which is exactly
 *   `np.random.rand() < prob` of tsu/gibbs.py:126 for uniforms of the form k / 2^32.
 *   d_lut holds n tables; d_lut_index[replica] picks one (NULL: all replicas use table 0).
 */
int64_t tsu_ising2d_words_per_row(int cols);
int64_t tsu_ising2d_state_words(int rows, int cols); /* per replica: 2 * rows * wpr */

/* iid Bernoulli(1/2) configuration from Philox (kind=2 stream); replaces np.random.randint(0,2,N)
 * of tsu/gibbs.py:201.  row0 = global index of local row 0, replica0 = global index of replica 0. */
int tsu_ising2d_init_random(uint32_t* d_state, int n_replicas, int rows, int cols, uint64_t seed,
                            uint32_t replica0, int row0, uintptr_t stream);
/* int8 spins[replica][row][col] (bit = value > 0) <-> packed state */
int tsu_ising2d_pack(const int8_t* d_spins, uint32_t* d_state, int n_replicas, int rows, int cols,
                     uintptr_t stream);
int tsu_ising2d_unpack(const uint32_t* d_state, int8_t* d_spins, int n_replicas, int rows, int cols,
                       int as_pm1, uintptr_t stream);

/* One half-sweep: every site of `colour` in the local rows [row_begin, row_end) is resampled (heat bath); the other
 * rows are neither read for writing nor written (0, rows: all).  Uniforms come from the in-register Philox stream
 * (seed, replica0+replica, sweep, row0+row, word), so the bits are identical for any split of the rows: a row-slab
 * driver can update its two boundary rows first, send them to the ring neighbours and update the interior while the
 * halo exchange is in flight.
 * d_halo_top / d_halo_bot: [n_replicas][wpr] words of the OPPOSITE colour for global rows
 * row0-1 / row0+rows (row-slab sharding); NULL = wrap inside the local array if wrap_rows,
 * else open edge.  wrap_cols: periodic in the column direction (cols must be even).
 * jit_handle > 0 selects the run-time specialised kernel of tsu_ising2d_jit_prepare where it applies (d_lut_index and
 * d_bonds NULL), 0 the prebuilt kernels; same bits either way.
 * d_bonds / d_bond_index: +-J bonds (tsu_ising2d_pack_bonds below) or NULL; bonds serve whole lattices only, so with
 * bonds a halo or row0 != 0 is TSU_ERR_INVALID_ARG. */
int tsu_ising2d_half_sweep(int jit_handle, uint32_t* d_state, int n_replicas, int rows, int cols,
                           int wrap_rows, int wrap_cols, int colour, const uint32_t* d_lut,
                           const int32_t* d_lut_index, const uint32_t* d_bonds, const int32_t* d_bond_index,
                           uint64_t seed, uint32_t sweep, uint32_t replica0, int row0,
                           const uint32_t* d_halo_top, const uint32_t* d_halo_bot,
                           int row_begin, int row_end, uintptr_t stream);

/* n_sweeps sweeps of ONE row slab of a lattice that is split over the GPUs of a box, halo exchange included: the
 * compute step and its exchange in one call, no collective library in the data path.  Per half-sweep
 *   side stream: wait for the neighbours' rows of the other colour -> update rows 0 and rows-1 -> copy them into
 *                the neighbours' halo buffers (peer-mapped pointers, NVLink) -> publish the message number
 *   main stream: update rows 1 .. rows-2 meanwhile (they need no halo)
 * d_halo [2 colours][2: above / below][n_replicas][wpr] and d_flags [>= 9 words: 2 x 2 arrival counters, word 8 =
 * status, set to 1 if a neighbour's rows did not arrive within ~20 s] are this rank's buffers (tsu_peer_alloc);
 * d_up_* / d_down_* are the mapped buffers of the ranks holding the rows above / below (NULL = open edge).
 * msgs_colour0/1: messages already exchanged per colour before this call (every rank passes the same numbers; the
 * call exchanges n_sweeps of colour 0 and n_sweeps + 1 of colour 1).  rows >= 4.  Bits are identical to the
 * unsharded lattice (global-row Philox counters).  Large slabs: the interior rows of a half-sweep are launched as up
 * to 8 row ranges on library-owned streams (see tsu_ising2d_sweeps); everything is joined back into main_stream
 * before the call returns. */
int tsu_ising2d_slab_sweeps_p2p(int jit_handle, uint32_t* d_state, int n_replicas, int rows, int cols,
                                int wrap_cols, const uint32_t* d_lut, const int32_t* d_lut_index,
                                uint64_t seed, uint32_t sweep0, int n_sweeps, uint32_t replica0, int row0,
                                uint32_t* d_halo, uint32_t* d_flags, uint32_t* d_up_halo,
                                uint32_t* d_up_flags, uint32_t* d_down_halo, uint32_t* d_down_flags,
                                uint32_t msgs_colour0, uint32_t msgs_colour1, uintptr_t main_stream,
                                uintptr_t side_stream);
/* n_sweeps full sweeps (black then white), sweep indices sweep0 .. sweep0+n_sweeps-1, no halos; jit_handle and
 * d_bonds / d_bond_index as in tsu_ising2d_half_sweep.
 * Two launches per sweep; lattices of at most 4096 words per replica in batches that would not fill the GPU
 * (BASELINE config 1: 50 x 50) run ALL sweeps of the call in ONE launch, one thread block per replica.  Same
 * bits either way (TSU_LATTICE_RESIDENT=0 disables the single-launch form).
 * Launches of 1e9 .. 6e10 sites with at least 2048 rows: every half-sweep is cut into 8 row ranges launched on
 * library-owned non-blocking streams (created once per device), range k waiting by events only for ranges k-1, k,
 * k+1 of the half-sweep before, so that the next half-sweep fills the SMs while this one drains (+3 .. 11 %).  The
 * extra streams fork from `stream` and are joined back into it before the call returns: to the caller the call is
 * still ordered on `stream` alone.  TSU_LATTICE_SPLIT=1 keeps one launch per half-sweep; same bits either way. */
int tsu_ising2d_sweeps(int jit_handle, uint32_t* d_state, int n_replicas, int rows, int cols,
                       int wrap_rows, int wrap_cols, const uint32_t* d_lut, const int32_t* d_lut_index,
                       const uint32_t* d_bonds, const int32_t* d_bond_index, uint64_t seed,
                       uint32_t sweep0, int n_sweeps, uint32_t replica0, uintptr_t stream);
/* Run-time specialisation (NVRTC) of the fast half-sweep kernel for ONE threshold table (all replicas at the
 * same temperature): the eight 5-bit truth tables of h_lut (host copy of the table, layout above) become
 * literals of csrc/ising2d_fast.cuh, which removes the jump tables from the inner loop (+17 % measured).
 * src_dir = directory that holds ising2d_fast.cuh and philox.cuh.  Returns a handle >= 1 to pass as jit_handle, or
 * 0 when NVRTC / the driver API is unavailable or compilation failed (log_buf gets the reason): callers then pass 0
 * and keep using the prebuilt kernels.  Results are bit-identical to the prebuilt kernels; geometries outside the
 * fast path silently use the prebuilt generic kernel. */
int tsu_ising2d_jit_prepare(const uint32_t* h_lut, const char* src_dir, char* log_buf, int log_len);

/* Parity mode: same update, but the uniform of site (replica,row,col) is read from
 * d_uniforms[replica][row][col] (uint32 k meaning k/2^32) instead of Philox.  Bonds as in tsu_ising2d_half_sweep. */
int tsu_ising2d_half_sweep_injected(uint32_t* d_state, int n_replicas, int rows, int cols,
                                    int wrap_rows, int wrap_cols, int colour, const uint32_t* d_lut,
                                    const int32_t* d_lut_index, const uint32_t* d_bonds,
                                    const int32_t* d_bond_index, const uint32_t* d_uniforms, int row0,
                                    const uint32_t* d_halo_top, const uint32_t* d_halo_bot, uintptr_t stream);
/* d_out[replica][0] = number of up spins, d_out[replica][1] = number of anti-aligned bonds
 * (right + down bonds of every local site, wiring of tsu/models/ising.py:343-361).
 * d_next_rows: [n_replicas][2][wpr] both colours of global row row0+rows (slab sharding) or NULL.
 * M and E follow on the host: M = (2 up - N)/N, E = -J (n_bonds - 2 anti) - h (2 up - N)
 * (tsu/models/ising.py:98-117,183-193).
 * With d_bonds (whole lattices only: d_next_rows NULL, row0 0), d_out[replica][1] counts the UNSATISFIED bonds
 * (sigma_ij s_i s_j = -1), so that tsu_ising2d_energy_from_observables gives E = -J sum sigma_ij s_i s_j - h sum s_i
 * unchanged. */
int tsu_ising2d_observables(const uint32_t* d_state, int n_replicas, int rows, int cols,
                            int wrap_rows, int wrap_cols, const uint32_t* d_bonds,
                            const int32_t* d_bond_index, int row0, const uint32_t* d_next_rows,
                            unsigned long long* d_out, uintptr_t stream);
/* d_energy[r] = -J (n_bonds - 2 anti_r) - h (2 up_r - n_sites)   (float64) */
int tsu_ising2d_energy_from_observables(const unsigned long long* d_obs, int n_replicas, double J,
                                        double h, int64_t n_bonds, int64_t n_sites,
                                        double* d_energy, uintptr_t stream);

/* Edwards-Anderson +-J lattices: coupling J_ij = J sigma_ij with a sign sigma_ij = +-1 per nearest-neighbour bond.
 * The field of the bit model is 4J u' + 2h - 2J d, with u' the number of neighbours j with b_j XOR [sigma_ij = -1]:
 * the ferromagnet's threshold tables (bias "physical") serve it unchanged, so every rule above (Philox stream, ties,
 * kernels chosen, launch paths) holds; the neighbour words are XOR-ed with bond words before the up-count.  Whole
 * lattices only (no row slabs or halos); the run-time specialised kernel has no bonded form.
 *
 * d_signs: int8 [n_real][2][rows][cols]; [k][0][i][j] is the bond (i,j)-(i,(j+1) mod cols), [k][1][i][j] the bond
 *   (i,j)-((i+1) mod rows,j); a value < 0 is antiferromagnetic.  Bonds the wiring does not create (open edges, a
 *   wrap that is off) are ignored.
 * d_bonds: uint32 [n_real][colour][4: N, S, W, E][rows][wpr], aligned with the state words: bit b of word w is 1 iff
 *   the bond between own-colour lane 32w+b and that neighbour is antiferromagnetic (absent neighbours and padding
 *   lanes 0).  8 * rows * wpr words per realisation.
 * d_bond_index: [n_replicas] realisation of each replica, or NULL (all use realisation 0). */
int tsu_ising2d_pack_bonds(const int8_t* d_signs, uint32_t* d_bonds, int n_real, int rows, int cols,
                           int wrap_rows, int wrap_cols, uintptr_t stream);
/* spin overlap: d_out[q] = number of sites where replicas d_pairs[2q] and d_pairs[2q+1] differ
 * (q_ab = 1 - 2 d_out / (rows cols)); 1 <= n_pairs <= 65535, indices in [0, n_replicas) */
int tsu_ising2d_overlap(const uint32_t* d_state, int n_replicas, int rows, int cols,
                        const int32_t* d_pairs, int n_pairs, unsigned long long* d_out,
                        uintptr_t stream);

/* Simulated annealing of whole lattices (tsu/gibbs.py:340-393 on the lattice): n_steps sweeps, step k with the
 * threshold table d_luts[k] (layout above) and sweep index sweep0 + k, for every replica; no host sync inside.
 * The initial state and the state after every step are evaluated: d_energy[r] gets E of the final state (formula and
 * float64 rounding of tsu_ising2d_energy_from_observables, exact integer counts), and with d_best_energy /
 * d_best_state (in/out, both set or both NULL) a replica whose E is strictly below d_best_energy[r] takes E and
 * copies its state words [2][rows][wpr] to d_best_state[r].  An anneal split into calls that share the best buffers
 * therefore equals one call.  The bits equal, step for step, tsu_ising2d_sweeps(n_sweeps = 1) with that table
 * followed by tsu_ising2d_observables and tsu_ising2d_energy_from_observables.
 * Bonds as in tsu_ising2d_sweeps; whole lattices only (no halos, row0 = 0); always the prebuilt kernels.
 * d_obs: [n_replicas][2] scratch (left holding flags, not counts).  n_steps = 0 evaluates the initial state only.
 * Lattices that tsu_ising2d_sweeps runs in one launch run the whole anneal in one launch, one thread block per
 * replica (TSU_LATTICE_RESIDENT=0 disables); the others run per step the sweep launches of tsu_ising2d_sweeps, the
 * counts, one select kernel and, for the replicas that improved, one copy kernel.  Replica chunks anneal on streams
 * of their own; everything is joined back into `stream` before the call returns. */
int tsu_ising2d_anneal(uint32_t* d_state, int n_replicas, int rows, int cols, int wrap_rows, int wrap_cols,
                       const uint32_t* d_luts, int n_steps, const uint32_t* d_bonds,
                       const int32_t* d_bond_index, uint64_t seed, uint32_t sweep0, uint32_t replica0,
                       double J, double h, long long n_bonds, long long n_sites,
                       unsigned long long* d_obs, double* d_energy, double* d_best_energy,
                       uint32_t* d_best_state, uintptr_t stream);

/* Population annealing of whole lattices (Hukushima-Iba, Machta): the n_replicas replicas form n_populations equal
 * contiguous populations of R_p = n_replicas / n_populations replicas, each resampled on its own; no host sync inside.
 * The caller guarantees one bond realisation per population (d_bond_index constant within each).  Step k of n_steps:
 *   1. count: exact (up, anti) of every replica as tsu_ising2d_observables, E_i with the rounding of
 *      tsu_ising2d_energy_from_observables; d_count_sums[k][p] = (sum up, sum anti), d_energy_ref[k][p] = min_i E_i.
 *   2. weigh: x_i = d_dbeta[k] (E_i - E_ref) (d_dbeta[k] = 1/T_k - 1/T_{k-1} >= 0, float64),
 *      q_i = floor(exp(-x_i) 2^s) with s = 62 - ceil(log2 R_p) and exp spelled out in float64 adds and multiplies
 *      rounded to nearest (range reduction, degree-13 polynomial, ldexp: within 1 ulp of exp on [0, 45], exp(0) = 1);
 *      q_i = 0 when rint(x_i / ln 2) > s + 1.  d_weight_sum[k][p] = W = sum q_i, 2^s <= W <= 2^62.  Dropping
 *      weights below 2^-s biases ln(W / (R_p 2^s)) by at most R_p 2^-s / W <= 2^-31.
 *   3. resample, systematically, R_p fixed: u = one 64-bit draw of the lattice stream (kind 3, replica
 *      replica0 + p R_p, sweep sweep0 + k sweeps_per_step), U = floor(u W / 2^64); with inclusive prefix sums C_i the
 *      parent of child j is the smallest i with R_p C_i > j W + U (integer arithmetic: any scan order gives the same).
 *   4. gather: state'[j] = state[parent(j)], family'[j] = d_family[parent(j)] (ping-pong with d_scratch /
 *      d_family_scratch; the result always ends in d_state / d_family).
 *   5. sweep: sweeps_per_step sweeps with table d_luts[k] and sweep indices sweep0 + k sweeps_per_step ...; the launches
 *      of tsu_ising2d_sweeps with the prebuilt kernels (each step's sweeps joined before the next counts).
 * After the last step the final states are counted into d_count_sums[n_steps] and d_energy[r] = E of replica r.
 * With d_dbeta all 0 every parent is its child, so the run equals tsu_ising2d_sweeps(n_steps sweeps_per_step).
 * A block of whole populations run on its own (its replica0, its family entries) equals that block of the whole run.
 * Buffers: d_scratch [n_replicas][2][rows][wpr], d_family / d_family_scratch int32 [n_replicas],
 *   d_weight_sum uint64 [n_steps][n_populations], d_energy_ref [n_steps][n_populations],
 *   d_count_sums uint64 [n_steps + 1][n_populations][2], d_obs [n_replicas][2] scratch, d_energy [n_replicas],
 *   d_work of at least tsu_ising2d_population_work_bytes(n_replicas, n_populations) bytes, 8-byte aligned (prefix
 *   sums; the library allocates nothing).  Bonds as in tsu_ising2d_sweeps; whole lattices only.
 * TSU_ERR_INVALID_ARG before any CUDA call for: n_replicas % n_populations != 0, n_populations outside [1, 65535],
 *   sweeps_per_step < 1, n_steps < 0, a NULL pointer, d_scratch == d_state, d_family_scratch == d_family, a work
 *   buffer below the size, and the lattice rules of tsu_ising2d_sweeps.  More than 65535 replicas of a lattice
 *   without full words (cols % 256 != 0) are counted by one warp per replica. */
int64_t tsu_ising2d_population_work_bytes(int n_replicas, int n_populations);
int tsu_ising2d_population_anneal(uint32_t* d_state, uint32_t* d_scratch, int n_replicas, int rows, int cols,
                                  int wrap_rows, int wrap_cols, const uint32_t* d_luts, const double* d_dbeta,
                                  int n_steps, int sweeps_per_step, int n_populations, const uint32_t* d_bonds,
                                  const int32_t* d_bond_index, uint64_t seed, uint32_t sweep0, uint32_t replica0,
                                  double J, double h, long long n_bonds, long long n_sites, int32_t* d_family,
                                  int32_t* d_family_scratch, unsigned long long* d_weight_sum, double* d_energy_ref,
                                  unsigned long long* d_count_sums, unsigned long long* d_obs, double* d_energy,
                                  void* d_work, size_t work_bytes, uintptr_t stream);

/* One resampling step of population annealing on the chain states of any back end (GibbsSampler.population_annealing):
 * n_chains rows of row_bytes bytes (d_state, read only), forming n_populations equal contiguous populations of
 * R_p = n_chains / n_populations chains, each resampled on its own; no host sync.  Steps 2-4 of
 * tsu_ising2d_population_anneal with E_i = d_energy[i] (float64):
 *   E_ref = min_i E_i of the population -> d_energy_ref[p];
 *   q_i = floor(exp(-x_i) 2^s), x_i = *d_dbeta (E_i - E_ref), s = 62 - ceil(log2 R_p), exp as spelled out there;
 *   W = sum q_i -> d_weight_sum[p];
 *   u = one 64-bit draw of the lattice stream (kind 3, replica chain0 + p R_p (mod 2^32), sweep `sweep`),
 *   U = floor(u W / 2^64); the parent of child j is the smallest i with R_p C_i > j W + U (C: inclusive prefix sums);
 *   gather: d_state_out[j] = d_state[parent(j)], d_family_out[j] = d_family[parent(j)] (int32).
 * Rows of a multiple of 16 bytes at 16-byte aligned bases are copied in 16-byte vectors, others byte by byte; only
 * the n_chains rows of d_state_out and entries of d_family_out are written.  A block of whole populations run on its
 * own (its chain0, its slices of every buffer) equals that block of the whole call.
 * d_work: at least tsu_ising2d_population_work_bytes(n_chains, n_populations) bytes, 8-byte aligned.
 * TSU_ERR_INVALID_ARG before any CUDA call for: a NULL pointer, n_chains < 1, n_populations outside [1, 65535] or not
 * dividing n_chains, row_bytes < 1, d_state_out == d_state, d_family_out == d_family, and a work buffer below the
 * size or not 8-byte aligned. */
int tsu_population_resample(const void* d_state, void* d_state_out, const int32_t* d_family, int32_t* d_family_out,
                            const double* d_energy, const double* d_dbeta, int n_chains, int n_populations,
                            long long row_bytes, uint64_t seed, uint32_t sweep, uint32_t chain0,
                            unsigned long long* d_weight_sum, double* d_energy_ref, void* d_work, size_t work_bytes,
                            uintptr_t stream);
/* Per population p of n_populations equal contiguous populations of d_energy [n_chains]:
 * d_moments[p][0] = sum E, d_moments[p][1] = sum E^2, in float64 with one fixed summation order per population, so a
 * block of whole populations run on its own gives the same bits.  TSU_ERR_INVALID_ARG before any CUDA call for a NULL
 * pointer, n_chains < 1, and n_populations outside [1, 65535] or not dividing n_chains. */
int tsu_population_moments(const double* d_energy, int n_chains, int n_populations, double* d_moments,
                           uintptr_t stream);

/* Swendsen-Wang cluster updates of whole lattices at h = 0 ("physical" bias); no host sync, nothing allocated.
 * One step at sweep index s, for replica r with threshold t = d_thresholds[d_lut_index ? d_lut_index[r] : 0]:
 *   1. satisfied bonds: J sigma_ij s_i s_j > 0 (sigma = +-1 bond sign, +1 without bonds; J's sign is
 *      coupling_sign = +1 or -1), over the bonds tsu_ising2d_observables counts (right and down of every site, wraps
 *      only where wrap_rows / wrap_cols are set).
 *   2. activation: a satisfied bond is active iff u < t, t = ceil(p 2^32) with p = -expm1(-2|J| / T) in float64
 *      (t = 2^32: always active).  u is a 32-bit uniform of the lattice stream built as the Gibbs uniform, for the
 *      site the bond starts from: bit-planes of kinds 16, 17 and low bits of kinds 24-31 (east bonds), kinds 18, 19
 *      and 32-39 (south bonds).
 *   3. clusters: connected components of the active bonds; a cluster's root is its site with the smallest
 *      row * cols + col.
 *   4. flip: a cluster flips iff bit b of word x of the lattice call (w, colour, kind 4, row, s, replica0 + r) is 1,
 *      (colour, row, w, b) being the root's packed position.
 * n_steps steps use sweep indices sweep0 .. sweep0 + n_steps - 1; n_steps = 0 is a no-op.  The bits depend on neither
 * the launch path nor the workspace: the replicas run in chunks of work_bytes / tsu_ising2d_cluster_work_bytes(1, ..)
 * replicas, each chunk through all its steps, all ordered on `stream`.  Lattices of at most 12288 sites run every
 * step in one launch, one block per replica with the labels in shared memory (TSU_LATTICE_RESIDENT=0 disables);
 * larger ones run four launches per step: activation and flip words, union-find in shared-memory tiles of 32 x 256
 * sites, unions across tiles and wraps in global memory, and the flips.
 * d_work: at least tsu_ising2d_cluster_work_bytes(1, rows, cols) bytes, 16-byte aligned (labels, activation and flip
 * words: about 4.4 bytes per site and replica); its layout is private.  Bonds as in tsu_ising2d_sweeps.
 * TSU_ERR_INVALID_ARG before any CUDA call for: n_steps < 0, a NULL d_state / d_thresholds / d_work, a work buffer
 * below one replica, rows * cols above 2^31 - 1, coupling_sign not +-1, and the lattice rules of tsu_ising2d_sweeps.
 * tsu_ising2d_cluster_work_bytes returns 0 for a lattice it cannot serve. */
int64_t tsu_ising2d_cluster_work_bytes(int n_replicas, int rows, int cols);
int tsu_ising2d_swendsen_wang(uint32_t* d_state, int n_replicas, int rows, int cols, int wrap_rows, int wrap_cols,
                              const uint64_t* d_thresholds, const int32_t* d_lut_index, int coupling_sign,
                              const uint32_t* d_bonds, const int32_t* d_bond_index, uint64_t seed,
                              uint32_t sweep0, int n_steps, uint32_t replica0,
                              void* d_work, size_t work_bytes, uintptr_t stream);

/* Houdayer cluster moves of replica pairs (two replicas of the same couplings at the same temperature); no host sync,
 * nothing allocated.  One step at sweep index s, for each pair (a, b) of d_pairs (int32 [n_pairs][2] on the device):
 *   1. differ: d_i = x^a_i xor x^b_i at every site.
 *   2. active: a bond the wiring creates (right and down of every site, wraps only where wrap_rows / wrap_cols are
 *      set) is active iff d = 1 at both its ends.  No randomness, temperature or bond sign enters.
 *   3. clusters: connected components of the active bonds over the sites with d = 1; a cluster's root is its site
 *      with the smallest row * cols + col.
 *   4. flip: a cluster flips, in both replicas, iff bit b of word x of the lattice call (w, colour, kind 5, row, s,
 *      replica0 + a) is 1, (colour, row, w, b) being the root's packed position.  Sites with d = 0 never change.
 * The move leaves E_a + E_b and q_ab unchanged for any couplings and any uniform field, and keeps the product of the
 * two Boltzmann distributions.  The caller guarantees that the pairs are disjoint and that the two replicas of a
 * pair share couplings and temperature; a pair with an index outside [0, n_replicas) or a == b is skipped (its
 * replicas' words are neither read nor written).
 * n_steps steps use sweep indices sweep0 .. sweep0 + n_steps - 1; n_steps = 0 is a no-op.  The bits depend on neither
 * the launch path nor the workspace: the pairs run in chunks of work_bytes / tsu_ising2d_cluster_work_bytes(1, ..)
 * pairs, each chunk through all its steps, all ordered on `stream`.  Launch paths and the work buffer (one replica's
 * share per pair) as in tsu_ising2d_swendsen_wang.
 * TSU_ERR_INVALID_ARG before any CUDA call for: a NULL d_state / d_pairs / d_work, n_steps < 0, n_pairs < 1 or
 * 2 n_pairs > n_replicas, a work buffer below one pair, rows * cols above 2^31 - 1, and the lattice rules of
 * tsu_ising2d_sweeps. */
int tsu_ising2d_houdayer(uint32_t* d_state, int n_replicas, int rows, int cols, int wrap_rows, int wrap_cols,
                         const int32_t* d_pairs, int n_pairs, uint64_t seed, uint32_t sweep0, int n_steps,
                         uint32_t replica0, void* d_work, size_t work_bytes, uintptr_t stream);

/* ------------------------------------------------------------------ dense-J Gibbs ----- */
/*
 * Replaces GibbsSampler.gibbs_sweep / sample_boltzmann / compute_energy and the sweep part of
 * parallel_tempering / simulated_annealing (tsu/gibbs.py:128-236,284-303,370-391) for a batch
 * of independent chains sharing one coupling matrix.
 *   d_Jt: [N][N] row-major TRANSPOSE of the coupling matrix, Jt[i*N+j] = J[j][i] (the same array as
 *     J when J is symmetric; the reference allows asymmetric J, gibbs.py:117); j_dtype 0 = float32,
 *     1 = float64;  d_bias: [N] same dtype or NULL.
 *   d_state: [n_chains][N] uint8 bits, updated in place.
 *   Local field includes the self term J_ii s_i (tsu/gibbs.py:97).  Site i of chain c in sweep s
 *   takes new bit = 1 iff u < sigmoid(h_i / T) (sigmoid clamped at |x| > 20, gibbs.py:73-77).
 *   Temperature of (chain c, sweep s): d_T_chain ? d_T_chain[c] : (d_T_sweep ? d_T_sweep[s] : T).
 *   d_order: [n_total_sweeps][V] int32 visiting order (NULL = 0..N-1, "sequential"); V =
 *     visits_per_sweep (0 means N; V < N gives partial sweeps, e.g. one sample_conditional).
 *   d_uniforms: [n_total_sweeps][n_chains][V] float64 in visiting order (parity mode) or NULL
 *     (Philox: counter = (site, chain0+chain, sweep0+s, 'DENS')).
 *   Schedule: n_burnin sweeps, then n_samples x sweeps_per_sample sweeps; after each group the
 *   state of every chain is written to d_samples[sample][chain][N] (uint8, may be NULL).
 *   d_energy: [n_chains] float64 energy -1/2 s^T J s - b^T s of the final state (may be NULL).
 *   track_best: after every sweep keep the lowest-energy state per chain in
 *     d_best_state[n_chains][N] / d_best_energy[n_chains] (simulated annealing, gibbs.py:387-391).
 *   acc_dtype: 0 = float32 fields, 1 = float64 fields.
 */
int tsu_dense_gibbs_run(const void* d_Jt, int j_dtype, const void* d_bias, uint8_t* d_state,
                        int n_chains, int N, double T, const double* d_T_chain,
                        const double* d_T_sweep, int n_burnin, int n_samples,
                        int sweeps_per_sample, const int32_t* d_order, const double* d_uniforms,
                        uint8_t* d_samples, double* d_energy, int track_best,
                        uint8_t* d_best_state, double* d_best_energy, uint64_t seed,
                        uint32_t sweep0, uint32_t chain0, int acc_dtype, int visits_per_sweep,
                        uintptr_t stream);
/* d_energy[c] = -1/2 s^T J s - b^T s   (tsu/gibbs.py:215-236), float64 accumulation */
int tsu_dense_energy(const void* d_Jt, int j_dtype, const void* d_bias, const uint8_t* d_state,
                     int n_chains, int N, double* d_energy, uintptr_t stream);
/* iid Bernoulli(1/2) chain states from Philox ('DINI' stream); np.random.randint(0,2,N) of gibbs.py:201 */
int tsu_dense_init_random(uint8_t* d_state, int n_chains, int N, uint64_t seed, uint32_t chain0,
                          uintptr_t stream);

/* Batched dense-J Gibbs sweeps on the tensor cores (BASELINE config 3; csrc/dense_tc.cu).  Same sequential
 * heat-bath rule as tsu_dense_gibbs_run (sites 0..N-1 in order, every update sees all earlier ones), blocked on two
 * levels: per 128-site PANEL the fields of a CTA's 128 (or 64) chains are one M x 128 x N tcgen05 GEMM (bf16 J by
 * TMA with 128-byte swizzle, spins expanded to bf16 0 / 2 straight into tensor memory, fp32 accumulation in TMEM);
 * per 32-site BLOCK the sites are walked in registers with rank-1 corrections, and one small MMA carries the
 * block's flips to the rest of the panel.  Identical to the site-by-site sweep for the same fields.
 *   d_J_bf16: [N][N] row-major bf16, row i = couplings into site i (J itself, not the transpose);
 *   d_bias: [N] float32 or NULL; d_state: [n_chains][N] uint8 bits in place; N % 128 == 0, N <= 4096
 *   (the host mirror pads other sizes with uncoupled sites).
 *   Uniform of (site, chain, sweep): 24 bits of word (site & 3) of Philox(counter = (site >> 2,
 *   chain0 + chain, sweep0 + sweep, 'DENT')).  Acceptance  u < sigmoid(h/T)  is evaluated as  h > T * logit(u)
 *   (strict; thresholds clamped to +-20 T = the reference's sigmoid clamp) with logit(u) from lg2.approx in fp32:
 *   against the float64 rule it can only disagree where |u - sigmoid(h/T)| < ~5e-6 for exactly representable
 *   couplings, ~5e-5 for Gaussian couplings up to N = 4096 (counted and bounded by tests/test_dense_gpu.py).
 *   d_fields_or_null: [n_chains][N] float32, diagnostics: the local field of every site as the kernel compares it on
 *   its last visit. */
int tsu_dense_gibbs_tc_run(const void* d_J_bf16, const float* d_bias, uint8_t* d_state, int n_chains,
                           int N, double T, const double* d_T_chain, int n_sweeps, uint64_t seed,
                           uint32_t sweep0, uint32_t chain0, float* d_fields_or_null, uintptr_t stream);

/* Tensor-core (tcgen05) evaluation of the local fields of EVERY site for a batch of chains:
 * d_fields[c][i] = sum_k J[i][k] * state[c][k]  (J bf16 [N][N] row-major, fp32 accumulation in TMEM).
 * This is _compute_local_field (tsu/gibbs.py:79-100) for all (chain, site) pairs at once; it is the GEMM
 * stage of the blocked tensor-core sweep and is exported so that it can be validated on its own.
 * N must be a multiple of 128 and <= 4096. */
int tsu_dense_tc_debug_fields(const void* d_J_bf16, const uint8_t* d_state, int n_chains, int N,
                              float* d_fields, uintptr_t stream);

/* Energy of every chain on the tensor cores (simulated annealing and replica exchange on the bf16 path):
 *   d_energy[c] = -1/2 s^T J s - b^T s   (tsu/gibbs.py:215-236)
 * for the bf16 couplings d_J_bf16 ([N][N] row-major, as tsu_dense_gibbs_tc_run) and the float32 bias d_bias (or NULL).
 * The fields f = S J^T come from the same GEMM as tsu_dense_tc_debug_fields (fp32 accumulation in TMEM); the thread of
 * chain c then sums s_i f_i and s_i b_i in float64 over the sites i = 0 .. N-1 in order, so the value does not depend on
 * the tile height or on how the chains are split into launches, and it is exact for couplings and bias of the form
 * m / 2^k.  d_state is read only.
 * Best-state tracking (tsu/gibbs.py:387-391): pass d_best_energy [n_chains] and d_best_state [n_chains][N] together
 * (or both NULL).  Where d_energy[c] < d_best_energy[c] (strict), both are replaced by the chain's energy and state;
 * rows of the other chains are not written.  N % 128 == 0, N <= 4096. */
int tsu_dense_tc_energy(const void* d_J_bf16, const float* d_bias, const uint8_t* d_state, int n_chains,
                        int N, double* d_energy, double* d_best_energy, uint8_t* d_best_state,
                        uintptr_t stream);

/* Chromatic Gibbs sweeps for SPARSE couplings (csrc/sparse_gibbs.cu): IsingChain (tsu/models/ising.py:265-304),
 * irregular graphs, MAX-CUT instances.  J in CSR (row i = couplings into site i, ascending columns, self term
 * allowed), sites grouped into colour classes such that no two coupled sites share one (d_colour_sites, offsets in
 * d_colour_ptr).  A sweep visits the classes in order; the sites of a class are updated concurrently, which equals
 * the reference's sequential sweep (tsu/gibbs.py:153-160) in that visiting order - update_order="random" with the
 * class order as the permutation.  One CTA per chain, bits in shared memory (N <= 204800), float64 fields;
 * schedule, outputs, per-chain / per-sweep temperatures and best-state tracking as in tsu_dense_gibbs_run, and the
 * same Philox uniforms per (site, chain, sweep).  d_uniforms (parity mode): [sweep][chain][N] in visiting order. */
int tsu_sparse_gibbs_run(const int32_t* d_rowptr, const int32_t* d_col, const double* d_val,
                         const double* d_bias, const int32_t* d_colour_ptr, const int32_t* d_colour_sites,
                         int n_colours, uint8_t* d_state, int n_chains, int N, double T,
                         const double* d_T_chain, const double* d_T_sweep, int n_burnin, int n_samples,
                         int sweeps_per_sample, const double* d_uniforms, uint8_t* d_samples, double* d_energy,
                         int track_best, uint8_t* d_best_state, double* d_best_energy, uint64_t seed,
                         uint32_t sweep0, uint32_t chain0, uintptr_t stream);

/* Houdayer cluster moves of chain pairs on SPARSE couplings (csrc/sparse_houdayer.cu), the overlap-cluster move of
 * ICM (Zhu, Ochoa & Katzgraber 2015) on any graph.  d_state is the [n_chains][N] uint8 state of tsu_sparse_gibbs_run,
 * couplings in its CSR form (d_rowptr, d_col, d_val, d_bias may be NULL).  No host sync, nothing allocated.  One step
 * at index s, for each pair (a, b) of d_pairs (int32 [n_pairs][2] on the device):
 *   1. differ: d_i = x^a_i xor x^b_i.
 *   2. graph: edge {i, j} for every stored entry J_ij != 0 of row i with j > i (self couplings never join); for the
 *      symmetric couplings the move is meant for, that is every coupled pair.
 *   3. clusters: connected components of the graph restricted to the sites with d = 1; a cluster's root is its
 *      smallest site index.
 *   4. flip: a cluster flips, x^a_i ^= 1 and x^b_i ^= 1 on all its sites (the two chains swap their bits there), iff
 *      bit 0 of word 0 of Philox(counter = (root, chain0 + a, s, 'HOUD'), key = seed) is 1.  Sites with d = 0 never
 *      change.
 * For symmetric J the move leaves E_a + E_b and the overlap unchanged, for any bias and self couplings, and keeps the
 * product of the two Boltzmann distributions.  The caller guarantees that the pairs are disjoint and that the two
 * chains of a pair share couplings and temperature; a pair with an index outside [0, n_chains) or a == b is skipped
 * (its rows are neither read nor written).  n_steps steps use the indices step0 .. step0 + n_steps - 1; n_steps = 0 is
 * a no-op.  With d_energy, every processed chain gets E = -1/2 s^T J s - b^T s of its final state, bit for bit the
 * value tsu_sparse_gibbs_run reports for that state.  Rows are written back as 0 / 1 bytes.
 * One CTA per pair runs all steps.  Up to N = 32768 the rows and labels stay in shared memory and d_work is unused;
 * above that (to the sweep kernel's N <= 204800) the labels go to d_work, tsu_sparse_houdayer_work_bytes(1, N) bytes
 * per pair (16-byte aligned), and the pairs run in chunks of work_bytes / that, each chunk through all its steps, all
 * ordered on `stream`.  The bits depend on neither path nor chunking.
 * TSU_ERR_INVALID_ARG before any CUDA call for: a NULL d_rowptr / d_col / d_val / d_state / d_pairs, N outside
 * [1, 204800], n_steps < 0, n_pairs < 1 or 2 n_pairs > n_chains, and (above N = 32768) a NULL or not 16-byte aligned
 * d_work or a work buffer below one pair.  tsu_sparse_houdayer_work_bytes returns 0 when no workspace is needed or the arguments cannot be
 * served. */
int64_t tsu_sparse_houdayer_work_bytes(int n_pairs, int N);
int tsu_sparse_houdayer(const int32_t* d_rowptr, const int32_t* d_col, const double* d_val, const double* d_bias,
                        uint8_t* d_state, int n_chains, int N, const int32_t* d_pairs, int n_pairs,
                        uint64_t seed, uint32_t step0, int n_steps, uint32_t chain0, double* d_energy,
                        void* d_work, size_t work_bytes, uintptr_t stream);

/* Replica-exchange pass (tsu/gibbs.py:308-323): for each ladder, pairs i = 0..R-2 in order;
 * delta = (1/T_i - 1/T_{i+1}) (E_{i+1} - E_i); accept if delta >= 0 or u < exp(delta) (u drawn
 * only when delta < 0).  Configurations stay in place; d_slot_replica[ladder][i] (the replica
 * currently at temperature slot i) is permuted instead, and d_lut_index[replica] (may be NULL)
 * is updated to the slot for the lattice kernels.  d_stats[0] += attempts, d_stats[1] += accepts.
 * d_uniforms: [n_ladders][R-1] float64 (parity mode) or NULL (Philox 'PTSW', step).
 * criterion: 0 = the reference's expression above (bit-parity with gibbs.py:317, which favours moving
 * HIGH-energy configurations to COLD slots); 1 = detailed-balance Metropolis rule
 * delta = (1/T_i - 1/T_{i+1}) (E_i - E_{i+1}). */
int tsu_pt_swap(const double* d_energy, const double* d_T_slot, int32_t* d_slot_replica,
                int32_t* d_lut_index, int n_ladders, int R, uint64_t seed, uint32_t step,
                unsigned long long* d_stats, const double* d_uniforms, int criterion,
                uintptr_t stream);

/* ------------------------------------------------------------------ Langevin ---------- */
/*
 * Replaces the loop of ThermalSamplingUnit.sample_from_energy (tsu/core.py:100-162) for
 * built-in analytic energies: every "sample" of the reference is an independent restarted chain
 * (core.py:140-143), so n_samples chains run in parallel, one per thread, state in registers.
 *   step (core.py:64-80):  x <- x - grad E(x) dt/gamma + sqrt(2 T dt / gamma) N(0, I)
 *   chain c starts at x_init + jitter * N(0, I) (core.py:142-143), except local chain 0 when
 *     first_chain_exact != 0, which starts exactly at x_init like the reference's first sample
 *   energy_kind / d_params (float64 device array):
 *     0 QUADRATIC    E = a * sum_i ((x_i - mu_i)^2 * w_i)         params = [a, mu[dim], w[dim]]
 *     1 MIXTURE      E = -log(sum_k p_k exp(-|x - c_k|^2 / 2) + 1e-10)   (tsu/api.py:143-149)
 *                                                                 params = [K, p[K], c[K][dim]]
 *     2 DOUBLE_WELL  E = sum_i a (x_i^2 - b)^2                    params = [a, b]
 *     3 QUADRATIC_FORM E = 1/2 x^T A x - b^T x                    params = [A[dim][dim], b[dim]]
 *   dtype 0 = float32, 1 = float64 for d_x / d_x_init / d_traj / d_normals.
 *   d_x: [n_chains][dim] final states (the reference's `samples`).
 *   d_traj: [n_chains][n_steps][dim] sampling-phase trajectory or NULL (core.py:155-156).
 *   d_normals: [n_chains][1 + n_burnin + n_steps][dim] injected N(0,1) draws (parity mode; row 0
 *     is the start jitter) or NULL (Philox + Box-Muller, counter = (chain, pair, step, 'LANG')).
 *   dim <= 64: one thread per chain, state in registers (every kind; MIXTURE needs n_params <= 20000).
 *   dim > 64 (csrc/langevin_wide.cu), TSU_ERR_INVALID_ARG past a cap:
 *     QUADRATIC, DOUBLE_WELL   dim <= 131072 (float64), 262144 (float32): the 16-bit Philox block field
 *     MIXTURE                  the same, with K <= 16 centres (K = (n_params - 1) / (dim + 1))
 *     QUADRATIC_FORM           dim <= 2048; A need not be symmetric
 *   Two rules make the wide kernels the same sampler as the register kernels:
 *     1. coordinate i takes element i % PER of Philox block b = i / PER, counter
 *        (chain lo, chain hi & 0xFFFF | b << 16, step, 'LANG'), PER = 2 (float64) or 4 (float32): its draw does not
 *        depend on dim;
 *     2. the gradient of coordinate i and its update are the same expressions in the same summation order
 *        (QUADRATIC_FORM: -b_i, then acc = fma(A_ij, x_j, acc) for ascending j; MIXTURE: d2_k over ascending i, tot and
 *        g_i over ascending k).
 *   So a coordinate that does not couple to the others gets the same bits at any dim.
 */
int tsu_langevin_run(void* d_x, int dtype, int64_t n_chains, int dim, int energy_kind,
                     const double* d_params, int n_params, const void* d_x_init, double jitter,
                     int first_chain_exact, double T, double dt, double gamma, int n_burnin, int n_steps, uint64_t seed,
                     uint64_t chain0, const void* d_normals, void* d_traj, uintptr_t stream);

/* Langevin chains for an energy that is not built in: the caller supplies the GRADIENT as CUDA source,
 *     template <typename real> __device__ __forceinline__ void tsu_user_grad(const real* x, real* g) { ... }
 * (tsu_emulator_b200/trace.py writes it from a traced and analytically differentiated Python callable - the
 * reference differentiates such callables numerically on the host, tsu/core.py:82-98), and NVRTC compiles it into
 * the same chain loop as the built-in energies (csrc/langevin_body.cuh) for one (dtype, dim).  src_dir = directory
 * of langevin_body.cuh and philox.cuh.  Returns a handle >= 1, or 0 when NVRTC / the driver API is unavailable or
 * the source does not compile (log_buf gets the reason).  tsu_langevin_run_jit takes the arguments of
 * tsu_langevin_run minus the energy description. */
int tsu_langevin_jit_prepare(const char* grad_source, int dtype, int dim, const char* src_dir,
                             char* log_buf, int log_len);
int tsu_langevin_run_jit(int handle, void* d_x, int64_t n_chains, const void* d_x_init, double jitter,
                         int first_chain_exact, double T, double dt, double gamma, int n_burnin,
                         int n_steps, uint64_t seed, uint64_t chain0, const void* d_normals,
                         void* d_traj, uintptr_t stream);

#ifdef __cplusplus
}
#endif
#endif /* TSU_B200_H */
