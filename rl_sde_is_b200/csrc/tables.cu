// K4: tabular transition tensor P[s', s, a] and reward table R[s, a]  (float64).
//
// Replaces compute_p_tensor_batch / compute_r_table (dynamic_programming.py:3-36), i.e. 180 300
// Python iterations x 4 scipy.stats.norm.cdf calls at h = 0.01, and the per-column arithmetic of
// state_action_transition_function (environments.py:87-102):
//     mu = x_s + (-gradV(x_s) + sigma a) dt,  sd = sigma sqrt(dt)
//     P[s', s, a] = Phi((x_s' + h - mu) / sd) - Phi((x_s' - h - mu) / sd)       s outside the target set
//     P[0,   s, a] += Phi((x_0 - h - mu) / sd);   P[N-1, s, a] += 1 - Phi((x_{N-1} + h - mu) / sd)
//     P[s', s, a] = 1/|TS| if s' in TS else 0                                     s in the target set
//
// Layout / mapping: the tensor is C-ordered with the action index innermost, so a warp's 32 lanes
// take 32 consecutive actions (each store instruction writes 256 contiguous bytes) and every thread
// walks TILE consecutive next-states, carrying the CDF of the shared cell edge from one cell to the
// next (TILE+1 CDF evaluations per TILE entries instead of 2 TILE).  The kernel is bound by the FP64
// pipe (erf/erfc), not by HBM: see DESIGN.md.
#include "aux_kernels.cuh"
#include "transition.cuh"

namespace rlsde {

constexpr int TABLE_TILE = 8;

__global__ void __launch_bounds__(128) tables_kernel(const double* __restrict__ sgrid, long long Ns,
                                                     const double* __restrict__ agrid, long long Na,
                                                     const unsigned char* __restrict__ in_ts, double inv_nts,
                                                     double alpha, double sigma, double dt, double h,
                                                     long long sp_begin, long long sp_end, double* __restrict__ P) {
  const long long a = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long s = blockIdx.y;
  const long long sp0 = sp_begin + (long long)blockIdx.z * TABLE_TILE;
  if (a >= Na || sp0 >= sp_end) return;
  const long long sp1 = sp0 + TABLE_TILE < sp_end ? sp0 + TABLE_TILE : sp_end;
  double* out = P + ((sp0 - sp_begin) * Ns + s) * Na + a;
  const long long stride = Ns * Na;
  if (in_ts[s]) {
    for (long long sp = sp0; sp < sp1; ++sp, out += stride) *out = in_ts[sp] ? inv_nts : 0.0;
    return;
  }
  const double xs = sgrid[s];
  const double act = agrid[a];
  // mu = state + (-gradient(state) + sigma * action) * dt,  gradient = 4 alpha x (x^2 - 1)
  const double grad = __dmul_rn(__dmul_rn(__dmul_rn(4.0, alpha), xs), __dsub_rn(__dmul_rn(xs, xs), 1.0));
  const double mu = __dadd_rn(xs, __dmul_rn(__dadd_rn(-grad, __dmul_rn(sigma, act)), dt));
  const double sd = __dmul_rn(sigma, sqrt(dt));
  double lo = ndtr(__ddiv_rn(__dsub_rn(__dsub_rn(sgrid[sp0], h), mu), sd));
  for (long long sp = sp0; sp < sp1; ++sp, out += stride) {
    // upper edge of cell sp = lower edge of cell sp+1 (x_{sp+1} - h), so each cell boundary has ONE value
    // whatever the tiling / slab; only the last cell of the grid uses its own x_sp + h
    const double edge = (sp + 1 < Ns) ? __dsub_rn(sgrid[sp + 1], h) : __dadd_rn(sgrid[sp], h);
    const double hi = ndtr(__ddiv_rn(__dsub_rn(edge, mu), sd));
    double p = hi - lo;
    if (sp == 0) p += lo;                 // left tail folded into the first row
    if (sp == Ns - 1) p += 1.0 - hi;      // right tail folded into the last row
    *out = p;
    lo = hi;
  }
}

// ---- fast path: uniform state grid with fine cells (cell width <= 0.2 sd): the Gauss-Legendre density recurrences of
// transition.cuh, one 8-byte store per entry.  One thread owns one (s, a) column of one chunk of at most GL_ANCHOR rows of
// one row class (see the kernel); columns are the flat index s * Na + a, so every lane of every warp is busy and a block
// stores 1 KB of contiguous bytes per row.

// Stores.  A row of P has Ns Na entries and Ns Na is odd at config 3 (401 x 601), so consecutive rows start 72 bytes
// apart modulo 128.  With one thread per column walking consecutive rows, a warp's 256-byte store sits at 8-byte alignment
// on three rows out of four: two partial 32-byte sectors per store instruction, and the SM-to-L2 write path -- not HBM --
// saturates (5.4 TB/s; 6.9 TB/s for the same kernel with an artificial Na = 608 or 600, i.e. rows sector-aligned;
// tools/bench_tables_align.py).  Staging the rows (shared memory + rotated stores, TMA bulk copies, in-warp shuffles) was
// measured slower than that (profiles/r02/tables_store_variants.log).  What is used instead: the rows are split into Q
// residue classes (Q = 4 for an odd row length, 2 for 2 mod 4, 1 for 0 mod 4).  Within one class every row has the SAME
// misalignment, so a block that owns (128-column tile, class j, chunk) shifts its tile left by that many columns and
// every store of every warp is 32-byte aligned; the thread then walks rows j, j + Q, j + 2Q, ... and the recurrences
// simply run with the step Q ds (their constants are formed on the host for that step).
__global__ void __launch_bounds__(128) tables_gl_kernel(const double* __restrict__ sgrid, long long Ns,
                                                        const double* __restrict__ agrid, long long Na,
                                                        const unsigned char* __restrict__ in_ts, double inv_nts,
                                                        double alpha, double sigma, double dt, double h,
                                                        long long sp_begin, long long sp_end, double* __restrict__ P,
                                                        int Q, int steps, long long kc_lo,
                                                        const __grid_constant__ GlConst C) {
  const long long stride = Ns * Na;
  const int j = (int)(blockIdx.y % (unsigned)Q);                      // row class
  const long long kc = kc_lo + blockIdx.y / (unsigned)Q;              // chunk of `steps` rows of that class
  // columns to shift left so that the first lane's address is a multiple of 32 bytes (the same for every row of the class)
  const unsigned long long rel = (unsigned long long)(((j - sp_begin) % 4 + 4) % 4) * (unsigned long long)(stride & 3);
  const long long shift = (long long)((((unsigned long long)P >> 3) + rel) & 3ull);
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x - shift;
  if (c < 0 || c >= stride) return;
  // anchors sit at absolute rows Q kc steps + j, so a slab holds exactly the entries of the full tensor
  const long long r0 = (long long)Q * kc * steps + j;
  if (r0 >= sp_end) return;
  const long long i_lo = r0 >= sp_begin ? 0 : (sp_begin - r0 + Q - 1) / Q;     // first stored step
  long long i_hi = (sp_end - r0 + Q - 1) / Q;                                  // one past the last stored step
  if (i_hi > steps) i_hi = steps;
  if (i_lo >= i_hi) return;
  const long long r_first = r0 + i_lo * Q, r_last = r0 + (i_hi - 1) * Q;
  const long long row_step = (long long)Q * stride;
  double* out = P + (r_first - sp_begin) * stride + c;                          // P points at row sp_begin
  const long long s = c / Na, a = c - s * Na;
  if (in_ts[s]) {
    for (long long sp = r_first; sp <= r_last; sp += Q, out += row_step) __stcs(out, in_ts[sp] ? inv_nts : 0.0);
    return;
  }
  const double xs = __ldg(sgrid + s);
  const double act = __ldg(agrid + a);
  const double x_lo = __ldg(sgrid + r0);
  const double inv_sd = C.inv_sd, rho = C.rho, mua = C.mu_a, mub = C.mu_b;
  const double grad = __dmul_rn(__dmul_rn(__dmul_rn(4.0, alpha), xs), __dsub_rn(__dmul_rn(xs, xs), 1.0));
  const double mu = __dadd_rn(xs, __dmul_rn(__dadd_rn(-grad, __dmul_rn(sigma, act)), dt));
  // tails folded into the first and the last row of the grid (environments.py:97-101): formed up front, added in registers
  const double tail_lo = r_first == 0 ? ndtr((__ldg(sgrid) - h - mu) * inv_sd) : 0.0;
  const double tail_hi = r_last == Ns - 1 ? 1.0 - ndtr((__ldg(sgrid + Ns - 1) + h - mu) * inv_sd) : 0.0;
  const double m = fma(x_lo - h - mu, inv_sd, 0.5 * C.dcell);       // midpoint of cell r0
  double phi = 0.3989422804014327 * exp(-0.5 * m * m);
  double r = exp(-fma(m, C.dstep, C.half_ds2));
  const double ea = exp(m * C.off_a), eb = exp(m * C.off_b);
  const double ia = 1.0 / ea, ib = 1.0 / eb;
  double ya = C.coef_a * (0.5 * (ea + ia)), yb = C.coef_b * (0.5 * (eb + ib));
  // first difference: cosh((m + ds) o) - cosh(m o) = 2 sinh((m + ds/2) o) sinh(ds o / 2)
  double da = C.coef_a * ((ea * C.eh_a - ia / C.eh_a) * C.sh_a);
  double db = C.coef_b * ((eb * C.eh_b - ib / C.eh_b) * C.sh_b);
  for (long long i = 0; i < i_lo; ++i) {                    // a slab that starts inside a chunk: advance without storing
    phi *= r; r *= rho;
    ya += da; da = fma(mua, ya, da);
    yb += db; db = fma(mub, yb, db);
  }
  const int n = (int)(i_hi - i_lo);
#pragma unroll 8
  for (int i = 0; i < n; ++i) {
    double p = phi * (ya + yb);
    if (i == 0) p += tail_lo;
    if (i == n - 1) p += tail_hi;
    __stcs(out, p);                         // streaming store: the tensor is written once and is larger than L2
    out += row_step;
    phi *= r; r *= rho;
    ya += da; da = fma(mua, ya, da);
    yb += db; db = fma(mub, yb, db);
  }
}

__global__ void rtable_kernel(long long Ns, const double* __restrict__ agrid, long long Na,
                              const unsigned char* __restrict__ in_ts, double dt, double* __restrict__ R) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= Ns * Na) return;
  const long long s = e / Na, a = e % Na;
  const double act = agrid[a];
  // where(done, -g(x) = -0.0, -(f + 0.5 |a|^2) dt)   environments.py:104-110
  R[e] = in_ts[s] ? -0.0 : -__dmul_rn(__dadd_rn(1.0, __dmul_rn(0.5, __dmul_rn(act, act))), dt);
}

int launch_tables(const double* state_grid, long long Ns, const double* action_grid, long long Na,
                  const unsigned char* in_ts, long long n_ts, double alpha, double sigma, double dt, double h_half,
                  double lb, double rb, long long sprime_begin, long long sprime_end, double* P, double* R,
                  int uniform_grid, double grid_step, cudaStream_t stream) {
  (void)lb; (void)rb;
  if (P && sprime_end > sprime_begin && gl_path(Ns, uniform_grid, grid_step, sigma, dt, h_half)) {
    // row classes (see tables_gl_kernel) and chunks of `steps` rows per class, both defined on the full grid so that a
    // slab reproduces the full tensor's entries bit for bit
    const long long cols = Ns * Na;
    const int Q = (cols & 3) == 0 ? 1 : ((cols & 1) == 0 ? 2 : 4);
    const long long rows_per_class = (Ns + Q - 1) / Q;
    const long long steps_cap = gl_anchor_steps(Q * grid_step / (sigma * sqrt(dt)));
    const long long n_chunks_full = (rows_per_class + steps_cap - 1) / steps_cap;
    const int steps = (int)((rows_per_class + n_chunks_full - 1) / n_chunks_full);
    const long long kc_lo = (sprime_begin >= Q ? (sprime_begin - (Q - 1)) / Q : 0) / steps;
    const long long kc_hi = ((sprime_end - 1) / Q) / steps;
    dim3 grid((unsigned)((cols + 3 + 127) / 128), (unsigned)((kc_hi - kc_lo + 1) * Q));
    tables_gl_kernel<<<grid, 128, 0, stream>>>(state_grid, Ns, action_grid, Na, in_ts, n_ts > 0 ? 1.0 / (double)n_ts : 0.0,
                                               alpha, sigma, dt, h_half, sprime_begin, sprime_end, P, Q, steps, kc_lo,
                                               make_gl_const(Q * grid_step, sigma, dt, h_half));
    note_kernel_launches(1);
  } else if (P && sprime_end > sprime_begin) {
    const long long nsp = sprime_end - sprime_begin;
    dim3 grid((unsigned)((Na + 127) / 128), (unsigned)Ns, (unsigned)((nsp + TABLE_TILE - 1) / TABLE_TILE));
    tables_kernel<<<grid, 128, 0, stream>>>(state_grid, Ns, action_grid, Na, in_ts, n_ts > 0 ? 1.0 / (double)n_ts : 0.0,
                                            alpha, sigma, dt, h_half, sprime_begin, sprime_end, P);
    note_kernel_launches(1);
  }
  if (R) {
    const long long n = Ns * Na;
    rtable_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(Ns, action_grid, Na, in_ts, dt, R);
    note_kernel_launches(1);
  }
  return (int)cudaGetLastError();
}

// colsum[s, a] += sum over the slab's next-states, in index order (deterministic)
__global__ void colsum_kernel(const double* __restrict__ P, long long n_sprime, long long cols, double* __restrict__ colsum) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  double a = colsum[c];
  for (long long sp = 0; sp < n_sprime; ++sp) a += P[sp * cols + c];
  colsum[c] = a;
}

int launch_tables_colsum(const double* P, long long n_sprime, long long Ns, long long Na, double* colsum,
                         cudaStream_t stream) {
  const long long cols = Ns * Na;
  colsum_kernel<<<(unsigned)((cols + 127) / 128), 128, 0, stream>>>(P, n_sprime, cols, colsum);
  note_kernel_launches(1);
  return (int)cudaGetLastError();
}

}  // namespace rlsde
