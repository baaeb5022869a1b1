/* fokl_b200.h -- C ABI of the B200-native FoKL.fit hot path (libfokl_b200.so).
 *
 * The reference (ESMS-Group-Public/FoKL-GPy) is pure Python and has no FFI boundary of its own; every
 * entry point below replaces a *stage* of `FoKL.fit` / its nested `gibbs` closure
 * (src/FoKL/FoKLRoutines.py, "FR").  The Python host (fokl-gpy_b200/FoKL/_engine.py) binds these
 * with ctypes; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success and a negative FOKL_E* code on failure; nothing throws
 *     across the ABI; fokl_last_error(ctx) returns a human-readable message for the last failure.
 *   - pointers documented "dev" are device pointers owned by the caller (e.g. torch tensors'
 *     data_ptr()); pointers documented "host" are plain host memory, read before the call returns.
 *   - work is enqueued on the ctx stream (given at creation) and is asynchronous unless stated; one ctx
 *     per (process, device, stream); a ctx is not thread-safe.
 *   - all floating point is IEEE float64; matrices are column-major unless stated.
 */
#ifndef FOKL_B200_H
#define FOKL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FOKL_ABI_VERSION 4

#define FOKL_OK 0
#define FOKL_EINVAL (-1)   /* bad argument                                  */
#define FOKL_ECUDA (-2)    /* CUDA runtime error (see fokl_last_error)      */
#define FOKL_ENOMEM (-3)   /* workspace allocation failed                   */
#define FOKL_ERANGE (-4)   /* inputs not normalised to [0, 1] (FR:590-591)  */
#define FOKL_ESTATE (-5)   /* call sequence error (e.g. phis not set)       */

#define FOKL_KERNEL_CUBIC 0      /* 'Cubic Splines'          (FR:834-836) */
#define FOKL_KERNEL_BERNOULLI 1  /* 'Bernoulli Polynomials'  (FR:841-843) */

#define FOKL_RNG_NONE 0      /* BIC / betahat only, no chain                                   */
#define FOKL_RNG_INJECTED 1  /* variates supplied by the caller (numpy legacy stream, parity)  */
#define FOKL_RNG_PHILOX 2    /* counter-based Philox4x32-10 on device (free-running)           */

typedef struct fokl_ctx fokl_ctx;

/* ---- context ------------------------------------------------------------------------------- */

int fokl_abi_version(void);

/* device: CUDA ordinal.  cuda_stream: the cudaStream_t all work is enqueued on; NULL is the CUDA legacy
 * default stream (PyTorch's default), never a private stream. */
int fokl_ctx_create(fokl_ctx **out, int device, void *cuda_stream);
int fokl_ctx_destroy(fokl_ctx *ctx);
const char *fokl_last_error(fokl_ctx *ctx);
/* blocks until all work enqueued on the ctx stream has finished; reports deferred range errors. */
int fokl_ctx_synchronize(fokl_ctx *ctx);
/* number of kernels this ctx has launched since creation (for bench.py's gpu_launches). */
int64_t fokl_launch_count(fokl_ctx *ctx);
/* SMs a batch of candidate models may plan its eigensolver clusters for (0 = the whole device).  A second context
 * whose batches run next to another context's work (the pipelined selection loop) is given the device minus the
 * other's share, so that the two together still fit in one wave. */
int fokl_ctx_set_sm_budget(fokl_ctx *ctx, int sms);
/* on != 0: the candidate stage of this context (fokl_candidates_eval, fokl_kill_loop, fokl_kill_scores) is enqueued on
 * a high-priority stream of the context, ordered after the context's stream on entry and before it on exit (same
 * semantics for the caller), so that its small, latency-bound kernels are dispatched ahead of the pending thread
 * blocks of a basis / Gram build that another context runs at the same time. */
int fokl_ctx_set_high_priority(fokl_ctx *ctx, int on);
/* make everything enqueued on `waiter` from now on wait until the eigensolver kernels of the most recent
 * fokl_candidates_eval on `src` have finished (no-op if there was none).  Used to start a basis / Gram build on a second
 * context only once the cluster launches of the candidate stage -- which need whole groups of free SMs -- are through. */
int fokl_ctx_wait_eig(fokl_ctx *waiter, fokl_ctx *src);

/* ---- basis tables: replaces getKernels.sp500()/bernoulli() output consumed at FR:1480-1482 ----
 * cubic:     tab (host) [n_orders][n_piece][4]  -- phis[s][k][piece] transposed to (s, piece, k)
 * bernoulli: tab (host) [n_orders][row_len]     -- row n holds its n + 2 monomial coefficients      */
int fokl_set_phis_cubic(fokl_ctx *ctx, const double *tab, int n_orders, int n_piece);
int fokl_set_phis_bernoulli(fokl_ctx *ctx, const double *tab, int n_orders, int row_len);

/* ---- K1: design-matrix columns, replaces the triple loop FR:1446-1485 (+ FR:570-589) -----------
 * x      dev  normalised inputs, column-major N x M, column k at x + k*ldx
 * terms  host C x M row-major; terms[j][k] = order of the basis function of input k in term j, 0 = absent
 *             (one row of `discmtx`, FR:1473)
 * Xnew   dev  output: column j written to Xnew + j*ld (N doubles each); ld % 2 == 0, Xnew 16B-aligned
 * X[i][j] = prod_{k: terms[j][k] != 0} phi_{terms[j][k]}(x[i][k]), multiplied in increasing k.     */
int fokl_basis_build(fokl_ctx *ctx, int kernel, const double *x, int64_t n, int64_t ldx, int m,
                     const int16_t *terms, int c, double *Xnew, int64_t ld);

/* K1, derivative form: the design-matrix columns of FoKL.bss_derivatives (FR:594-805; factor evaluation FR:770-781,
 * evaluate_basis d = 1, 2 at FR:837-847).
 * deriv     host C x M row-major, 0 / 1 / 2: derivative order of the factor of input k in term j (0 = plain factor)
 * divisors  host M x 3 row-major: divisors[k][e] = span_L[e] of FR:762-763 for input k ([k][0] is not read)
 * Column j = prod_k f_jk, f_jk = phi_{terms[j][k]}(X_ik) or its e-th derivative divided by divisors[k][e]; every
 * factor is evaluated at the twice-normalised input X of FR:584-586 (cubic) or at x itself (Bernoulli).             */
int fokl_basis_build_deriv(fokl_ctx *ctx, int kernel, const double *x, int64_t n, int64_t ldx, int m,
                           const int16_t *terms, const uint8_t *deriv, const double *divisors, int c,
                           double *Xnew, int64_t ld);

/* fill a column with ones (X[:, 0], FR:1436). */
int fokl_fill_ones(fokl_ctx *ctx, double *col, int64_t n);

/* ---- K2: Gram / projection update, replaces XtX = X'X, Xty = X'y (FR:1492-1494) ----------------
 * Computes only what is new when columns [p_old, p_old + c) were appended to X:
 *   block[(i) * c + j] = sum_n A_i[n] * X[n][p_old + j],  i = 0 .. p_old + c   (row-major (p+1) x c)
 * where A_i = column i of X for i < p_old + c and A_{p_old+c} = y.  Deterministic summation order.
 * Entries strictly below the diagonal of the symmetric X_new' X_new part (p_old + j < i < p_old + c) are optional:
 * 8 x 8 fragments lying entirely there are skipped and read back as 0; fokl_gram_scatter mirrors the upper triangle. */
int fokl_gram_update(fokl_ctx *ctx, const double *X, int64_t ld, int64_t n, int p_old, int c,
                     const double *y, double *block);

/* The same block for new columns that are NOT stored right behind the old ones: the new block occupies X columns
 * [new_col0, new_col0 + c), new_col0 >= p_old (it was built ahead of time -- while the previous substage's candidate
 * stage was still running -- above the columns that substage may yet delete); the output block keeps the layout above
 * ((p_old + c + 1) x c, logical row order old | new | y).  flags: FOKL_GRAM_CROSS_ONLY = only the (old | y) x new rows
 * (rows of the new x new part are left zero: an earlier call formed them).  A context with an SM budget
 * (fokl_ctx_set_sm_budget) sizes the grid for that many SMs. */
#define FOKL_GRAM_CROSS_ONLY 1
int fokl_gram_update_ex(fokl_ctx *ctx, const double *X, int64_t ld, int64_t n, int p_old, int c, int new_col0,
                        int flags, const double *y, double *block);
/* what the last fokl_gram_update(_ex) on this context launched (host record, for tests and tuning):
 * out (host, 9 values) = { pipeline (0 = cp.async ring, 1 = bulk-copy / mbarrier ring, 2 = tensor-map ring),
 * consumer warps, rows per slab (kb), ring stages, tiles, row splits, rows per split, staged-column slots per tile,
 * slot cap }.  FOKL_ESTATE if the context has not launched one yet. */
int fokl_gram_last_config(fokl_ctx *ctx, int64_t out[9]);

/* moments of y: out (dev, 3 doubles) = { n, sum y, sum y^2 } (dtd, FR:1374). */
int fokl_y_moments(fokl_ctx *ctx, const double *y, int64_t n, double *out);

/* scatter a (reduced) block into the symmetric master Gram G (dev, row-major ldg x ldg) and Xty (dev):
 * G[i][p_old+j] = G[p_old+j][i] = block[i][j]; Xty[p_old+j] = block[p_old+c][j]. */
int fokl_gram_scatter(fokl_ctx *ctx, const double *block, int p_old, int c, double *G, int64_t ldg,
                      double *Xty);

/* keep (host, ascending, p_new entries): G_out[a][b] = G[keep[a]][keep[b]], Xty_out[a] = Xty[keep[a]]. */
int fokl_gram_compact(fokl_ctx *ctx, const double *G, int64_t ldg, const double *Xty, const int32_t *keep,
                      int p_new, double *G_out, int64_t ldg_out, double *Xty_out);

/* move column keep[a] of X to position a (keep ascending, keep[a] >= a): the X <- xers step (FR:1695). */
int fokl_columns_compact(fokl_ctx *ctx, double *X, int64_t ld, int64_t n, const int32_t *keep, int p_new);

/* ---- K3/K4: per-candidate spectral factorisation, betahat, BIC, Gibbs chain ---------------------
 * replaces, per `gibbs` invocation: eigh (FR:1499), betahat (FR:1502-1504), the draw loop
 * (FR:1519-1548), BIC (FR:1551-1554) and the column statistics the selection loop derives from the
 * draws (FR:1656-1658, 1671).                                                                        */
typedef struct fokl_hypers {
    double a, b, atau, btau;   /* inverse-gamma hyper-parameters (FR:1304-1307)           */
    double sigsqd0, tausqd0;   /* chain start (FR:1371-1372)                              */
    double yty, sum_y;         /* data moments (global over all ranks)                    */
    int64_t n;                 /* number of data rows (global)                            */
    int32_t draws;             /* chain length D = burnin + draws (FR:1309)               */
    int32_t stat_from0;        /* ceil(D/2)      first row of the "mean0" window (FR:1658)*/
    int32_t stat_from1;        /* ceil(D/2 + 1)  first row of mean1/std1 window (FR:1656) */
    int32_t reserved;
} fokl_hypers;

/* Candidate c uses the p_c = set_offsets[c+1] - set_offsets[c] columns col_sets[set_offsets[c] ..] of G.
 * Packed output offsets (both sides compute them the same way):
 *   vec_off[c] = sum_{c' < c} p_c'          (betahat, lamb, stats/3)
 *   mat_off[c] = sum_{c' < c} p_c'^2        (Q, column-major p x p, ascending eigenvalues like eigh)
 *   betas for candidate c start at D * vec_off[c], row-major D x p_c; sigs/taus at D * c.
 * run_chain (host, n_cand flags or NULL = all): 0 -> only eig/betahat/ev for that candidate.
 * rng_mode FOKL_RNG_INJECTED: variates (dev) holds for candidate c, at D * (vec_off[c] + 2c), D rows of
 *   [z_0 .. z_{p-1}, g1, g2] = normal(p), standard_gamma(astar), standard_gamma(atau_star) in the
 *   order one reference `gibbs` call consumes them (FR:1527, 1541, 1547).
 * rng_mode FOKL_RNG_PHILOX: stream_ids (host, n_cand) select independent Philox streams of `seed`; every eigenvector
 *   is oriented so that its projection on X'y is non-negative (z_j *= sign(q_j . Xty)): the chain is then a function
 *   of the Gram alone, whatever sign the eigensolver happened to return (FR:1525-1528 leaves it to LAPACK).
 * sign_fix (dev, packed like betahat, or NULL): z_j is multiplied by sign_fix[j] (parity harness only:
 *   aligns eigenvector signs with another eigensolver).
 * Outputs (dev; any of betahat/lamb/Q/betas/sigs/taus/stats may be NULL):
 *   ev[c]        BIC (FR:1554), without the aic adjustment (FR:1654, host side)
 *   stats        per candidate 3 x p_c: row 0 mean over rows [stat_from1, D), row 1 std (ddof 0) over the
 *                same rows, row 2 mean over rows [stat_from0, D); NaN over an empty window (start >= D, D <= 3)
 *   info[c]      bit 0: bstar < 0 seen (FR:1538); bits 8..: Jacobi sweeps used                      */
int fokl_candidates_eval(fokl_ctx *ctx, const double *G, int64_t ldg, const double *Xty,
                         const int32_t *col_sets, const int32_t *set_offsets, int n_cand,
                         const fokl_hypers *hyp, const uint8_t *run_chain, int rng_mode, uint64_t seed,
                         const uint64_t *stream_ids, const double *variates, const double *sign_fix,
                         double *ev, double *betahat, double *lamb, double *Q, double *betas,
                         double *sigs, double *taus, double *stats, int32_t *info);

/* ---- chains of nested models (csrc/nested.cu) ------------------------------------------------------------------------
 * The accepted models of one kill loop (FR:1669-1690) are nested: each is its predecessor with one column removed, and
 * the selection loop needs, from the chain of each (FR:1690), only the posterior mean of the intercept (FR:1671).
 * fokl_secular_step carries a spectral decomposition from a model to the next: lam (dev, p ascending eigenvalues),
 * u (dev, p: the components of the p eigenvectors on the variable being removed) -> mu (dev, p - 1 ascending eigenvalues
 * of the compressed matrix) and zt (dev, (p - 1) x ldz row-major: row i = new eigenvector i in the old eigenbasis), so
 * that Q_new = zt Q (rows = eigenvectors) by a plain GEMM.  work: dev, 4 p doubles.  status (dev int, OR-ed, caller
 * zeroes it): 1 = two equal eigenvalues (the step is not valid: fall back to fokl_candidates_eval), 2 = non-finite input.
 * fokl_chain_icpt runs the eigenbasis draw loop (FR:1519-1548) of n_models models side by side from their
 * (lam, ct = Q'X'y, q0 = intercept components of the eigenvectors), packed at off[i] (dev int64) with widths p[i] (dev
 * int32), Philox streams stream_ids[i] (dev) -- the variates fokl_candidates_eval would use -- and returns
 * mean0[i] = mean over draws stat_from0 .. of the intercept's draw, info[i] = 1 if bstar < 0 was seen. */
int fokl_secular_step(fokl_ctx *ctx, const double *lam, const double *u, int p, double *mu, double *zt, int64_t ldz,
                      double *work, int32_t *status);
int fokl_chain_icpt(fokl_ctx *ctx, int n_models, const int32_t *p, const int64_t *off, const uint64_t *stream_ids,
                    const double *lam, const double *ct, const double *q0, const fokl_hypers *hyp, uint64_t seed,
                    double *mean0, int32_t *info);

/* ---- update fits: `fitupdate` / update=True (FR:1850-2583; entered from `fit` at FR:1365-1367) -------------------------
 * The draw loops of the three-case sampler gibbs_Xin_update (FR:2057-2430) in spectral coordinates (csrc/update_math.cuh):
 *   mode 1 (FR:2062-2147, first fit of an update model): pn = p, po = 0; lam_n = eigenvalues of X'X, c_n = Q'X'y,
 *          squerr = |y - X betahat|^2.  gam_n[d] = Q' betas[d].
 *   mode 2 (FR:2150-2264, same terms as the prior model): po = p, pn = 0; with Sigma_old^-1 = L L' and
 *          L^-1 X'X L^-T = V D V', T = L^-T V:  lam_o = D, c_o = T'X'y, m_o = T^-1 mu_old.  betas[d] = T gam_o[d].
 *          (One generalised eigendecomposition replaces the reference's eigh + inv per draw, FR:2197-2203: same
 *          conditional law at every draw, another square root of its covariance.)
 *   mode 3 (FR:2267-2426, new terms): lam_o, Q_o = eigh(Xo'Xo + Sigma_old^-1) (FR:2296), lam_n, Q_n = eigh(Xn'Xn)
 *          (FR:2312); c_o = Q_o'(Xo'y + Sigma_old^-1 mu_old), t_o = Q_o'Xo'y, m_o = Q_o'mu_old, c_n = Q_n'Xn'y,
 *          M = Q_o'Xo'Xn Q_n (po x pn row-major), Mt = M' (pn x po row-major), K = Q_o'Xo'Xo Q_o, W = Q_o'Sigma_old^-1 Q_o
 *          (po x po row-major).  betas[d] = [Q_o gam_o[d], Q_n gam_n[d]].
 * All arrays dev.  rng_mode FOKL_RNG_INJECTED: variates = draws rows of [z (po), z (pn), G1, G2] in the order the
 * reference consumes them; FOKL_RNG_PHILOX: stream `stream_id` of `seed`.  Outputs: gam_o (draws x po), gam_n
 * (draws x pn), sigs, taus, lik (draws each; ev = (mmtx + 1) log n - 2 max(lik), FR:2143 / 2257 / 2419, host side),
 * info (1 int): 1 if bstar < 0 was seen (FR:2128).                                                                  */
typedef struct fokl_update_model {
    int32_t mode, po, pn, draws;
    double a_star, atau_star;  /* gamma shapes (FR:2086-2087 / 2176-2177 / 2327-2328)            */
    double b, btau;            /* FR:1926-1929                                                  */
    double sigsqd0;            /* chain start (FR:1936); tausqd starts at 1 / sigsqd0 (FR:2067) */
    double yty, squerr;
    int64_t n;
} fokl_update_model;
int fokl_update_chain(fokl_ctx *ctx, const fokl_update_model *mdl, const double *lam_o, const double *c_o,
                      const double *t_o, const double *m_o, const double *lam_n, const double *c_n, const double *M,
                      const double *Mt, const double *K, const double *W, int rng_mode, uint64_t seed,
                      uint64_t stream_id, const double *variates, double *gam_o, double *gam_n, double *sigs,
                      double *taus, double *lik, int32_t *info);

/* BIC of every single-column deletion of one model, from ONE Cholesky factorisation of its Gram
 * (SSE_{-q} = SSE + betahat_q^2 / (A^-1)_qq): what the kill loop FR:1669-1690 asks of `gibbs` for all its
 * proposals at once.  cols (host, p entries, cols[0] = intercept) selects the model in G; props (host, k positions
 * into cols, each >= 1) the columns proposed for deletion.  ev (dev, k + 1): ev[j] = BIC without props[j],
 * ev[k] = BIC of the model itself (no aic adjustment).  info (dev, 1 int): 1 if the Gram is not numerically
 * positive definite (scores invalid: use fokl_candidates_eval instead). */
int fokl_kill_scores(fokl_ctx *ctx, const double *G, int64_t ldg, const double *Xty, const int32_t *cols, int p,
                     const int32_t *props, int k, const fokl_hypers *hyp, double *ev, int32_t *info);

/* The whole kill loop of one substage (FR:1666-1690) in one launch: sweep-operator inverse of the model's Gram, then
 * for every proposal in the reference's order the BIC of the model without it, accepting the first that lowers the
 * BIC and continuing from the next candidate against the reduced model (one O(p^2) reverse sweep per accepted kill).
 * cols (host, p, cols[0] = intercept): the model; cand_pos (host, vm): position in cols of candidate i (candidates in
 * ascending |mean| order, FR:1664); bv0 / bv1 (host, vm): |mean| and std/|mean| of each candidate (FR:1656-1658).
 * kp->icpt is the |mean intercept draw| the threshold test FR:1671 uses for the whole loop (the caller verifies it
 * against the accepted models' chains).  Outputs (dev): out_i (3 + 2 vm ints) = { accepted kills, proposals tested,
 * error flag (1 Gram not positive definite, 2 breakdown), candidate index of each accepted kill [vm], proposals tested
 * up to and including it [vm] }; out_ev (vm doubles) = BIC incl. aic adjustment after each accepted kill. */
typedef struct fokl_kill_params {
    double threshav, threshstda, threshstdb;   /* FR:1670-1671                                     */
    double icpt;                               /* |mean(beters[h0:, 0])|                           */
    double evmin;                              /* BIC (incl. aic adjustment) of the starting model */
    double aic_adj;                            /* (2 - ln n) if aic else 0, per model column       */
    int32_t start;                             /* first candidate index to consider                */
    int32_t reserved;
    /* Optional (both or neither; dev): the eigendecomposition of the model's Gram G[cols][cols] as fokl_candidates_eval
     * returns it (lamb ascending, Qt[k * p + i] = component i of eigenvector k).  The tableau the loop starts from is
     * then formed from it by the whole device instead of by p sequential pivots; an ill-conditioned model
     * (lamb[0] <= 1e-10 max diag) takes the sequential form regardless. */
    const double *lamb;
    const double *Qt;
} fokl_kill_params;
int fokl_kill_loop(fokl_ctx *ctx, const double *G, int64_t ldg, const double *Xty, const int32_t *cols, int p,
                   const int32_t *cand_pos, const double *bv0, const double *bv1, int vm, const fokl_hypers *hyp,
                   const fokl_kill_params *kp, int32_t *out_i, double *out_ev);

/* ---- checks / "next" rows ------------------------------------------------------------------- */

/* residual moments of an explicit model: out (dev, 2 doubles) = { sum r, sum r^2 },
 * r = y - X[:, cols] beta  (cols host, p entries, or NULL for the first p columns; beta dev, p).
 * The N-length form of FR:1551; used to refine / cross-check the Gram-only BIC. */
int fokl_residual_moments(fokl_ctx *ctx, const double *X, int64_t ld, int64_t n, int p,
                          const int32_t *cols, const double *beta, const double *y, double *out);

/* evaluate (FR:966-969): out[i][d] = sum_j X[i][j] * betas[d][j]; X column-major (ld), betas row-major
 * n_draws x p (dev), out row-major n x n_draws (dev). */
int fokl_predict_draws(fokl_ctx *ctx, const double *X, int64_t ld, int64_t n, int p, const double *betas,
                       int n_draws, double *out);

/* evaluate at training-set scale: with v[i][d] = sum_j X[i][j] * betas[d][j] (the bits of fokl_predict_draws),
 * mean_out[i] = np.mean(v[i]) and, unless rank_lo = rank_hi = -1 (mean only; lo_out / hi_out may be NULL),
 * lo_out[i] / hi_out[i] = np.sort(v[i])[rank_lo / rank_hi], bit for bit (NaN sorts last; only the sign of a zero may
 * differ).  X column-major (ld), betas row-major n_draws x p, outputs n doubles each (all dev).  The product is
 * formed in L2-sized row chunks and never written out: device scratch depends on n_draws, not on n. */
int fokl_predict_summary(fokl_ctx *ctx, const double *X, int64_t ld, int64_t n, int p, const double *betas,
                         int n_draws, int rank_lo, int rank_hi, double *mean_out, double *lo_out, double *hi_out);

/* bss_derivatives at training-set scale, one row chunk: rows [r0, r0 + rows) of x (dev, column-major, ldx, m inputs).
 * terms / deriv / divisors / c as fokl_basis_build_deriv (host); the chunk's c derivative columns are built with its
 * kernels into device scratch.  pairs (host, n_pairs x 5 int64): {column offset, width, betas offset, input, order - 1};
 * pair k's betas block is betas[offset .. + n_draws * width) (dev, row-major n_draws x width) and its values are
 * v[i][d] = sum_j W[i][offset + j] * b[d][j] with the FMA order of fokl_predict_draws (the same bits).  out (dev) gets
 * the C-order slice dy[r0 : r0 + rows] of bss_derivatives' dy: mean_only = 0: [rows][m][2][n_draws] of v;
 * mean_only = 1: [rows][m][2] of np.mean(v[i]) over the draws (the bits of fokl_predict_summary).  (input, order)
 * slots no pair names, and pairs of width 0, get 0.0.  Device scratch: 8 * c * rows bytes, plus (mean_only) at most
 * 32 MB of values; it does not depend on the rows outside the chunk.  A bad pointer, column range, betas offset, input,
 * order, repeated slot, n_draws or term list returns FOKL_EINVAL before anything is written to out; inputs outside
 * [0, 1] set the deferred FOKL_ERANGE flag (cubic). */
int fokl_deriv_summary(fokl_ctx *ctx, int kernel, const double *x, int64_t ldx, int m, int64_t r0, int64_t rows,
                       const int16_t *terms, const uint8_t *deriv, const double *divisors, int c,
                       const int64_t *pairs, int n_pairs, const double *betas, int n_draws, int mean_only,
                       double *out);

/* clean/_normalize on device (FR:377, 436-437): minmax_out (dev, 2*m) = per-column min, max of x
 * (column-major n x m, ldx); then fokl_normalize applies x = (x - min) / (max - min) in place with
 * minmax (host, 2*m), for any m >= 1. */
int fokl_column_minmax(fokl_ctx *ctx, const double *x, int64_t n, int64_t ldx, int m, double *minmax_out);
int fokl_normalize(fokl_ctx *ctx, double *x, int64_t n, int64_t ldx, int m, const double *minmax);

/* train split of clean (FR:532-542, `inputs[trainlog, :]`, `data[trainlog]`): the rows i < n with keep[i] != 0
 * (dev, n bytes) of x (dev, column-major [m][ldx]) and y (dev, n) are written in ascending row order to x_out
 * (dev, [m][ldx_out]) and y_out (dev, ldx_out); rows [*n_out, ldx_out) of every output column and of y_out are set to
 * 0.0.  *n_out (host) = kept row count.  The outputs must not overlap the inputs.  Synchronises the context's stream
 * once (the kept count).  A null pointer, n < 1, m < 1, ldx < n or ldx_out below the kept count returns FOKL_EINVAL
 * before anything is written to the outputs. */
int fokl_rows_compact(fokl_ctx *ctx, const double *x, const double *y, int64_t n, int64_t ldx, int m,
                      const uint8_t *keep, double *x_out, double *y_out, int64_t ldx_out, int64_t *n_out);

/* train split of clean (FR:509-530 `generate_trainlog(train, n)`), bit for bit with numpy's legacy RandomState: from
 * the MT19937 state key[624] (host) / pos (0 .. 624), with l_log = max(int(n * train), 2) computed by the caller,
 * keep (dev, n bytes) = 1 for the rows the reference's mask keeps and 0 elsewhere; key_out[624] / *pos_out (host) = the
 * state after the last word the reference consumes (np.random.set_state(('MT19937', key_out, *pos_out, has_gauss,
 * cached_gaussian)) leaves numpy where generate_trainlog would); *words_out = words consumed.  Synchronises the
 * context's stream.  Device memory: about n / 8 + 12 n bytes plus a 41 MB word window, allocated and freed within the
 * call.  A null pointer, pos outside [0, 624] or l_log outside [2, n], n >= 2^31 returns FOKL_EINVAL before anything
 * is written to the outputs. */
int fokl_trainlog(fokl_ctx *ctx, const uint32_t *key, int pos, int64_t n, int64_t l_log, uint8_t *keep,
                  uint32_t *key_out, int *pos_out, int64_t *words_out);

#ifdef __cplusplus
}
#endif
#endif /* FOKL_B200_H */
