// Pivoted stage-wise KKT solve: the QP's last resort when the Riccati recursion cannot certify.
//
// Why it exists (DESIGN.md section 2.3, profiles/r2_h100_order1_analysis.md): with the order-1 (Euler) model every
// transition frequency gives |eig A_t| > 1, at H = 100 the open-loop transition has norm 4e13 and neither the
// cost-to-go (entries ~1e27) nor any rollout through the dynamics keeps digits.  The reference's solver (cvxpy -> OSQP,
// optimize.py:59; our CPU oracle: a sparse LU of the KKT matrix) never propagates through prod A_t, because states AND
// costates are unknowns of one banded system.  This is the device equivalent: the KKT system of the working set,
//   stationarity  2 R_t (u_t - ub_t) + B_t^T lam_{t+1} = 0     (free controls; pinned ones: u_t[i] = bound)
//   dynamics      x_{t+1} - A_t x_t - B_t u_t = D_t
//   costate       lam_t - 2 Q_t x_t - A_t^T lam_{t+1} = -2 Q_t r_t        (lam_H = 2 Qf (x_H - r_H))
// ordered stage by stage -- block s holds [u_{s-1} | x_s | lam_s], W = 2N + M unknowns -- is almost block diagonal and
// is eliminated block column by block column with ROW PARTIAL PIVOTING over every row that touches the column: the N
// rows carried over from the previous block, the block's own stationarity and costate rows and the next stage's
// dynamics rows (3N + M candidates, two block columns + the right-hand side wide).  Pivot rows go to a per-warp array
// in global memory (H W (2W + 2) doubles: 2.4 MB for the transmon at H = 100), back-substitution runs block by block
// from the end, and the multipliers of the box constraints come from the solve's own costates, so they carry the
// accuracy of the solve (1e-7 at worst on the captured H = 100 problems, tools/analysis/abd_full.py) instead of the
// noise of an adjoint sweep through the unstable dynamics.
//
// Working set: a primal-dual interior-point method whose every iteration is one such solve (kkt_active_set below).
//
// One warp per member as everywhere else; the elimination window (3N + M rows) lives in the same per-warp global
// array and is served by L1/L2.  This path is cold for every configuration that the Riccati path certifies.
#pragma once

// measurement aids (build variants): interior-point iteration cap, polish rounds per pass
#ifndef M4Q_IPM_ITERS
#define M4Q_IPM_ITERS 80
#endif
#ifndef M4Q_KKT_POLISH
#define M4Q_KKT_POLISH 16
#endif

namespace m4q {

template <class CF> struct Kkt {
    static constexpr int N = CF::N, M = CF::M, C = CF::C;
    static constexpr int W = 2 * N + M;        // unknowns per block: u_{s-1} | x_s | lam_s
    static constexpr int ROWS = W + N;         // candidate rows of a block column
    static constexpr int RHS = 2 * W;          // column of the right-hand side
    static constexpr int LD = 2 * W + 2;       // row length (even)
    static constexpr int CH = cdiv(LD, 32);    // column chunks of a row per lane
    static constexpr int CR = cdiv(ROWS, 32);  // rows of a column per lane
    static constexpr int CW = cdiv(W, 32);     // unknowns of a block per lane
    // window | pivot rows of every block | the last solution [H + 2][W] (iterative refinement)
    __host__ __device__ static constexpr long long doubles(int H) {
        return (long long)(ROWS + (long long)H * W) * LD + (long long)(H + 2) * W;
    }
};

// realified entry (k, j) of a complex C x C block stored with row stride CA: [[Re, -Im], [Im, Re]]
template <class CF> __device__ __forceinline__ double realified(const double2 *At, int k, int j) {
    constexpr int C = CF::C;
    const double2 a = At[(k % C) * Rec<CF>::CA + (j % C)];
    return ((k < C) == (j < C)) ? a.x : (k >= C ? a.y : -a.y);
}

// One solve of the KKT system.  Out: Uo (slab), Xo (workspace), the gradient of the objective w.r.t. every control in
// slab.kk (= the multipliers on pinned controls, ~0 on free ones).
//   sigmu < 0:  working-set mode: controls with slab.mask != 0 are pinned to their bound.
//               refine: the right-hand side is the residual of the previous solution (kept in the workspace) and the
//               result is added to it -- one step of iterative refinement, a second elimination with the same pivots.
//   sigmu >= 0: interior-point mode: every control is free and carries the barrier terms of the iterate
//               (u, z_lo, z_hi) = (slab.z, slab.y, slab.hl):  (2 R + Sigma) u+ + B^T lam = 2 R ub + Sigma u +
//               sigma mu (1 / s_lo - 1 / s_hi),  Sigma = z_lo / s_lo + z_hi / s_hi,  s_lo = u - lo,  s_hi = hi - u.
// Returns false if a pivot vanished or the solution is not finite.
template <class CF, bool FUSED>
__device__ __noinline__ bool kkt_solve(SlabRef sr, const QPData &qp_in, double *kkt, int lane, double sigmu, bool refine) {
    using K_ = Kkt<CF>;
    using R_ = Rec<CF>;
    constexpr int N = CF::N, M = CF::M, W = K_::W, LD = K_::LD, CH = K_::CH, CR = K_::CR, CW = K_::CW, RHS = K_::RHS;
    const Slab<CF> s = slab_view<CF>(sr);
    const QPData qp = localize<FUSED>(qp_in);
    const int H = sr.H;
    double *win = kkt;                         // [ROWS][LD] elimination window
    double *Ust = kkt + K_::ROWS * LD;         // [H][W][LD] pivot rows
    double *zst = Ust + (size_t)H * W * LD;    // [H + 2][W] last solution, block s at s * W (blocks 0 and H + 1: zeros)
    const bool ipm = sigmu >= 0.0;
    bool ok = true;
    if (!refine) {
#pragma unroll 1
        for (int e = lane; e < W; e += 32) {
            zst[e] = 0.0;
            zst[(H + 1) * W + e] = 0.0;
        }
    }

    // rows of block s (1-based): fills window rows row0.. with stat_s, cos_s and (s < H) dyn_{s+1}; columns of block s
    // at 0, of block s+1 at W
    auto fill_row = [&](int row, int kind, int s_, int k) {
        // kind 0: stat (control k of stage s_-1), 1: cos (state k of stage s_), 2: dyn_{s_+1} (state k), 3: dyn_1
        double *wr = win + row * LD;
        const int t = s_ - 1;
        const double *rec_t = ws_rec<CF>(sr, t < 0 ? 0 : t);
        const double *rec_s = ws_rec<CF>(sr, s_ < H ? s_ : H - 1);
#pragma unroll
        for (int cc = 0; cc < CH; ++cc) {
            const int c = lane + 32 * cc;
            if (c >= LD) continue;
            double v = 0.0;
            if (kind == 0) {
                const int mk = ipm ? 0 : s.mask[t * M + k];
                if (mk) {
                    if (c == k) v = 1.0;
                    else if (c == RHS) v = mk == 1 ? box_lo(s, qp.sat, t, k) : box_hi(s, qp.sat, t, k);
                } else {
                    if (c < M) v = 2.0 * qp.R[t * qp.r_stride + k * M + c];
                    else if (c >= M + N && c < W) v = rec_t[R_::B + R_::pair(k, c - M - N)];
                    else if (c == RHS) v = 2.0 * qp.Rub[t * M + k];
                    if (ipm && (c == k || c == RHS)) {
                        const double u = s.z[t * M + k];
                        const double isl = 1.0 / fmax(u - box_lo(s, qp.sat, t, k), 1e-300);
                        const double isu = 1.0 / fmax(box_hi(s, qp.sat, t, k) - u, 1e-300);
                        const double sig = s.y[t * M + k] * isl + s.hl[t * M + k] * isu;
                        v += c == k ? sig : fma(sig, u, sigmu * (isl - isu));
                    }
                }
            } else if (kind == 1) {
                const double *Qs = s_ == H ? qp.Qf : qp.Q + s_ * qp.q_stride;
                if (c >= M && c < M + N) v = -2.0 * Qs[k * N + (c - M)];
                else if (c >= M + N && c < W) v = (c - M - N == k) ? 1.0 : 0.0;
                else if (c >= W + M + N && c < 2 * W) {
                    if (s_ < H) v = -realified<CF>(reinterpret_cast<const double2 *>(rec_s + R_::AT), c - W - M - N, k);
                } else if (c == RHS) v = -2.0 * (s_ == H ? qp.qlinf[k] : qp.qlin[s_ * N + k]);
            } else if (kind == 2) {
                if (c >= M && c < M + N) v = -realified<CF>(reinterpret_cast<const double2 *>(rec_s + R_::AT), k, c - M);
                else if (c >= W && c < W + M) v = -rec_s[R_::B + R_::pair(c - W, k)];
                else if (c == W + M + k) v = 1.0;
                else if (c == RHS) v = rec_s[R_::D + k];
            } else {
                if (c < M) v = -rec_t[R_::B + R_::pair(c, k)];
                else if (c == M + k) v = 1.0;
                else if (c == RHS) v = rec_t[R_::D + k];   // + (A_0 x_0)[k], added by the caller
            }
            wr[c] = v;
        }
        if (refine) {
            // right-hand side -> residual of the previous solution: b - K z, z = [block s_ | block s_ + 1]
            double part = 0.0;
#pragma unroll
            for (int cc = 0; cc < CH; ++cc) {
                const int c = lane + 32 * cc;
                if (c < 2 * W) part = fma(wr[c], zst[(size_t)s_ * W + c], part);
            }
            part = warp_sum(part);
            if (lane == RHS % 32) wr[RHS] -= part;
        }
    };

    // ---- block 1: the "carried" rows are the dynamics of stage 0 (x_0 is data)
    {
        const double2 *A0 = reinterpret_cast<const double2 *>(ws_rec<CF>(sr, 0) + R_::AT);
        double ax = 0.0;
        if (lane < N)
            for (int j = 0; j < N; ++j) ax = fma(realified<CF>(A0, lane, j), s.x0[j], ax);
#pragma unroll 1
        for (int k = 0; k < N; ++k) {
            fill_row(k, 3, 1, k);
            const double axk = __shfl_sync(FULL, ax, k);
            __syncwarp();
            if (lane == 0) win[k * LD + RHS] += axk;
        }
    }
    __syncwarp();

#pragma unroll 1
    for (int sblk = 1; sblk <= H; ++sblk) {
        const int nrows = sblk < H ? K_::ROWS : W;
#pragma unroll 1
        for (int i = 0; i < M; ++i) fill_row(N + i, 0, sblk, i);
#pragma unroll 1
        for (int k = 0; k < N; ++k) fill_row(N + M + k, 1, sblk, k);
        if (sblk < H) {
#pragma unroll 1
            for (int k = 0; k < N; ++k) fill_row(W + k, 2, sblk, k);
        }
        __syncwarp();
        double *Us = Ust + (size_t)(sblk - 1) * W * LD;
        // ---- eliminate the W columns of this block
#pragma unroll 1
        for (int k = 0; k < W; ++k) {
            double a[CR];
            double best = -1.0;
            int bi = 0;
#pragma unroll
            for (int q = 0; q < CR; ++q) {
                const int r = k + lane + 32 * q;
                a[q] = r < nrows ? win[r * LD + k] : 0.0;
                const double av = r < nrows ? fabs(a[q]) : -1.0;
                if (av > best) {
                    best = av;
                    bi = lane + 32 * q;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ob = __shfl_xor_sync(FULL, best, o);
                const int oi = __shfl_xor_sync(FULL, bi, o);
                if (ob > best || (ob == best && oi < bi)) {
                    best = ob;
                    bi = oi;
                }
            }
            if (!(best > 0.0) || !isfinite(best)) ok = false;
            const int prow = k + bi;
            // pivot row -> registers and the pivot-row store; what sat in row k moves to the pivot's place
            double pr[CH];
#pragma unroll
            for (int cc = 0; cc < CH; ++cc) {
                const int c = lane + 32 * cc;
                pr[cc] = c < LD ? win[prow * LD + c] : 0.0;
            }
            if (bi != 0) {
#pragma unroll
                for (int cc = 0; cc < CH; ++cc) {
                    const int c = lane + 32 * cc;
                    if (c < LD) win[prow * LD + c] = win[k * LD + c];
                }
            }
#pragma unroll
            for (int cc = 0; cc < CH; ++cc) {
                const int c = lane + 32 * cc;
                if (c < LD) Us[k * LD + c] = pr[cc];
            }
            double akk = __shfl_sync(FULL, a[0], 0);
            double pv = 0.0;
#pragma unroll
            for (int q = 0; q < CR; ++q) {
                const double cand = __shfl_sync(FULL, a[q], bi & 31);
                if ((bi >> 5) == q) pv = cand;
            }
            if (bi != 0 && lane == (bi & 31)) {
#pragma unroll
                for (int q = 0; q < CR; ++q)
                    if ((bi >> 5) == q) a[q] = akk;
            }
            const double ipv = 1.0 / pv;
            __syncwarp();
            // rank-1 update of the rows below, RB rows per trip so that their loads are in flight together (the window
            // is served by L1 / L2: a row at a time is one memory round trip per row); rows whose entry in column k is
            // zero are skipped (warp-uniform test)
            constexpr int RB = 8;
#pragma unroll 1
            for (int j0 = 1; k + j0 < nrows; j0 += RB) {
                double lj[RB], v[RB][CH];
#pragma unroll
                for (int b = 0; b < RB; ++b) {
                    const int j = j0 + b;
                    double cand = 0.0;
#pragma unroll
                    for (int q = 0; q < CR; ++q) {
                        const double cq = __shfl_sync(FULL, a[q], j & 31);
                        if ((j >> 5) == q) cand = cq;
                    }
                    lj[b] = (k + j < nrows) ? cand * ipv : 0.0;
                }
#pragma unroll
                for (int b = 0; b < RB; ++b) {
                    const double *wr = win + (k + j0 + b) * LD;
#pragma unroll
                    for (int cc = 0; cc < CH; ++cc) {
                        const int c = lane + 32 * cc;
                        v[b][cc] = (lj[b] != 0.0 && c > k && c < LD - 1) ? wr[c] : 0.0;
                    }
                }
#pragma unroll
                for (int b = 0; b < RB; ++b) {
                    double *wr = win + (k + j0 + b) * LD;
#pragma unroll
                    for (int cc = 0; cc < CH; ++cc) {
                        const int c = lane + 32 * cc;
                        if (lj[b] != 0.0 && c > k && c < LD - 1) wr[c] = fma(-lj[b], pr[cc], v[b][cc]);
                    }
                }
            }
            __syncwarp();
        }
        // ---- carry: rows W.., columns of block s+1 and the right-hand side -> rows 0.., columns of the next block
        if (sblk < H) {
#pragma unroll 1
            for (int i = 0; i < N; ++i) {
                double v[CH];
#pragma unroll
                for (int cc = 0; cc < CH; ++cc) {
                    const int c = lane + 32 * cc;
                    v[cc] = 0.0;
                    if (c < W) v[cc] = win[(W + i) * LD + W + c];
                    else if (c == RHS) v[cc] = win[(W + i) * LD + RHS];
                }
#pragma unroll
                for (int cc = 0; cc < CH; ++cc) {
                    const int c = lane + 32 * cc;
                    if (c < LD) win[i * LD + c] = v[cc];
                }
            }
            __syncwarp();
        }
    }

    // ---- back-substitution, block by block from the end; z of the next block stays in registers
    double zn[CW];
#pragma unroll
    for (int q = 0; q < CW; ++q) zn[q] = 0.0;
    double *Xo = ws_Xo<CF>(sr);
    double *zb = s.scr;   // W doubles of scratch (the factor scratch is dead here)
    bool finite = true;
#pragma unroll 1
    for (int sblk = H; sblk >= 1; --sblk) {
        const double *Us = Ust + (size_t)(sblk - 1) * W * LD;
        double b[CW];
#pragma unroll
        for (int q = 0; q < CW; ++q) {
            const int r = lane + 32 * q;
            b[q] = r < W ? Us[r * LD + RHS] : 0.0;
        }
        if (sblk < H) {
#pragma unroll 1
            for (int c = 0; c < W; ++c) {
                double zc = 0.0;
#pragma unroll
                for (int q = 0; q < CW; ++q) {
                    const double cand = __shfl_sync(FULL, zn[q], c & 31);
                    if ((c >> 5) == q) zc = cand;
                }
#pragma unroll
                for (int q = 0; q < CW; ++q) {
                    const int r = lane + 32 * q;
                    if (r < W) b[q] = fma(-Us[r * LD + W + c], zc, b[q]);
                }
            }
        }
#pragma unroll 1
        for (int k = W - 1; k >= 0; --k) {
            double zk = 0.0;
#pragma unroll
            for (int q = 0; q < CW; ++q) {
                const int r = lane + 32 * q;
                double cand = (r == k) ? b[q] / Us[k * LD + k] : 0.0;
                if (r == k) b[q] = cand;
                cand = __shfl_sync(FULL, cand, k & 31);
                if ((k >> 5) == q) zk = cand;
            }
#pragma unroll
            for (int q = 0; q < CW; ++q) {
                const int r = lane + 32 * q;
                if (r < k) b[q] = fma(-Us[r * LD + k], zk, b[q]);
            }
        }
#pragma unroll
        for (int q = 0; q < CW; ++q) {
            zn[q] = b[q];
            const int r = lane + 32 * q;
            if (r < W) {
                const double full = refine ? zst[(size_t)sblk * W + r] + b[q] : b[q];
                zst[(size_t)sblk * W + r] = full;
                zb[r] = full;
                finite &= isfinite(full) != 0;
            }
        }
        __syncwarp();
        // unpack: controls, state, and the gradient 2 R (u - ub) + B^T lam of stage t = s - 1
        const int t = sblk - 1;
        const double *rec = ws_rec<CF>(sr, t);
        if (lane < N) Xo[sblk * N + lane] = zb[M + lane];
        double g[M];
#pragma unroll
        for (int i = 0; i < M; ++i) g[i] = lane < N ? rec[R_::B + R_::pair(i, lane)] * zb[M + N + lane] : 0.0;
        warp_sum_vec<M>(g, lane);
        if (lane == 0) {
            const double *Rt = qp.R + t * qp.r_stride;
#pragma unroll
            for (int i = 0; i < M; ++i) {
                const int mk = ipm ? 0 : s.mask[t * M + i];
                const double u = mk == 1 ? box_lo(s, qp.sat, t, i) : (mk == 2 ? box_hi(s, qp.sat, t, i) : zb[i]);
                s.Uo[t * M + i] = u;
            }
#pragma unroll
            for (int i = 0; i < M; ++i) {
                double gi = g[i];
#pragma unroll
                for (int j = 0; j < M; ++j) gi = fma(2.0 * Rt[i * M + j], s.Uo[t * M + j] - qp.ub[t * M + j], gi);
                s.kk[t * M + i] = gi;
            }
        }
        __syncwarp();
    }
    if (lane < N) Xo[lane] = s.x0[lane];
    __syncwarp();
    return ok && !__any_sync(FULL, !finite);
}

// The QP on top of kkt_solve: a primal-dual interior-point method finds the working set, an active-set polish makes
// the answer exact.
//   * Interior point (box constraints only, so the barrier terms are a diagonal shift of R and every iteration is ONE
//     KKT solve with all controls free): iterate (u, z_lo, z_hi) strictly inside, centring sigma = 0.1, fraction to the
//     boundary 0.995, until the complementarity mu is below 1e-8 (1e-11 in a second pass if needed).  9..17 solves on every captured H = 100 problem
//     (tools/analysis/ipm_proto.py), including those on which primal-dual active-set rounds from any start cycle and the
//     textbook primal method needs hundreds of solves -- unconstrained optima of these QPs lie ten box widths outside.
//   * Polish: working set = bounds whose slack is smaller than their multiplier; primal-dual rounds from there (one or
//     two on the captured problems), each solve followed by one step of iterative refinement (accuracy 1e-7 -> 1e-10).
// Returns 0 (KKT point found; z, y set for the next warm start), 2 (not settled) or 3 (singular / non-finite).
template <class CF, bool FUSED>
__device__ __noinline__ int kkt_active_set(SlabRef sr, const QPData &qp_in, const QPSet &set, int lane, Counters &cnt) {
    constexpr int M = CF::M;
    const Slab<CF> s = slab_view<CF>(sr);
    const QPData qp = localize<FUSED>(qp_in);
    const int HM = sr.H * M;
    // set.kkt is the array of all resident warps' workspaces; this warp's slice follows the launch geometry
    double *kkt = set.kkt + (size_t)(blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * Kkt<CF>::doubles(sr.H);
    // ---- interior point: u in slab.z, z_lo in slab.y, z_hi in slab.hl
#pragma unroll 1
    for (int e = lane; e < HM; e += 32) {
        const int t = e / M, i = e % M;
        s.z[e] = 0.5 * (box_lo(s, qp.sat, t, i) + box_hi(s, qp.sat, t, i));
        s.y[e] = 1.0;
        s.hl[e] = 1.0;
    }
    __syncwarp();
    constexpr double SIGMA = 0.1, TAU = 0.995;
    // two passes: the working set is read off at mu = 1e-8 (the same set as at 1e-11 on all but the odd problem, four
    // solves earlier); if the polish does not settle from there the iteration carries on to 1e-11 and it is tried again
    bool found = false;
    int it = 0;
#pragma unroll 1
    for (int pass = 0; pass < 2 && !found; ++pass) {
    const double mu_stop = pass == 0 ? 1e-8 : 1e-11;
#pragma unroll 1
    for (; it < M4Q_IPM_ITERS; ++it) {
        double comp = 0.0;
#pragma unroll 1
        for (int e = lane; e < HM; e += 32) {
            const int t = e / M, i = e % M;
            if (!(box_hi(s, qp.sat, t, i) > box_lo(s, qp.sat, t, i))) continue;   // pinned: see below
            const double u = s.z[e];
            comp += (u - box_lo(s, qp.sat, t, i)) * s.y[e] + (box_hi(s, qp.sat, t, i) - u) * s.hl[e];
        }
        const double mu = warp_sum(comp) / (2.0 * HM);
        if (!(mu >= mu_stop)) break;
        cnt.kkt++;
        if (!kkt_solve<CF, FUSED>(sr, qp_in, kkt, lane, SIGMA * mu, false)) return 3;
        // step lengths: primal (slacks) and dual (multipliers) stay positive
        // A zero-width box (|u_0 - u_prev| <= 0, or u_prev = sat + du) has no interior: its control stays at the box,
        // where the solve's barrier diagonal (1e300) pins it, and its multipliers stay 1 so that the working set below
        // holds it on its bound.  Its zero slacks would otherwise stop the primal steps and turn mu into NaN.
        double ap = 1.0, ad = 1.0;
#pragma unroll 1
        for (int e = lane; e < HM; e += 32) {
            const int t = e / M, i = e % M;
            if (!(box_hi(s, qp.sat, t, i) > box_lo(s, qp.sat, t, i))) continue;
            const double u = s.z[e], du = s.Uo[e] - u;
            const double sl = u - box_lo(s, qp.sat, t, i), su = box_hi(s, qp.sat, t, i) - u;
            const double zl = s.y[e], zu = s.hl[e];
            const double dzl = SIGMA * mu / sl - zl - zl / sl * du, dzu = SIGMA * mu / su - zu + zu / su * du;
            if (du < 0.0) ap = fmin(ap, -TAU * sl / du);
            if (du > 0.0) ap = fmin(ap, TAU * su / du);
            if (dzl < 0.0) ad = fmin(ad, -TAU * zl / dzl);
            if (dzu < 0.0) ad = fmin(ad, -TAU * zu / dzu);
        }
        ap = -warp_max(-ap);
        ad = -warp_max(-ad);
#pragma unroll 1
        for (int e = lane; e < HM; e += 32) {
            const int t = e / M, i = e % M;
            if (!(box_hi(s, qp.sat, t, i) > box_lo(s, qp.sat, t, i))) continue;
            const double u = s.z[e], du = s.Uo[e] - u;
            const double sl = u - box_lo(s, qp.sat, t, i), su = box_hi(s, qp.sat, t, i) - u;
            const double zl = s.y[e], zu = s.hl[e];
            const double dzl = SIGMA * mu / sl - zl - zl / sl * du, dzu = SIGMA * mu / su - zu + zu / su * du;
            s.z[e] = fma(ap, du, u);
            s.y[e] = fma(ad, dzl, zl);
            s.hl[e] = fma(ad, dzu, zu);
        }
        __syncwarp();
    }
    // ---- working set from the interior-point estimate, then primal-dual rounds with refined solves
#pragma unroll 1
    for (int e = lane; e < HM; e += 32) {
        const int t = e / M, i = e % M;
        const double u = s.z[e];
        s.mask[e] = (u - box_lo(s, qp.sat, t, i) < s.y[e]) ? 1 : ((box_hi(s, qp.sat, t, i) - u < s.hl[e]) ? 2 : 0);
        s.flips[e] = 0;
    }
    __syncwarp();
#pragma unroll 1
    for (int round = 0; round < M4Q_KKT_POLISH && !found; ++round) {
        cnt.kkt += 2;
        if (!kkt_solve<CF, FUSED>(sr, qp_in, kkt, lane, -1.0, false)) return 3;
        if (!kkt_solve<CF, FUSED>(sr, qp_in, kkt, lane, -1.0, true)) return 3;
        double gmax = 0.0;
#pragma unroll 1
        for (int e = lane; e < HM; e += 32) gmax = fmax(gmax, fabs(s.kk[e]));
        const double gs = fmax(1.0, warp_max(gmax));
        bool changed = false;
#pragma unroll 1
        for (int e = lane; e < HM; e += 32) {
            const int t = e / M, i = e % M;
            const int mk = s.mask[e];
            const double u = s.Uo[e], g = s.kk[e];
            int nm = mk;
            if (mk == 0) {
                if (u < box_lo(s, qp.sat, t, i) - 1e-12) nm = 1;
                else if (u > box_hi(s, qp.sat, t, i) + 1e-12) nm = 2;
            } else {
                const double gn = mk == 1 ? -g : g;   // > 0: the multiplier has the wrong sign
                if (gn > 1e-10 * gs) {
                    const int fl = s.flips[e];
                    if (fl < 2 || gn > 1e-5 * gs) {
                        nm = 0;
                        s.flips[e] = fl + 1;
                    }
                }
            }
            if (nm != mk) {
                s.mask[e] = nm;
                changed = true;
            }
        }
        __syncwarp();
        found = !__any_sync(FULL, changed);
    }
    }   // passes
    if (!found) return 2;
    const double inv_rho = 1.0 / set.rho;
#pragma unroll 1
    for (int e = lane; e < HM; e += 32) {
        const int t = e / M, i = e % M;
        s.z[e] = fmin(fmax(s.Uo[e], box_lo(s, qp.sat, t, i)), box_hi(s, qp.sat, t, i));
        s.Uo[e] = s.z[e];
        s.y[e] = s.mask[e] ? -s.kk[e] * inv_rho : 0.0;
    }
    __syncwarp();
    return 0;
}

}   // namespace m4q
