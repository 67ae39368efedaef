// Warp-level building blocks of the MPC hot path (sm_100a).  One warp owns one ensemble member.  Its Riccati scratch,
// control trajectories and staging rings live in a warp-private slab of shared memory; the horizon-length data
// (stage records, state trajectories) live in an L2-resident workspace and are streamed through the slab with
// cp.async; the model blocks / costs are CTA-shared and read-only.  DESIGN.md section 2 has the full picture.
//
// Reference semantics restated here (paths relative to the reference repository):
//   linearize      mpc4quantum/linearize.py:37-70   (A_t = sum_k phi_k(u_t) * block_k, formed once per stage)
//   QP             mpc4quantum/optimize.py:12-60    (warm active set / ADMM on the control box, Riccati inner solve
//                                                     on the fp64 tensor cores, KKT certificate)
//   line search    mpc4quantum/mpc.py:101-125       (time-major metric paired with state-major vectors)
//   plant          mpc4quantum/experiment.py:202-212 + mpc.py:256-260 (expm conjugation per segment)
//   lift / proj    mpc4quantum/experiment.py:29-37, 225-235, 248-306 (and 357-388 for gate synthesis, in m4q_kernels.cu)
//   exact_stage    extension (SURVEY 8f rank 1): expm of the generator + Frechet derivative applied to x_t, per stage
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

namespace m4q {

constexpr unsigned FULL = 0xffffffffu;
constexpr int MAXBLK = 16;   // max monomial blocks (p + 1)

__host__ __device__ constexpr int cdiv(int a, int b) { return (a + b - 1) / b; }
__host__ __device__ constexpr int rup(int a, int b) { return cdiv(a, b) * b; }
__host__ __device__ constexpr int cmax(int a, int b) { return a > b ? a : b; }

// ---------------------------------------------------------------------------------------------------------
// Compile-time configuration for a (complex state dim, control dim) pair.
// The two dense products of a Riccati stage run on the fp64 tensor cores (mma.sync m8n8k4, "DMMA"):
// W^T = G^T P stays in the DMMA accumulators and feeds the second product T = W^T G straight from registers.  That
// works without a single shuffle because the contraction index of a k-step is free to be permuted: step (kt, e)
// contracts over k = 8 kt + 2 c4 + e, which is exactly the column the accumulator fragment of lane (g8, c4) holds.
// Operand rows are then 2 LD apart between neighbouring c4, so conflict-free fragment loads want LD = 2 or 6 (mod 8).
// MAXW: most warps (members) a CTA is ever launched with; it fixes the register budget (__launch_bounds__).
// ---------------------------------------------------------------------------------------------------------
__host__ __device__ constexpr int next_mod(int x, int r, int m) { return x + ((r - x % m) % m + m) % m; }
__host__ __device__ constexpr int cmin(int a, int b) { return a < b ? a : b; }

#ifndef M4Q_MAXW_4
#define M4Q_MAXW_4 32
#endif
// C = 4: 32 warps x 64 registers (+18 % on the qubit, spills and all); C = 16: 8 x 255 (the factor and sweeps of
// N = 32 do not fit 128 registers); else 16 x 128
template <int C_, int M_> struct Tiles { static constexpr int MAXW = C_ == 4 ? M4Q_MAXW_4 : C_ == 16 ? 8 : 16; };
#ifndef M4Q_MAXW_92
#define M4Q_MAXW_92 16
#endif
template <> struct Tiles<9, 2> { static constexpr int MAXW = M4Q_MAXW_92; };   // 12: 3 warps per scheduler, 168 registers, no spills
template <> struct Tiles<8, 2> { static constexpr int MAXW = 16; };   // 15 fit; measured faster than 12 x 168 registers

template <int C_, int M_> struct Cfg {
    static constexpr int C = C_, N = 2 * C_, M = M_, Q = N + M_;
    static constexpr int MAXW = Tiles<C_, M_>::MAXW;
    static constexpr int NT = cdiv(N, 8), GT = cdiv(Q + 1, 8), TT = cdiv(Q, 8);   // tile counts
    // operand rows: the N real ones plus, when N is not a multiple of 8, ONE row of zeros that every padding index of
    // the last contraction tile is mapped to (instead of 8 NT - N zero rows: 2 x 130 doubles less per member for N = 18)
    static constexpr int KR = (N % 8 == 0) ? N : N + 1;
    static constexpr int LDP = cmin(next_mod(8 * NT, 2, 8), next_mod(8 * NT, 6, 8));
    static constexpr int LDG = cmin(next_mod(8 * GT, 2, 8), next_mod(8 * GT, 6, 8));
    // the factor runs in Hermitian coordinates (HermCfg) when the QP allows it; the other instantiations keep the
    // realified factor for every QP
    static constexpr bool HERM = C_ == 9 && M_ == 2;
};

// ---------------------------------------------------------------------------------------------------------
// Factor coordinates of the Hermitian subspace (DESIGN.md section 2.4).  sigma is the index involution of the lift
// (transpose of vec(rho), ...).  When every model block has N_k[sigma, sigma] = conj(N_k), the costs are sigma-symmetric
// and the guess trajectory is sigma-conjugate-symmetric, the Riccati recursion leaves the Hermitian subspace
// {x_sigma(k) = conj(x_k)} (real dimension C) invariant and K_t, S_t^-1, dv_t depend only on P restricted to it.
// Coordinates (unnormalised, +-1 basis): Re x_k for a fixed point k; (Re x_k + Re x_sk) / 2 and (Im x_k - Im x_sk) / 2
// for a pair k < sk.  Padded with one zero coordinate to an even count (the P update stores column pairs).
// ---------------------------------------------------------------------------------------------------------
template <class CF> struct HermCfg {
    static constexpr int C = CF::C, N = rup(CF::C, 2), M = CF::M, Q = N + M;
    static constexpr int NT = cdiv(N, 8), GT = cdiv(Q + 1, 8), TT = cdiv(Q, 8);
    static constexpr int KR = (N % 8 == 0) ? N : N + 1;
    static constexpr int LDP = cmin(next_mod(8 * NT, 2, 8), next_mod(8 * NT, 6, 8));
    static constexpr int LDG = cmin(next_mod(8 * GT, 2, 8), next_mod(8 * GT, 6, 8));
    // the complex A_t is staged behind the reduced G, inside the realified G buffer.  Only instantiations with
    // CF::HERM run this factor; riccati_factor instantiates HermCfg for every CF, so the layout checks bind only there.
    static constexpr int ASTAGE = rup(KR * LDG, 2);
    static_assert(!CF::HERM || ASTAGE + 2 * C * C <= CF::KR * CF::LDG, "staged A_t does not fit the G buffer");
    static_assert(!CF::HERM || KR * LDP <= CF::KR * CF::LDP, "reduced P does not fit the P buffer");
    static_assert(!CF::HERM || M * N + N <= M * CF::N, "reduced dv does not fit behind T21");
};
// Basis descriptors (ints, built once per launch from sigma, m4q_kernels.cu build_tables):
//   coordinate a < N:  HB_J1 / HB_J2 [a]: the two realified indices it averages (equal for a fixed point; -1: padding);
//                      HB_SG [a]: +1 (real part) or -1 (imaginary part: (x_j1 - x_j2) / 2)
//   realified j < 2C:  HB_CO [j]: the coordinate j belongs to; HB_WT [j]: 2 x its weight in the map back (2, 1, -1, 0);
//                      HB_PA [j]: the realified index sigma(j) (same part)
//   HB_OK: 1 when the shared model and the costs are sigma-symmetric (and the reduced factor is enabled)
template <class CF> struct HermBasis {
    static constexpr int NR = HermCfg<CF>::N, N = CF::N;
    static constexpr int J1 = 0, J2 = NR, SG = 2 * NR, CO = 3 * NR, WT = CO + N, PA = WT + N, OK = PA + N, INTS = OK + 1;
};

// ---------------------------------------------------------------------------------------------------------
// Memory plan of one member (= one warp).
//   * shared-memory slab: the Riccati scratch (P, [A|B], W), a 2-slot ring of stage records, the control
//     trajectories and a few vectors -- 17.4 KB for the transmon, (almost) independent of the horizon: 12 members
//     are resident per SM;
//   * L2-resident workspace in global memory (one per resident warp, re-used member after member): the
//     horizon-length data.  Per stage one RECORD [K_t | S_t^-1 | dv_t | B_t | D_t | A_t | x_t - r_t], then the trajectories
//     Xg, Xo [(H+1) N].  Records are written with plain stores where they are produced (factor: K, S^-1, dv;
//     linearisation: B, D) and streamed back one stage ahead of their use through the ring with cp.async
//     (LDGSTS, 16-byte chunks), so the sweeps never wait on L2.
// ---------------------------------------------------------------------------------------------------------
template <class CF> struct Rec {
    // K and B are kept in "complex pair" layout [M][C] double2: element (a, r) = (X[.][r], X[.][C + r]), so that
    // a control row K_a (or a column of B) is read by the same complex mat-vec loop as a row of A_t.
    static constexpr int K = 0;                                  // [M][C] pairs (K[a][r], K[a][C + r])
    static constexpr int SINV = K + rup(CF::M * CF::N, 2);       // [M][M]
    static constexpr int DV = SINV + rup(CF::M * CF::M, 2);      // [N]
    static constexpr int B = DV + CF::N;                         // [M][C] pairs (B[r][i], B[C + r][i])
    static constexpr int D = B + rup(CF::N * CF::M, 2);          // [N]
    static constexpr int SMALL = D + CF::N;                      // end of the part the factor reads back ([B | D])
    static constexpr int AT = SMALL;                             // [C][CA] complex: A_t = sum_k phi_k(u_t) block_k
    // row stride of A_t in complex elements: the rows read by different lanes of the mat-vec (16-byte loads, one row
    // per lane) must start in different banks; with C = 8 or 16 the rows are a multiple of 128 bytes apart, an 8-way
    // conflict (measured: +10 % / +15 % on the crosstalk / gate workloads with the odd stride; C = 4 is 2-way only and
    // was faster unpadded)
    static constexpr int CA = (CF::C % 8 == 0) ? CF::C + 1 : CF::C;
    static constexpr int XC = AT + 2 * CF::C * CA;               // [N] x_t - r_t of the last rollout (adjoint sweep)
    static constexpr int SIZE = XC + CF::N;
    // ring slots start on 128-byte boundaries: a 512-byte cp.async request then covers 4 shared-memory lines, not 5
    static constexpr int SLOT = rup(SIZE, 16), BDSLOT = rup(D + CF::N - B, 16);
    static_assert(B % 2 == 0 && SMALL % 2 == 0 && SIZE % 2 == 0, "records are moved in 16-byte chunks");
    // offset of K[a][k] / B[k][i] (k = realified state index) inside their pair blocks
    __host__ __device__ static constexpr int pair(int ctl, int k) { return (ctl * CF::C + (k % CF::C)) * 2 + (k >= CF::C); }
    // during the vector sweeps whole records are staged in the [P | G] buffers (only live inside the factor).  With
    // C = 4 and three or more controls two records are longer than [P | G] (242 / 280 doubles against 224): the ring
    // then gets a slab region of its own (Slab::layout), at least as long as [P | G] so that the exact-stage scratch,
    // which also lives at the ring, fits either way.
    static constexpr bool ALIAS = SLOT + SIZE <= CF::KR * (CF::LDP + CF::LDG);
    static constexpr int OWN = cmax(SLOT + SIZE, CF::KR * (CF::LDP + CF::LDG));   // length of the ring's own region
};
template <class CF> __host__ __device__ constexpr int ws_doubles(int H) {
    return H * Rec<CF>::SIZE + 2 * (H + 1) * CF::N;
}

template <class CF> struct Slab {
    double *P, *AB, *W, *T21, *S, *ring, *kk, *hl, *Ug, *Uo, *z, *y, *x0, *va, *vb, *xT, *lo0, *hi0, *xcur, *xmeas, *scr;
    double *recring;   // 2-slot ring of whole stage records for the vector sweeps (aliases the factor scratch if it fits)
    double *xd;        // 2 N doubles of scratch for the general-cost adjoint sweep
    int *mask;
    int *flips;        // how often a control has been released from the working set during the current QP solve

    __host__ __device__ static int doubles(int H, int nblk, int dd) {
        return layout(nullptr, nullptr, H, nblk, dd);
    }
    // scratch of the linearisation (2 x [p][M] derivative weights) and of the plant step (4 complex d x d):
    // aliases G, which is only live inside the Riccati factor
    __host__ __device__ static constexpr int scratch_doubles() { return CF::KR * CF::LDG; }
    __host__ __device__ static bool scratch_fits(int nblk, int dd) {
        return cmax(8 * dd, 2 * CF::M * nblk) <= scratch_doubles();
    }
    // dd = plant state length in complex numbers (d*d)
    __host__ __device__ static int layout(Slab *s, double *base, int H, int nblk, int dd) {
        constexpr int N = CF::N, M = CF::M;
        int o = 0;
        auto take = [&](double **dst, int cnt, int align = 2) {
            o = rup(o, align);
            if (s) *dst = base + o;
            o += rup(cnt, 2);
        };
        Slab dummy;
        Slab *q = s ? s : &dummy;
        take(&q->P, CF::KR * CF::LDP, 16);   // P_{t+1}, zero padded, [KR][LDP]
        take(&q->AB, CF::KR * CF::LDG);      // G = [A_t | B~_t | D~_t], zero padded, [KR][LDG]
        take(&q->W, M * N);                  // K_t for the update of P (W = P G itself never leaves the registers)
        q->scr = q->AB;
        if (Rec<CF>::ALIAS) q->recring = q->P;
        take(&q->xd, 2 * N);
        take(&q->T21, M * N);
        take(&q->S, M * M);
        take(&q->ring, 2 * Rec<CF>::BDSLOT, 16);   // factor: [B_t | D_t] of two stages
        take(&q->kk, H * M);
        take(&q->hl, H * M);
        take(&q->Ug, H * M);
        take(&q->Uo, H * M);
        take(&q->z, H * M);
        take(&q->y, H * M);
        take(&q->x0, N);
        take(&q->va, N + 2);   // sweep vectors: imaginary half at offset rup(C, 2)
        take(&q->vb, N + 2);
        take(&q->xT, N);
        take(&q->lo0, M);
        take(&q->hi0, M);
        take(&q->xcur, 2 * dd);
        take(&q->xmeas, 2 * dd);
        double *mk = nullptr;
        take(&mk, cdiv(H * M, 2));
        if (s) s->mask = reinterpret_cast<int *>(mk);
        take(&mk, cdiv(H * M, 2));
        if (s) s->flips = reinterpret_cast<int *>(mk);
        if (!Rec<CF>::ALIAS) take(&q->recring, Rec<CF>::OWN, 16);
        return o;
    }
    // the part that must survive between launches in host-stepped mode: Xg | Ug | z | y | xcur | xmeas
    __host__ __device__ static int persistent_doubles(int H, int dd) {
        return (H + 1) * CF::N + 3 * H * CF::M + 4 * dd;
    }
};

// ---------------------------------------------------------------------------------------------------------
// The large device functions below are __noinline__ (one copy each: the hot code has to stay resident in the
// instruction cache) and therefore re-derive every shared-memory pointer from the dynamic shared-memory base, so
// that the compiler keeps emitting LDS/STS instead of generic loads.  A slab is named by its offset (in doubles);
// ws is the member's workspace (global memory in the fused loop and the QP kernel).
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double *dyn_smem() {
    extern __shared__ double2 m4q_dyn_smem[];
    return reinterpret_cast<double *>(m4q_dyn_smem);
}
struct SlabRef {
    int off, H, nblk, dd;
    double *ws;
};
template <class CF> __device__ __forceinline__ Slab<CF> slab_view(const SlabRef &r) {
    Slab<CF> s;
    Slab<CF>::layout(&s, dyn_smem() + r.off, r.H, r.nblk, r.dd);
    return s;
}
template <class CF> __device__ __forceinline__ double *ws_rec(const SlabRef &r, int t) { return r.ws + t * Rec<CF>::SIZE; }
template <class CF> __device__ __forceinline__ double *ws_Xg(const SlabRef &r) { return r.ws + r.H * Rec<CF>::SIZE; }
template <class CF> __device__ __forceinline__ double *ws_Xo(const SlabRef &r) {
    return r.ws + r.H * Rec<CF>::SIZE + (r.H + 1) * CF::N;
}

// cp.async (LDGSTS): 16 bytes global -> shared, L2 only
__device__ __forceinline__ void cp_async16(double *smem_dst, const double *gsrc) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(__cvta_generic_to_global(gsrc)) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
// stream COUNT doubles (even, compile time) global -> shared; one group per call
template <int COUNT> __device__ __forceinline__ void prefetch_block(double *dst, const double *src, int lane) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(dst) + 16 * lane;
    unsigned long long ga = (unsigned long long)__cvta_generic_to_global(src) + 16 * lane;
#pragma unroll
    for (int c = 0; c < cdiv(COUNT / 2, 32); ++c, sa += 512, ga += 512)
        if (c * 32 + lane < COUNT / 2) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(ga) : "memory");
    cp_async_commit();
}

// ---------------------------------------------------------------------------------------------------------
// Stage operator A_t = sum_k w_k(t) block_k.  Fused loop: blocks = shared model [A, N_1..N_p], w = monomials of
// the guess control (held in slab.phi).  Stand-alone QP: one dense block per stage, w = 1.
// ---------------------------------------------------------------------------------------------------------
struct StageOps {
    const double2 *blocks;   // [nblk][C][C] (fused: shared memory) or [H][C][C] (dense: global memory)
    int nblk;
    int stage_stride;        // in complex elements; 0 for the fused model
    int soff;                // FUSED: offset (doubles) of the blocks in dynamic shared memory
    int soffT;               // FUSED, c multiple of 8: offset of the transposed copies of blocks 1..p (0: none)
    // block weights of a stage: w_0 = 1, w_k = the k-th monomial of the stage's guess control (linearize.py:123-128),
    // evaluated where they are needed from the exponent table instead of being stored per stage (H (p + 1) doubles of
    // shared memory per member, 4.8 KB at H = 100 with the order-2 library).  pow == nullptr: dense stage operators, w = 1.
    const int *pow;          // [p][M] exponents (FUSED: re-derived from pow_soff)
    int pow_soff;            // FUSED: offset (doubles) of the exponent table in dynamic shared memory
    int first_order;         // the library is (u_1, .., u_M): w_k = u_{k-1}
};
template <int M> __device__ __forceinline__ double stage_weight(const StageOps &o, const double *u, int kb) {
    if (kb == 0 || o.pow == nullptr) return 1.0;
    if (o.first_order) return u[kb - 1];
    double ph = 1.0;
#pragma unroll
    for (int l = 0; l < M; ++l) {
        const int e = o.pow[(kb - 1) * M + l];
        const double ul = u[l];
#pragma unroll 1
        for (int q = 0; q < e; ++q) ph *= ul;
    }
    return ph;
}
// FUSED = true: model blocks and cost matrices live in dynamic shared memory at known offsets
template <bool FUSED> __device__ __forceinline__ StageOps localize(const StageOps &o) {
    StageOps r = o;
    if (FUSED) {
        r.blocks = reinterpret_cast<const double2 *>(dyn_smem() + o.soff);
        r.pow = reinterpret_cast<const int *>(dyn_smem() + o.pow_soff);
    }
    return r;
}

// Data of one QP instance that is not in the slab (targets and costs, pre-realified by a prep kernel).
struct QPData {
    const double *Q;      // stage cost Qbar(t) = Q + t*q_stride, t < H   [N][N] symmetric, realified
    int q_stride;
    const double *Qf;     // terminal cost
    const double *R;      // R(t) = R + t*r_stride  [M][M] symmetric
    int r_stride;
    const double *r;      // realified targets r(t) = r + t*N, t <= H
    const double *qlin;   // Qbar(t) r(t) for t < H:  qlin + t*N
    const double *qlinf;  // Qf r(H)
    const double *ub;     // control targets ub(t) = ub + t*M
    const double *Rub;    // R(t) ub(t)
    double sat;
    int q_diag;           // 1 if every Qbar is diagonal (fast path of the line search / adjoint)
    int Q_soff, Qf_soff, R_soff;   // FUSED: offsets (doubles) of Q, Qf, R in dynamic shared memory
    // Hermitian coordinates (HermCfg): reduced costs T^T Q T, T^T Qf T (global), basis descriptors (HermBasis) and
    // whether this QP may use them (herm != 0)
    const double *Qh, *Qfh;
    const int *hb;
    int herm;
};
template <bool FUSED> __device__ __forceinline__ QPData localize(const QPData &q) {
    QPData r = q;
    if (FUSED) {
        r.Q = dyn_smem() + q.Q_soff;
        r.Qf = dyn_smem() + q.Qf_soff;
        r.R = dyn_smem() + q.R_soff;
    }
    return r;
}

struct QPSet {
    double rho, alpha, eps;
    int max_admm, polish, max_polish, admm_first, adaptive_rho;
    int kkt_mode;   // 0: off; 1: pivoted KKT solve as the last resort (where status 2 would be returned); 2: as soon as the
                    // Riccati active-set rounds fail once, and from then on for every QP of the member (m4q_kkt.cuh)
    double *kkt;    // this warp's KKT workspace (Kkt<CF>::doubles(H)), nullptr: none
};

struct Counters {
    int admm, factor, polish, solves;
    int kkt;        // pivoted KKT solves (reported with the polish rounds)
    int sticky;     // kkt_mode 2: a QP of this member broke down numerically in the Riccati path; later QPs skip it
    int fac_herm, fac_full;   // factorisations in Hermitian / realified coordinates
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
// Sum M values over the warp, result in every lane.  Two values share one butterfly: the first exchange sends the
// value a lane does not keep, so 6 shuffle stages replace 10.
template <int M> __device__ __forceinline__ void warp_sum_vec(double (&g)[M], int lane) {
    if constexpr (M >= 2) {
        const bool hi = (lane & 16) != 0;
        double keep = hi ? g[1] : g[0];
        keep += __shfl_xor_sync(FULL, hi ? g[0] : g[1], 16);
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) keep += __shfl_xor_sync(FULL, keep, o);
        const double other = __shfl_xor_sync(FULL, keep, 16);
        g[0] = hi ? other : keep;
        g[1] = hi ? keep : other;
#pragma unroll
        for (int i = 2; i < M; ++i) g[i] = warp_sum(g[i]);
    } else {
        g[0] = warp_sum(g[0]);
    }
}

// D (8x8) += A (8x4, row) * B (4x8, col) on the fp64 tensor cores.  Lane l holds A[l/4][l%4], B[l%4][l/4] and
// D[l/4][2*(l%4) + {0, 1}].
__device__ __forceinline__ void dmma(double (&d)[2], double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(d[0]), "+d"(d[1])
        : "d"(a), "d"(b));
}

// inverse of a small symmetric positive definite matrix held in registers (Gauss-Jordan, no pivoting)
template <int M> __device__ __forceinline__ void spd_inverse(double (&a)[M][M], double (&inv)[M][M]) {
    if constexpr (M == 1) {
        inv[0][0] = 1.0 / a[0][0];
        return;
    }
    if constexpr (M == 2) {   // adjugate / determinant: one division
        const double r = 1.0 / fma(a[0][0], a[1][1], -a[0][1] * a[1][0]);
        inv[0][0] = a[1][1] * r;
        inv[1][1] = a[0][0] * r;
        inv[0][1] = -a[0][1] * r;
        inv[1][0] = -a[1][0] * r;
        return;
    }
#pragma unroll
    for (int i = 0; i < M; ++i)
#pragma unroll
        for (int j = 0; j < M; ++j) inv[i][j] = (i == j) ? 1.0 : 0.0;
#pragma unroll
    for (int col = 0; col < M; ++col) {
        const double piv = 1.0 / a[col][col];
#pragma unroll
        for (int j = 0; j < M; ++j) {
            a[col][j] *= piv;
            inv[col][j] *= piv;
        }
#pragma unroll
        for (int r = 0; r < M; ++r) {
            if (r == col) continue;
            const double f = a[r][col];
#pragma unroll
            for (int j = 0; j < M; ++j) {
                a[r][j] = fma(-f, a[col][j], a[r][j]);
                inv[r][j] = fma(-f, inv[col][j], inv[r][j]);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// y[lane] = (A_t x)[lane] (TRANS = false) or (A_t^T x)[lane] (TRANS = true) for lane < N; x realified
// [Re | Im] in shared memory, A_t complex [C][C].  With m = A_t[r][j] (or [j][r]),
//   A,   re row:  sum m.x xr - m.y xi      A,   im row:  sum m.x xi + m.y xr
//   A^T, re row:  sum m.x xr + m.y xi      A^T, im row:  sum m.x xi - m.y xr
// so each lane reads x through two lane-dependent base pointers and one sign: no selects in the loop.
// ---------------------------------------------------------------------------------------------------------
template <class CF, bool TRANS, int LDA = CF::C>
__device__ __forceinline__ double cmatvec(const double2 *At, const double *x, int lane) {
    constexpr int C = CF::C, N = CF::N;
    if (lane >= N) return 0.0;
    const bool im = lane >= C;
    const int r = im ? lane - C : lane;
    const double *xp = x + (im ? C : 0), *xq = x + (im ? 0 : C);
    const double sgn = (im != TRANS) ? 1.0 : -1.0;
    const double2 *blk = At + (TRANS ? r : r * LDA);
    double p0 = 0.0, p1 = 0.0, q0 = 0.0, q1 = 0.0;
#pragma unroll
    for (int j = 0; j < C; ++j) {
        const double2 m = blk[TRANS ? j * LDA : j];
        if (j & 1) {
            p1 = fma(m.x, xp[j], p1);
            q1 = fma(m.y, xq[j], q1);
        } else {
            p0 = fma(m.x, xp[j], p0);
            q0 = fma(m.y, xq[j], q0);
        }
    }
    return fma(sgn, q0 + q1, p0 + p1);
}
// The same loop with M extra rows in the lanes N .. N+M-1: row a of Ext ([M][C] pairs (e[r], e[C + r])) dotted with
// x.  Backward sweep: Ext = B_t -> B_t^T v;  forward sweep: Ext = K_t -> K_t x.  The control-space reductions thus
// cost no shuffle tree: lane N + a holds the result and broadcasts it.
// x is held with its imaginary half at offset XP = rup(C, 2) (sweep_idx), so that both halves can be read as 16-byte
// pairs: C / 2 + 1 wide loads per half instead of C narrow ones.
template <class CF> __device__ __forceinline__ int sweep_idx(int lane) {
    return lane + (lane >= CF::C ? rup(CF::C, 2) - CF::C : 0);
}
template <class CF, bool TRANS>
__device__ __forceinline__ double cmatvec_ext(const double2 *At, const double2 *Ext, const double *x, int lane) {
    constexpr int C = CF::C, N = CF::N, M = CF::M, XP = rup(C, 2);
    static_assert(N + M <= 32, "no free lanes for the control rows");
    if (lane >= N + M) return 0.0;
    const bool ext = lane >= N;
    const bool im = !ext && lane >= C;
    const int r = ext ? lane - N : (im ? lane - C : lane);
    const double *xp = x + (im ? XP : 0), *xq = x + (im ? 0 : XP);
    const double sgn = (ext || im != TRANS) ? 1.0 : -1.0;
    constexpr int CA = Rec<CF>::CA;   // At is the record's A_t block (row stride CA), Ext a pair block (row stride C)
    const double2 *blk = ext ? Ext + r * C : At + (TRANS ? r : r * CA);
    const int stride = (!ext && TRANS) ? CA : 1;
    double p0 = 0.0, p1 = 0.0, q0 = 0.0, q1 = 0.0;
#pragma unroll
    for (int j = 0; j + 1 < C; j += 2) {
        const double2 ma = blk[0], mb = blk[stride];
        blk += 2 * stride;
        const double2 xa = *reinterpret_cast<const double2 *>(xp + j), xb = *reinterpret_cast<const double2 *>(xq + j);
        p0 = fma(ma.x, xa.x, p0);
        q0 = fma(ma.y, xb.x, q0);
        p1 = fma(mb.x, xa.y, p1);
        q1 = fma(mb.y, xb.y, q1);
    }
    if constexpr (C % 2 == 1) {
        const double2 m = *blk;
        p0 = fma(m.x, xp[C - 1], p0);
        q0 = fma(m.y, xq[C - 1], q0);
    }
    return fma(sgn, q0 + q1, p0 + p1);
}
// same product straight from the model blocks, A_t = sum_k phi_k block_k (cold paths: one call per MPC step)
template <class CF>
__device__ __forceinline__ double apply_A(const StageOps &ops, const double *phi_t, int t, const double *x, int lane) {
    constexpr int C = CF::C;
    double out = 0.0;
#pragma unroll 1
    for (int kb = 0; kb < ops.nblk; ++kb)
        out = fma(phi_t[kb], cmatvec<CF, false>(ops.blocks + (size_t)t * ops.stage_stride + kb * C * C, x, lane), out);
    return out;
}

// ---------------------------------------------------------------------------------------------------------
// Bounds of the control box (optimize.py:29-30, :43)
// ---------------------------------------------------------------------------------------------------------
template <class CF> __device__ __forceinline__ double box_lo(const Slab<CF> &s, double sat, int t, int i) {
    return t == 0 ? s.lo0[i] : -sat;
}
template <class CF> __device__ __forceinline__ double box_hi(const Slab<CF> &s, double sat, int t, int i) {
    return t == 0 ? s.hi0[i] : sat;
}

// ---------------------------------------------------------------------------------------------------------
// Riccati matrix sweep.  masked: controls with mask != 0 are pinned to their bound (polish), rho_half = 0.
// Produces K_t, S_t^-1, dv_t = P_{t+1} (D_t + B_fixed b) for all stages (written to the stage records).
// Per stage  T = G^T P_{t+1} G,  S = R + rho/2 + T22,  P_t = Qbar_t + T11 - T21^T S^-1 T21.  Shared memory is the
// resource this kernel is bound by, so the products keep their traffic through it small:
//   * W^T = G^T P (G = [A_t | B~_t | D~_t], N x (Q + 1)) is accumulated in DMMA fragments and consumed by the second
//     product T = W^T G straight from the registers: a k-step (kt, e) contracts over k = 8 kt + 2 c4 + e, the very
//     column of W^T that lane (g8, c4) holds in accumulator element e, so the A operand of the second product IS
//     the accumulator -- no store, no reload, no shuffle (the permutation of the contraction index is harmless as
//     long as both operands use it);
//   * the G fragments are the A operand of the first product and the B operand of the second;
//   * dv_t = P_{t+1} D~_t is row Q of W^T and goes from the accumulators to the stage record;
//   * P_t = Qbar_t + T11 - T21^T K is applied to the accumulator fragments of T11; each lane stores its part of the
//     upper block triangle and its mirror image, so P stays exactly symmetric.
// ---------------------------------------------------------------------------------------------------------
// FC: the factor's coordinates.  FC = CF: the realified state (N = 2C).  FC = HermCfg<CF>: Hermitian coordinates
// (N = rup(C, 2)); A_t is projected from the complex A_t staged behind G, [B | D] from the ring, the costs are the
// reduced tables, and K_t, dv_t are mapped back to the realified record layout (halving and sign flips).  One DMMA core
// for both.
template <class CF, class FC, bool FUSED>
__device__ __noinline__ void riccati_factor(SlabRef sr, const StageOps &ops_in, const QPData &qp_in, double rho_half,
                                            bool masked, int lane) {
    constexpr int C = CF::C, M = CF::M;
    constexpr int N = FC::N, Q = FC::Q;
    constexpr int NT = FC::NT, GT = FC::GT, TT = FC::TT, KR = FC::KR, LDP = FC::LDP, LDG = FC::LDG;
    constexpr bool RED = FC::N != CF::N;
    constexpr bool LASTNAT = (N % 8 != 0) && (N % 8 <= 4);   // ragged last contraction tile: one k-step of 4 indices
    constexpr int KSTEPS = 2 * NT - (LASTNAT ? 1 : 0);
    using R_ = Rec<CF>;
    using HB = HermBasis<CF>;
    const Slab<CF> s = slab_view<CF>(sr);
    const StageOps ops = localize<FUSED>(ops_in);
    const QPData qp = localize<FUSED>(qp_in);
    const int H = sr.H;
    const int g8 = lane >> 2, c4 = lane & 3;   // fragment coordinates of this lane
    const double *Qfac = RED ? qp.Qh : qp.Q, *Qffac = RED ? qp.Qfh : qp.Qf;
    // P <- Qf with zero padding; G zeroed once (padding rows / columns are never written afterwards)
#pragma unroll 1
    for (int e = lane; e < KR * LDP; e += 32) {
        const int i = e / LDP, j = e % LDP;
        s.P[e] = (i < N && j < N) ? Qffac[i * N + j] : 0.0;
    }
#pragma unroll 1
    for (int e = lane; e < KR * LDG; e += 32) s.AB[e] = 0.0;
    // Hermitian coordinates: what this lane projects and maps back (constant over the stages)
    constexpr int NEA = RED ? cdiv(C * C, 32) : 1;
    int a_o1[NEA], a_o2[NEA], a_g[NEA];
    double a_s2[NEA], a_sg[NEA];
    bool a_re[NEA];
    int h_j1 = 0, h_j2 = 0, h_co = 0;
    double h_sg = 0.0, h_wt = 0.0;
    double2 *astage = reinterpret_cast<double2 *>(s.AB + HermCfg<CF>::ASTAGE);
    if constexpr (RED) {
#pragma unroll
        for (int q = 0; q < NEA; ++q) {
            // entry (a, b) of A~ = T^+ A_t T: column b of A_t T is A[:, kc] + s2 A[:, kc2] (times i for an imaginary
            // coordinate), read at the representative row kr of coordinate a (real or imaginary part)
            const int e = lane + 32 * q, a = e < C * C ? e / C : 0, b = e < C * C ? e % C : 0;
            const int r1 = qp.hb[HB::J1 + a], c1 = qp.hb[HB::J1 + b], c2 = qp.hb[HB::J2 + b];
            const bool row_im = r1 >= C, col_im = c1 >= C;
            const int kr = r1 % C, kc = c1 % C, kc2 = c2 % C;
            a_o1[q] = kr * C + kc;
            a_o2[q] = kr * C + kc2;
            a_s2[q] = c1 == c2 ? 0.0 : (double)qp.hb[HB::SG + b];
            a_re[q] = row_im == col_im;
            a_sg[q] = (col_im && !row_im) ? -1.0 : 1.0;
            a_g[q] = e < C * C ? a * LDG + b : -1;
        }
        if (lane < C) {
            h_j1 = qp.hb[HB::J1 + lane];
            h_j2 = qp.hb[HB::J2 + lane];
            h_sg = (double)qp.hb[HB::SG + lane];
        }
        if (lane < CF::N) {
            h_co = qp.hb[HB::CO + lane];
            h_wt = 0.5 * (double)qp.hb[HB::WT + lane];
        }
    }
    // where the entries of A_t this lane forms go: element e = lane + 32 q of the row-major C x C block
    constexpr int NE = cdiv(C * C, 32);
    int g_off[NE], r_off[NE];
#pragma unroll
    for (int q = 0; q < NE; ++q) {
        const int e = lane + 32 * q, r = e / C, j = e % C;
        g_off[q] = e < C * C ? r * LDG + j : -1;
        r_off[q] = r * R_::CA + j;
    }
    constexpr int BD = R_::SMALL - R_::B;   // [B_t | D_t]
    prefetch_block<BD>(s.ring + ((H - 1) & 1) * R_::BDSLOT, ws_rec<CF>(sr, H - 1) + R_::B, lane);
#pragma unroll 1
    for (int t = H - 1; t >= 0; --t) {
        const double *ug_t = s.Ug + t * M;
        const double2 *blk0 = ops.blocks + (size_t)t * ops.stage_stride;
        const double *Bt = s.ring + (t & 1) * R_::BDSLOT, *Dt = Bt + (R_::D - R_::B);
        double *rec = ws_rec<CF>(sr, t);
        cp_async_wait_all();
        __syncwarp();   // B_t, D_t have landed; P_{t+1} of the previous stage is complete
        if (t > 0) prefetch_block<BD>(s.ring + ((t - 1) & 1) * R_::BDSLOT, ws_rec<CF>(sr, t - 1) + R_::B, lane);
        // realified A_t = sum_k phi_k block_k into G[:, 0:N] (and, complex, into the record for the vector sweeps)
        {
            double ar[NE], ai[NE];
#pragma unroll
            for (int q = 0; q < NE; ++q) ar[q] = ai[q] = 0.0;
            const double2 *bp = blk0 + lane;
            const int qlast = (C * C - 1 - lane) >> 5;   // last valid q of this lane (loads clamped, not predicated)
#pragma unroll 1
            for (int kb = 0; kb < ops.nblk; ++kb, bp += C * C) {
                const double ph = stage_weight<M>(ops, ug_t, kb);
                double2 v[NE];
#pragma unroll
                for (int q = 0; q < NE; ++q) v[q] = bp[32 * (q < qlast ? q : qlast)];
#pragma unroll
                for (int q = 0; q < NE; ++q) {
                    ar[q] = fma(ph, v[q].x, ar[q]);
                    ai[q] = fma(ph, v[q].y, ai[q]);
                }
            }
#pragma unroll
            for (int q = 0; q < NE; ++q) {
                if (g_off[q] >= 0) {
                    if constexpr (RED) {
                        astage[lane + 32 * q] = make_double2(ar[q], ai[q]);
                    } else {
                        double *g = s.AB + g_off[q];
                        g[0] = ar[q];
                        g[C] = -ai[q];
                        g[C * LDG] = ai[q];
                        g[C * LDG + C] = ar[q];
                    }
                    reinterpret_cast<double2 *>(rec + R_::AT)[r_off[q]] = make_double2(ar[q], ai[q]);
                }
            }
        }
        if constexpr (RED) {
            __syncwarp();   // the complex A_t is staged
#pragma unroll
            for (int q = 0; q < NEA; ++q) {
                const double2 z1 = astage[a_o1[q]], z2 = astage[a_o2[q]];
                const double zr = fma(a_s2[q], z2.x, z1.x), zi = fma(a_s2[q], z2.y, z1.y);
                if (a_g[q] >= 0) s.AB[a_g[q]] = a_re[q] ? zr : a_sg[q] * zi;
            }
        }
        // B~ into G[:, N:Q], D~ into G[:, Q]: lane k < N owns row k; the working set of the stage is read once
        int mk[M];
#pragma unroll
        for (int i = 0; i < M; ++i) mk[i] = masked ? s.mask[t * M + i] : 0;
        if (RED && lane < C) {
            // coordinate lane of B_t, D_t: (x_j1 +- x_j2) / 2 (a fixed point: j1 == j2, +)
            double dt = 0.5 * fma(h_sg, Dt[h_j2], Dt[h_j1]);
#pragma unroll
            for (int i = 0; i < M; ++i) {
                const double b = 0.5 * fma(h_sg, Bt[R_::pair(i, h_j2)], Bt[R_::pair(i, h_j1)]);
                s.AB[lane * LDG + N + i] = mk[i] ? 0.0 : b;
                if (mk[i]) dt = fma(b, mk[i] == 1 ? box_lo(s, qp.sat, t, i) : box_hi(s, qp.sat, t, i), dt);
            }
            s.AB[lane * LDG + Q] = dt;
        } else if (!RED && lane < N) {
            double dt = Dt[lane];
#pragma unroll
            for (int i = 0; i < M; ++i) {
                const double b = Bt[R_::pair(i, lane)];
                s.AB[lane * LDG + N + i] = mk[i] ? 0.0 : b;
                if (mk[i]) dt = fma(b, mk[i] == 1 ? box_lo(s, qp.sat, t, i) : box_hi(s, qp.sat, t, i), dt);
            }
            s.AB[lane * LDG + Q] = dt;
        }
        __syncwarp();
        // ---- W^T = G^T P: tile (qi, mi) holds W^T[qi*8 + g8][mi*8 + 2*c4 + {0,1}]
        double w[GT][NT][2];
#pragma unroll
        for (int qi = 0; qi < GT; ++qi)
#pragma unroll
            for (int mi = 0; mi < NT; ++mi) w[qi][mi][0] = w[qi][mi][1] = 0.0;
        {
            // operand rows of k-step ks: tile kt = ks / 2, e = ks % 2 -> 8 kt + 2 c4 + e; when the last tile holds at most 4
            // real indices (N = 18: two) it is ONE step over 8 kt + c4 instead, padding indices -> the zero row
            auto row_of = [&](int ks) {
                int r = (ks >> 1) * 8 + 2 * c4 + (ks & 1);
                if (LASTNAT && ks == KSTEPS - 1) r = (NT - 1) * 8 + c4;
                return r < N ? r : KR - 1;
            };
            const double *gb0 = s.AB + g8, *pb0 = s.P + g8;
            double gf[GT], pf[NT];
            {
                const int r = row_of(0);
#pragma unroll
                for (int qi = 0; qi < GT; ++qi) gf[qi] = gb0[r * LDG + qi * 8];
#pragma unroll
                for (int mi = 0; mi < NT; ++mi) pf[mi] = pb0[r * LDP + mi * 8];
            }
#pragma unroll 1
            for (int ks = 0; ks < KSTEPS; ++ks) {
                // next step's fragments in flight while this step's MMAs issue; the last step reloads its own
                const int r = row_of(ks + 1 < KSTEPS ? ks + 1 : ks);
                double gn[GT], pn[NT];
#pragma unroll
                for (int qi = 0; qi < GT; ++qi) gn[qi] = gb0[r * LDG + qi * 8];
#pragma unroll
                for (int mi = 0; mi < NT; ++mi) pn[mi] = pb0[r * LDP + mi * 8];
#pragma unroll
                for (int qi = 0; qi < GT; ++qi)
#pragma unroll
                    for (int mi = 0; mi < NT; ++mi) dmma(w[qi][mi], gf[qi], pf[mi]);
#pragma unroll
                for (int qi = 0; qi < GT; ++qi) gf[qi] = gn[qi];
#pragma unroll
                for (int mi = 0; mi < NT; ++mi) pf[mi] = pn[mi];
            }
        }
        // dv_t = P_{t+1} D~_t = row Q of W^T: held by the lanes with g8 == Q % 8, columns mi*8 + 2 c4 + {0, 1}
        // (Hermitian coordinates: to the scratch behind T21, mapped back below)
        double *dvb = s.T21 + M * N;
        if (g8 == Q % 8) {
#pragma unroll
            for (int mi = 0; mi < NT; ++mi) {
                const int j = mi * 8 + 2 * c4;
                if (j < N) *reinterpret_cast<double2 *>((RED ? dvb : rec + R_::DV) + j) = make_double2(w[Q / 8][mi][0], w[Q / 8][mi][1]);
            }
        }
        // ---- T = W^T G, upper block triangle of the leading Q x Q part: A operand = the accumulators of W^T
        double tt[TT][TT][2];
#pragma unroll
        for (int qi = 0; qi < TT; ++qi)
#pragma unroll
            for (int ni = qi; ni < TT; ++ni) tt[qi][ni][0] = tt[qi][ni][1] = 0.0;
        {
            const double *gb0 = s.AB + g8;
#pragma unroll
            for (int kt = 0; kt < NT; ++kt)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    if (LASTNAT && kt == NT - 1 && e == 1) continue;
                    int r = kt * 8 + 2 * c4 + e;
                    if (LASTNAT && kt == NT - 1) r = kt * 8 + c4;
                    if (kt == NT - 1 && N % 8 != 0) r = r < N ? r : KR - 1;
                    double gb[TT];
#pragma unroll
                    for (int ni = 0; ni < TT; ++ni) gb[ni] = gb0[r * LDG + ni * 8];
#pragma unroll
                    for (int qi = 0; qi < TT; ++qi) {
                        double a = w[qi][kt][e];
                        if (LASTNAT && kt == NT - 1) {
                            // natural step of the last tile: index 8 kt + c4 is held by lane (g8, c4 / 2) in element c4 % 2
                            // (in the first product that tile was accumulated in the natural order too, so element e of
                            // lane c4' holds column 8 kt + 2 c4' + e as everywhere else)
                            const int src = (lane & ~3) | (c4 >> 1);
                            const double a0 = __shfl_sync(FULL, w[qi][kt][0], src), a1 = __shfl_sync(FULL, w[qi][kt][1], src);
                            a = (c4 & 1) ? a1 : a0;
                        }
#pragma unroll
                        for (int ni = qi; ni < TT; ++ni) dmma(tt[qi][ni], a, gb[ni]);
                    }
                }
        }
        // ---- publish the control columns: T12[i][a] (i < N) -> T21[a][i], T22 -> S (upper part, mirrored)
#pragma unroll
        for (int a = 0; a < M; ++a) {
            const int ja = N + a, na = ja / 8, ca = (ja % 8) / 2, ea = ja % 2;   // constants after unrolling
            if (c4 == ca) {
#pragma unroll
                for (int qi = 0; qi < TT; ++qi) {
                    if (qi <= na) {
                        const int i = qi * 8 + g8;
                        const double v = tt[qi][na][ea];
                        if (qi * 8 + 7 < N || i < N) s.T21[a * N + i] = v;
                        else if (i <= ja) {
                            s.S[(i - N) * M + a] = v;
                            s.S[a * M + (i - N)] = v;
                        }
                    }
                }
            }
        }
        __syncwarp();
        // S = R~ + rho/2 + B~^T P B~ ; invert (every lane redundantly, M <= 3)
        double Sm[M][M], Si[M][M];
        const double *Rt = qp.R + t * qp.r_stride;
#pragma unroll
        for (int a = 0; a < M; ++a) {
            const bool fa = mk[a] != 0;
#pragma unroll
            for (int b = 0; b < M; ++b) {
                const bool fb = mk[b] != 0;
                double v = s.S[a * M + b];
                if (fa || fb) v = (a == b) ? 1.0 : 0.0;
                else v += Rt[a * M + b] + (a == b ? rho_half : 0.0);
                Sm[a][b] = v;
            }
        }
        spd_inverse<M>(Sm, Si);
        if (lane == 0) {
#pragma unroll
            for (int a = 0; a < M; ++a)
#pragma unroll
                for (int b = 0; b < M; ++b) rec[R_::SINV + a * M + b] = Si[a][b];
        }
        if (lane < N) {
#pragma unroll
            for (int a = 0; a < M; ++a) {
                double kv = 0.0;
#pragma unroll
                for (int b = 0; b < M; ++b) kv = fma(Si[a][b], s.T21[b * N + lane], kv);
                if (!RED) rec[R_::K + R_::pair(a, lane)] = kv;
                s.W[a * N + lane] = kv;
            }
        }
        __syncwarp();
        if (RED && lane < CF::N) {
            // back to the realified record: x_j = w_j y_co(j) with w_j in {1, 1/2, -1/2, 0}
#pragma unroll
            for (int a = 0; a < M; ++a) rec[R_::K + R_::pair(a, lane)] = h_wt == 0.0 ? 0.0 : h_wt * s.W[a * N + h_co];
            rec[R_::DV + lane] = h_wt == 0.0 ? 0.0 : h_wt * dvb[h_co];
        }
        // ---- P_t = Qbar_t + T11 - T21^T K on the accumulator fragments; upper block triangle + mirror image
        const double *Qt = Qfac + t * qp.q_stride;
#pragma unroll
        for (int qi = 0; qi < NT; ++qi) {
            const int i = qi * 8 + g8;
            const int ic = i < N ? i : N - 1;
            double t21[M];
#pragma unroll
            for (int a = 0; a < M; ++a) t21[a] = s.T21[a * N + ic];
#pragma unroll
            for (int ni = qi; ni < NT; ++ni) {
                const int j0 = ni * 8 + 2 * c4;
                const int jc = j0 < N ? j0 : N - 2;     // N is even: the pair (j0, j0 + 1) is inside or outside together
                double v0 = tt[qi][ni][0], v1 = tt[qi][ni][1];
#pragma unroll
                for (int a = 0; a < M; ++a) {
                    const double2 kp = *reinterpret_cast<const double2 *>(s.W + a * N + jc);
                    v0 = fma(-t21[a], kp.x, v0);
                    v1 = fma(-t21[a], kp.y, v1);
                }
                const bool in = i < N && j0 < N;
                if (qp.q_diag) {
                    if (ni == qi) {
                        const double qd = Qt[ic * N + ic];
                        v0 += (i == j0) ? qd : 0.0;
                        v1 += (i == j0 + 1) ? qd : 0.0;
                    }
                } else {
                    v0 += Qt[ic * N + jc];
                    v1 += Qt[ic * N + jc + 1];
                }
                if (ni > qi) {
                    // off-diagonal tile: whole pair + its transpose (padding stays zero)
                    if (in) {
                        *reinterpret_cast<double2 *>(s.P + i * LDP + j0) = make_double2(v0, v1);
                        s.P[j0 * LDP + i] = v0;
                        s.P[(j0 + 1) * LDP + i] = v1;
                    }
                } else {
                    // diagonal tile: the elements on or above the diagonal, each with its mirror image
                    if (in && i <= j0) {
                        s.P[i * LDP + j0] = v0;
                        s.P[j0 * LDP + i] = v0;
                    }
                    if (in && i <= j0 + 1) {
                        s.P[i * LDP + j0 + 1] = v1;
                        s.P[(j0 + 1) * LDP + i] = v1;
                    }
                }
            }
        }
    }
    __syncwarp();
}

// The factor a QP runs: Hermitian coordinates when the instantiation has them and the QP's premise holds (qp.herm, set
// per QP by the closed loop), else realified.  Counted per member.
template <class CF, bool FUSED>
__device__ __forceinline__ void factor(SlabRef sr, const StageOps &ops, const QPData &qp, double rho_half, bool masked,
                                       int lane, Counters &cnt) {
    if constexpr (CF::HERM && FUSED) {
        if (qp.herm) {
            riccati_factor<CF, HermCfg<CF>, FUSED>(sr, ops, qp, rho_half, masked, lane);
            cnt.fac_herm++;
            return;
        }
    }
    riccati_factor<CF, CF, FUSED>(sr, ops, qp, rho_half, masked, lane);
    cnt.fac_full++;
}

// stage record t of the workspace -> slot (t & 1) of the record ring in the [P | G] buffers
template <class CF> __device__ __forceinline__ double *rec_slot(const Slab<CF> &s, int t) {
    return s.recring + (t & 1) * Rec<CF>::SLOT;
}
template <class CF>
__device__ __forceinline__ void prefetch_stage(const Slab<CF> &s, const SlabRef &sr, int t, int lane) {
    prefetch_block<Rec<CF>::SIZE>(rec_slot<CF>(s, t), ws_rec<CF>(sr, t), lane);
}

// ---------------------------------------------------------------------------------------------------------
// Vector sweeps.  One routine, three modes (one copy of the code in the instruction cache):
//   SWEEP_ADMM    backward costate + forward rollout of the ADMM u-update (mask must be all zero)
//   SWEEP_POLISH  the same with the controls of the working set (mask != 0) pinned to their bound
//   SWEEP_ADJOINT backward only: adjoint gradient of the condensed cost at the last rollout -> kk, returns max |grad|
//                 lam_H = 2 Qf (x_H - r_H);  grad_t = 2 R (u_t - ub_t) + B_t^T lam_{t+1};
//                 lam_t = 2 Q (x_t - r_t) + A_t^T lam_{t+1}          (diagonal costs; else adjoint_gradient())
//   SWEEP_REFINE  one step of iterative refinement of the polish solve: the correction (du, dx) that cancels the
//                 gradient left in kk on the free controls (same factorisation, homogeneous dynamics, x0 = 0) is
//                 ADDED to Uo, Xo and the records' x - r
// All three are the recursion  v = dv + p;  g = B^T v - h;  p <- A^T v - q - K^T g  with different (dv, h, q, K).
// A pre-pass folds the control-space terms into one array hl: the linear term h of a free control, the bound of a
// pinned one.  Stage records arrive through the ring one stage ahead; the per-lane scalars needed before the
// stage's only warp sync are register-prefetched.  Writes Uo and, if WRITE_X, Xo (workspace).
// ---------------------------------------------------------------------------------------------------------
enum { SWEEP_ADMM = 0, SWEEP_POLISH = 1, SWEEP_ADJOINT = 2, SWEEP_REFINE = 3 };

template <class CF, bool FUSED, bool REFINE = false>
__device__ __noinline__ double riccati_solve(SlabRef sr, const QPData &qp_in, double rho_half, int mode, bool WRITE_X,
                                             int lane) {
    constexpr int C = CF::C, N = CF::N, M = CF::M;
    using R_ = Rec<CF>;
    const Slab<CF> s = slab_view<CF>(sr);
    const QPData qp = localize<FUSED>(qp_in);
    const int H = sr.H;
    const bool act = lane < N;
    const int vix = (N + M <= 32) ? sweep_idx<CF>(lane) : lane;   // layout of the sweep vectors (cmatvec_ext)
    // the refinement variant is a separate (cold) instantiation: the hot copy stays small for the instruction cache
    const bool adj = !REFINE && mode == SWEEP_ADJOINT, refine = REFINE;
    double *Xo = ws_Xo<CF>(sr);
    prefetch_stage<CF>(s, sr, H - 1, lane);
#pragma unroll 1
    for (int e = lane; e < H * M; e += 32) {
        const int t = e / M, i = e % M;
        const double *Rt = qp.R + t * qp.r_stride;
        double h;
        if (mode == SWEEP_ADMM) {
            h = qp.Rub[e] + rho_half * (s.z[e] - s.y[e]);
        } else if (refine) {
            h = s.mask[e] ? 0.0 : -0.5 * s.kk[e];   // cost term g^T du = -2 h^T du; a pinned control does not move
        } else if (adj) {
            h = 0.0;
#pragma unroll
            for (int j = 0; j < M; ++j) h = fma(-2.0 * Rt[i * M + j], s.Uo[t * M + j] - qp.ub[t * M + j], h);
        } else {
            // h_F = R_FF ub_F - R_F,fix (b - ub_fix); a pinned control gets its bound
            const int mi = s.mask[e];
            if (mi) {
                h = mi == 1 ? box_lo(s, qp.sat, t, i) : box_hi(s, qp.sat, t, i);
            } else {
                h = 0.0;
#pragma unroll
                for (int j = 0; j < M; ++j) {
                    const int mk = s.mask[t * M + j];
                    const double ubj = qp.ub[t * M + j];
                    h += mk ? -Rt[i * M + j] * ((mk == 1 ? box_lo(s, qp.sat, t, j) : box_hi(s, qp.sat, t, j)) - ubj)
                            : Rt[i * M + j] * ubj;
                }
            }
        }
        s.hl[e] = h;
    }
    // q_t per lane: Qbar_t r_t (table, register-prefetched) for the Riccati modes; the adjoint takes
    // -2 Qbar_t (x_t - r_t) (diagonal Qbar) from the record, where the last rollout left x_t - r_t
    double p = 0.0, dv_n = 0.0, ql_n = 0.0;
    if (act && !refine) {
        p = adj ? 2.0 * qp.Qf[lane * N + lane] * s.xT[lane] : -qp.qlinf[lane];
        if (!adj) {
            dv_n = ws_rec<CF>(sr, H - 1)[R_::DV + lane];
            ql_n = qp.qlin[(H - 1) * N + lane];
        }
    }
    if (REFINE) __syncwarp();   // hl has been derived from kk before the backward sweep overwrites kk
#pragma unroll 1
    for (int t = H - 1; t >= 0; --t) {
        const double *slot = rec_slot<CF>(s, t);
        const double2 *At = reinterpret_cast<const double2 *>(slot + R_::AT);
        double *vec = (t & 1) ? s.vb : s.va;
        const double v = dv_n + p;
        double ql = ql_n;
        if (act) vec[vix] = v;
        if (t > 0 && act && !adj && !refine) {
            dv_n = ws_rec<CF>(sr, t - 1)[R_::DV + lane];
            ql_n = qp.qlin[(t - 1) * N + lane];
        }
        cp_async_wait_all();
        __syncwarp();
        if (t > 0) prefetch_stage<CF>(s, sr, t - 1, lane);
        if (adj && act) ql = -2.0 * qp.Q[t * qp.q_stride + lane * N + lane] * slot[R_::XC + lane];
        // control-space operands first: their latency hides behind the mat-vec
        int mk[M];
        double hv[M], kq[M];
#pragma unroll
        for (int i = 0; i < M; ++i) {
            mk[i] = adj ? 0 : s.mask[t * M + i];
            hv[i] = s.hl[t * M + i];
            kq[i] = (!adj && act) ? slot[R_::K + R_::pair(i, lane)] : 0.0;
        }
        double g[M], atv;
        if constexpr (N + M <= 32) {
            atv = cmatvec_ext<CF, true>(At, reinterpret_cast<const double2 *>(slot + R_::B), vec, lane);
#pragma unroll
            for (int i = 0; i < M; ++i) g[i] = __shfl_sync(FULL, atv, N + i);
        } else {
#pragma unroll
            for (int i = 0; i < M; ++i) g[i] = act ? slot[R_::B + R_::pair(i, lane)] * v : 0.0;
            warp_sum_vec<M>(g, lane);
            atv = cmatvec<CF, true, R_::CA>(At, vec, lane);
        }
#pragma unroll
        for (int i = 0; i < M; ++i) {
            g[i] = mk[i] ? 0.0 : g[i] - hv[i];
        }
        double pn = atv - ql;
        if (lane < M) {
            double kkv = 0.0;
#pragma unroll
            for (int b = 0; b < M; ++b) kkv = fma(adj ? (b == lane ? 1.0 : 0.0) : slot[R_::SINV + lane * M + b], g[b], kkv);
            s.kk[t * M + lane] = kkv;
        }
#pragma unroll
        for (int a = 0; a < M; ++a) pn = fma(-kq[a], g[a], pn);
        p = pn;
    }
    __syncwarp();   // kk complete; va/vb free again
    if (adj) {      // max |grad| over the horizon
        double gm = 0.0;
#pragma unroll 1
        for (int e = lane; e < H * M; e += 32) gm = fmax(gm, fabs(s.kk[e]));
        return warp_max(gm);
    }
    // forward: record 0 is still in slot 0
    double x = (act && !refine) ? s.x0[lane] : 0.0;
    double dumax = 0.0;   // REFINE: largest correction of a control (its convergence measure)
    if (WRITE_X && act && !refine) Xo[lane] = x;
    double r_n = (WRITE_X && act && !refine) ? qp.r[lane] : 0.0;   // target of the stage, register-prefetched
#pragma unroll 1
    for (int t = 0; t < H; ++t) {
        const double *slot = rec_slot<CF>(s, t);
        const double2 *At = reinterpret_cast<const double2 *>(slot + R_::AT);
        double *vec = (t & 1) ? s.vb : s.va;
        if (act) {
            vec[vix] = x;
            if (refine) {
                ws_rec<CF>(sr, t)[R_::XC + lane] += x;
            } else if (WRITE_X) {
                ws_rec<CF>(sr, t)[R_::XC + lane] = x - r_n;
                r_n = qp.r[(t + 1) * N + lane];
            }
        }
        if (t > 0) cp_async_wait_all();   // record 0 is still in its slot from the backward sweep
        __syncwarp();
        if (t + 1 < H) prefetch_stage<CF>(s, sr, t + 1, lane);
        int mk[M];
        double hv[M], bq[M];
        const double dq = (act && !refine) ? slot[R_::D + lane] : 0.0;
#pragma unroll
        for (int a = 0; a < M; ++a) {
            mk[a] = s.mask[t * M + a];
            hv[a] = mk[a] ? s.hl[t * M + a] : -s.kk[t * M + a];
            bq[a] = act ? slot[R_::B + R_::pair(a, lane)] : 0.0;
        }
        double u[M], ax;
        if constexpr (N + M <= 32) {
            ax = cmatvec_ext<CF, false>(At, reinterpret_cast<const double2 *>(slot + R_::K), vec, lane);
#pragma unroll
            for (int a = 0; a < M; ++a) u[a] = __shfl_sync(FULL, ax, N + a);
        } else {
#pragma unroll
            for (int a = 0; a < M; ++a) u[a] = act ? slot[R_::K + R_::pair(a, lane)] * x : 0.0;
            warp_sum_vec<M>(u, lane);
            ax = cmatvec<CF, false, R_::CA>(At, vec, lane);
        }
#pragma unroll
        for (int a = 0; a < M; ++a) u[a] = mk[a] ? hv[a] : hv[a] - u[a];
        if (lane < M) {
            double uv = u[0];
#pragma unroll
            for (int a = 1; a < M; ++a) uv = (lane == a) ? u[a] : uv;
            s.Uo[t * M + lane] = refine ? s.Uo[t * M + lane] + uv : uv;
            if (refine) dumax = fmax(dumax, fabs(uv));
        }
        if (act) {
            double xn = ax + dq;
#pragma unroll
            for (int a = 0; a < M; ++a) xn = fma(bq[a], u[a], xn);
            x = xn;
            if (refine) Xo[(t + 1) * N + lane] += x;
            else if (WRITE_X) Xo[(t + 1) * N + lane] = x;
        }
    }
    if (act) s.xT[lane] = refine ? s.xT[lane] + x : x - (WRITE_X ? r_n : qp.r[H * N + lane]);
    __syncwarp();
    // a non-finite state anywhere in the rollout propagates to x_H
    const bool bad = __any_sync(FULL, !isfinite(x));
    if (refine) return bad ? -1.0 : warp_max(dumax);   // size of the correction (negative: non-finite)
    return bad ? 1.0 : 0.0;
}

// (Qbar v)[lane] for v in shared memory
template <class CF>
__device__ __forceinline__ double apply_Q(const double *Qm, int q_diag, const double *v, int lane) {
    constexpr int N = CF::N;
    if (lane >= N) return 0.0;
    if (q_diag) return Qm[lane * N + lane] * v[lane];
    double a0 = 0.0, a1 = 0.0;
#pragma unroll
    for (int j = 0; j < N; j += 2) {
        a0 = fma(Qm[j * N + lane], v[j], a0);
        a1 = fma(Qm[(j + 1) * N + lane], v[j + 1], a1);
    }
    return a0 + a1;
}

// ---------------------------------------------------------------------------------------------------------
// Adjoint gradient of the condensed cost at (Xo, Uo) -> s.kk[t*M+i] (re-used as scratch); returns max |grad|.
//   lam_H = 2 Qf (x_H - r_H);  grad_t = 2 R (u_t - ub_t) + B_t^T lam_{t+1};  lam_t = 2 Q (x_t - r_t) + A_t^T lam_{t+1}
// General (non-diagonal cost) version; the diagonal case runs as a mode of riccati_solve.
// B_t, A_t through the ring, x_t - r_t register-prefetched; vectors double-buffered (va/vb, and P as scratch).
// ---------------------------------------------------------------------------------------------------------
template <class CF, bool FUSED>
__device__ __noinline__ double adjoint_gradient(SlabRef sr, const QPData &qp_in, int lane) {
    constexpr int C = CF::C, N = CF::N, M = CF::M;
    using R_ = Rec<CF>;
    const Slab<CF> s = slab_view<CF>(sr);
    const QPData qp = localize<FUSED>(qp_in);
    const int H = sr.H;
    const bool act = lane < N;
    const double *Xo = ws_Xo<CF>(sr);
    prefetch_stage<CF>(s, sr, H - 1, lane);
    double xd_n = act ? Xo[(H - 1) * N + lane] - qp.r[(H - 1) * N + lane] : 0.0;
    if (act) s.xd[lane] = Xo[H * N + lane] - qp.r[H * N + lane];
    __syncwarp();
    double lam = 2.0 * apply_Q<CF>(qp.Qf, qp.q_diag, s.xd, lane);
    double gmax = 0.0;
    __syncwarp();
#pragma unroll 1
    for (int t = H - 1; t >= 0; --t) {
        const double *Bt = rec_slot<CF>(s, t) + R_::B;
        const double2 *At = reinterpret_cast<const double2 *>(rec_slot<CF>(s, t) + R_::AT);
        const double *Rt = qp.R + t * qp.r_stride;
        double *lamv = (t & 1) ? s.vb : s.va;
        double *xdv = s.xd + (t & 1) * N;
        const double xd = xd_n;
        if (act) {
            lamv[lane] = lam;
            xdv[lane] = xd;
            if (t > 0) xd_n = Xo[(t - 1) * N + lane] - qp.r[(t - 1) * N + lane];
        }
        cp_async_wait_all();
        __syncwarp();
        if (t > 0) prefetch_stage<CF>(s, sr, t - 1, lane);
        double g[M];
#pragma unroll
        for (int i = 0; i < M; ++i) g[i] = act ? Bt[R_::pair(i, lane)] * lam : 0.0;
        warp_sum_vec<M>(g, lane);
#pragma unroll
        for (int i = 0; i < M; ++i) {
#pragma unroll
            for (int j = 0; j < M; ++j) g[i] = fma(2.0 * Rt[i * M + j], s.Uo[t * M + j] - qp.ub[t * M + j], g[i]);
            gmax = fmax(gmax, fabs(g[i]));
        }
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < M; ++i) s.kk[t * M + i] = g[i];
        }
        const double atl = cmatvec<CF, true, R_::CA>(At, lamv, lane);
        lam = atl + 2.0 * apply_Q<CF>(qp.Q + t * qp.q_stride, qp.q_diag, xdv, lane);
    }
    __syncwarp();
    return gmax;
}

// ---------------------------------------------------------------------------------------------------------
// One ADMM block on the control box (u = z, z in [lo, hi]) down to residual eps; cold in the tight mode (it only
// re-seeds the working set when the active-set rounds do not settle), hence a function of its own: the hot loop of
// qp_solve stays small for the instruction cache.
// ---------------------------------------------------------------------------------------------------------
template <class CF, bool FUSED>
__device__ __noinline__ void admm_block(SlabRef sr, const StageOps &ops_in, const QPData &qp_in, const QPSet &set,
                                        double eps, int lane, Counters &cnt) {
    constexpr int M = CF::M;
    const Slab<CF> s = slab_view<CF>(sr);
    const QPData qp = localize<FUSED>(qp_in);
    const int HM = sr.H * M;
    const double rho_half = 0.5 * set.rho;
#pragma unroll 1
            for (int e = lane; e < HM; e += 32) s.mask[e] = 0;   // the sweeps read the working set: none in ADMM
            __syncwarp();
            // rho is adapted like OSQP does (optimize.py:59 -> OSQP's adaptive_rho): at a few check points the penalty
            // is rescaled by sqrt(normalised primal residual / normalised dual residual) when that ratio is far from
            // one, the scaled dual y follows, and the Riccati factorisation is redone with the new rho.
            double rho = set.rho, rh = rho_half;
            factor<CF, FUSED>(sr, ops_in, qp_in, rh, false, lane, cnt);
            cnt.factor++;
            int next_check = 5;
            for (int it = 0; it < set.max_admm; ++it) {
                riccati_solve<CF, FUSED>(sr, qp_in, rh, SWEEP_ADMM, !set.polish, lane);
                cnt.admm++;
                bool bad = false;
                double rp = 0.0, rd = 0.0, nu = 0.0, ny = 0.0;
#pragma unroll 1
                for (int e = lane; e < HM; e += 32) {
                    const int t = e / M, i = e % M;
                    const double u = s.Uo[e], zo = s.z[e];
                    const double uh = set.alpha * u + (1.0 - set.alpha) * zo;
                    const double zn = fmin(fmax(uh + s.y[e], box_lo(s, qp.sat, t, i)), box_hi(s, qp.sat, t, i));
                    const double yn = s.y[e] + uh - zn;
                    s.y[e] = yn;
                    s.z[e] = zn;
                    bad |= !(fabs(u - zn) < eps) || !(rho * fabs(zn - zo) < eps);
                    rp = fmax(rp, fabs(u - zn));
                    rd = fmax(rd, fabs(zn - zo));
                    nu = fmax(nu, fmax(fabs(u), fabs(zn)));
                    ny = fmax(ny, fabs(yn));
                }
                __syncwarp();
                if (!__any_sync(FULL, bad)) break;   // warp vote: every lane's slice of the residuals is below eps
                if (set.adaptive_rho && it + 1 == next_check && it + 1 < set.max_admm) {
                    next_check = 2 * next_check + 5;
                    rp = warp_max(rp);
                    rd = warp_max(rd);
                    nu = warp_max(nu);
                    ny = warp_max(ny);
                    // both residuals relative to the size of what they are residuals of (u = z; the dual rho y)
                    const double pr = rp / fmax(nu, 1e-12), dr = rd / fmax(ny, 1e-12);
                    double ratio = sqrt(fmax(pr, 1e-12) / fmax(dr, 1e-12));
                    ratio = fmin(fmax(ratio, 0.05), 20.0);
                    const double rho_new = fmin(fmax(rho * ratio, 1e-6), 1e6);
                    if (rho_new > 5.0 * rho || rho_new < 0.2 * rho) {
                        const double sc = rho / rho_new;
#pragma unroll 1
                        for (int e = lane; e < HM; e += 32) s.y[e] *= sc;
                        __syncwarp();
                        rho = rho_new;
                        rh = 0.5 * rho;
                        factor<CF, FUSED>(sr, ops_in, qp_in, rh, false, lane, cnt);
                        cnt.factor++;
                    }
                }
            }
            if (rho != set.rho) {   // hand y over in the units of the configured rho (warm start of the next solve)
                const double sc = rho / set.rho;
#pragma unroll 1
                for (int e = lane; e < HM; e += 32) s.y[e] *= sc;
                __syncwarp();
            }
        }

}   // namespace m4q
#include "m4q_kkt.cuh"
namespace m4q {

// ---------------------------------------------------------------------------------------------------------
// The QP (optimize.py:12-60).  Two building blocks share the Riccati kernels:
//   * ADMM on the control box (u = z, z in [lo, hi]); u-update = equality-constrained LQ problem solved exactly by
//     the time-varying Riccati recursion; convergence by warp vote over each lane's slice of the residuals.
//   * primal-dual active set ("polish"): controls in the working set are pinned to their bound and folded into
//     the dynamics, one masked Riccati factor + solve gives the equality-constrained optimum, and an adjoint
//     gradient certifies the KKT conditions (multiplier signs on pinned controls, feasibility of free ones) or
//     updates the set.  The certificate is a full KKT check: stationarity of the free controls (1e-8 relative),
//     primal feasibility (1e-12), multiplier signs (1e-10 relative).
// Tight mode (polish = 1): the working set is warm-started from the previous solve's (z, y) -- the previous SQP
// iterate or the shifted previous MPC step -- and the active-set rounds run first; an ADMM block (which needs no
// guess) is the fallback that re-seeds the set when the rounds do not certify.  admm_first = 1 always runs the ADMM
// block before the rounds.  polish = 0 is plain ADMM to residual eps (OSQP-equivalent mode).
// In: slab {B, D, phi, x0, lo0, hi0, z, y(warm)}.  Out: Xo, Uo; z, y updated.  Returns status 0 / 2 / 3.
// ---------------------------------------------------------------------------------------------------------
template <class CF, bool FUSED>
__device__ int qp_solve(SlabRef sr, const StageOps &ops_in, const QPData &qp_in, const QPSet &set, int lane, Counters &cnt) {
    constexpr int N = CF::N, M = CF::M;
    const Slab<CF> s = slab_view<CF>(sr);
    const StageOps ops = localize<FUSED>(ops_in);
    const QPData qp = localize<FUSED>(qp_in);
    const int H = sr.H;
    const int HM = H * M;
    const double rho_half = 0.5 * set.rho;
    // clip the warm start into the current box
#pragma unroll 1
    for (int e = lane; e < HM; e += 32) {
        const int t = e / M, i = e % M;
        s.z[e] = fmin(fmax(s.z[e], box_lo(s, qp.sat, t, i)), box_hi(s, qp.sat, t, i));
        s.flips[e] = 0;
    }
    __syncwarp();
    cnt.solves++;
    double eps = set.eps;
    int status = 0;
    bool x_nonfinite = false;   // a non-finite state of the reported rollout (it propagates to x_H)
    bool run_admm = !set.polish || set.admm_first;
    const bool kkt_ok = set.kkt != nullptr && set.kkt_mode > 0 && set.polish;
    for (;;) {
        if (kkt_ok && ((set.kkt_mode >= 2 && cnt.sticky) || set.kkt_mode >= 4)) {
            // an earlier QP of this member needed the pivoted KKT solve (cost-to-go beyond fp64: order-1 model at long
            // horizons): go straight to it.  One factor call forms the stage operators A_t in the records.
            riccati_factor<CF, CF, FUSED>(sr, ops_in, qp_in, 0.0, false, lane);
            cnt.fac_full++;
            status = kkt_active_set<CF, FUSED>(sr, qp_in, set, lane, cnt);
            break;
        }
        if (run_admm) admm_block<CF, FUSED>(sr, ops_in, qp_in, set, eps, lane, cnt);
        if (!set.polish) {
            // OSQP-equivalent mode: report the feasible iterate z and its rollout
#pragma unroll 1
            for (int e = lane; e < HM; e += 32) s.Uo[e] = s.z[e];
            __syncwarp();
            double *Xo = ws_Xo<CF>(sr);
            double x = (lane < N) ? s.x0[lane] : 0.0;
            if (lane < N) Xo[lane] = x;
#pragma unroll 1
            for (int t = 0; t < H; ++t) {
                const double *rec = ws_rec<CF>(sr, t);
                if (lane < N) s.va[lane] = x;
                __syncwarp();
                if (lane < ops.nblk) s.xd[lane] = stage_weight<M>(ops, s.Ug + t * M, lane);
                __syncwarp();
                const double ax = apply_A<CF>(ops, s.xd, t, s.va, lane);
                if (lane < N) {
                    double xn = ax + rec[Rec<CF>::D + lane];
#pragma unroll
                    for (int a = 0; a < M; ++a) xn = fma(rec[Rec<CF>::B + Rec<CF>::pair(a, lane)], s.Uo[t * M + a], xn);
                    x = xn;
                    Xo[(t + 1) * N + lane] = x;
                }
                __syncwarp();
            }
            x_nonfinite = __any_sync(FULL, !isfinite(x));
            break;
        }
        // ---- working set from the (z, y) estimate: at a bound with the multiplier pushing outwards
#pragma unroll 1
        for (int e = lane; e < HM; e += 32) {
            const int t = e / M, i = e % M;
            const double zz = s.z[e], yy = s.y[e];
            int mk = 0;
            if (zz <= box_lo(s, qp.sat, t, i) && yy < 0.0) mk = 1;
            else if (zz >= box_hi(s, qp.sat, t, i) && yy > 0.0) mk = 2;
            s.mask[e] = mk;
        }
        __syncwarp();
        bool certified = false;
        bool numeric = false;   // the rounds ended on a settled working set whose solve is not stationary, or not finite
        for (int round = 0; round < set.max_polish; ++round) {
            factor<CF, FUSED>(sr, ops_in, qp_in, 0.0, true, lane, cnt);
            cnt.factor++;
            cnt.polish++;
            x_nonfinite = riccati_solve<CF, FUSED>(sr, qp_in, 0.0, SWEEP_POLISH, true, lane) != 0.0;
            double gmax = qp.q_diag ? riccati_solve<CF, FUSED>(sr, qp_in, 0.0, SWEEP_ADJOINT, false, lane)
                                    : adjoint_gradient<CF, FUSED>(sr, qp_in, lane);
            bool stable = false;
            double du_last = -1.0;   // size of the last refinement correction (< 0: none yet)
#pragma unroll 1
            for (int rf = 0;; ++rf) {
                const double gs = fmax(1.0, gmax);
                // strict certificate first; once the ADMM re-seeding has been tightened below 1e-6 without settling the
                // working set (a multiplier or a control within round-off of zero / of its bound keeps flipping), the
                // same tests are applied with tolerances 1e4 times wider -- still a KKT point to 1e-6 relative
                const double rx = eps <= 1e-6 ? 1e4 : 1.0;
                bool changed = false, visible = false, unstationary = false, rough = false;
                double umax = 0.0;
#pragma unroll 1
                for (int e = lane; e < HM; e += 32) {
                    const int t = e / M, i = e % M;
                    const int mk = s.mask[e];
                    const double u = s.Uo[e], g = s.kk[e];
                    const double lo = box_lo(s, qp.sat, t, i), hi = box_hi(s, qp.sat, t, i);
                    int nm = mk;
                    umax = fmax(umax, fabs(u));
                    if (mk == 0) {
                        if (u < lo - 1e-12 * rx) nm = 1;
                        else if (u > hi + 1e-12 * rx) nm = 2;
                        // stationarity of a free control: exact up to the round-off of the Riccati solve, unless the
                        // cost-to-go is badly scaled (long horizons with the order-1 model, DESIGN.md section 2.3)
                        visible |= !(fabs(g) <= 1e-9 * gs);
                        unstationary |= !(fabs(g) <= 1e-8 * gs);
                        rough |= !(fabs(g) <= 1e-5 * gs);
                    } else {
                        // A weakly active bound (multiplier within the evaluation noise of zero) would otherwise be
                        // released, violated, pinned and released again for ever: a control that has come back twice
                        // stays pinned unless its multiplier is negative beyond that noise.
                        const double gn = mk == 1 ? -g : g;       // > 0: the multiplier has the wrong sign
                        if (gn > 1e-10 * rx * gs) {
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
                if (__any_sync(FULL, changed)) break;   // the working set moved: next round
                // Same working set again: certified if the free controls are stationary.  A visible gradient means the
                // Riccati solve lost accuracy (ill-conditioned cost-to-go): iterative refinement with the same
                // factorisation (feedback form: the correction is rolled out through A - B K, so it does not
                // re-amplify).  The adjoint gradient itself is evaluated through the unstable open-loop dynamics and
                // has a noise floor of ~ eps * ||prod A_t||^2; once the refinement has CONVERGED (its correction is
                // below 1e-9 of the control scale) what is left of the gradient is that evaluation noise, and the point
                // is the optimum of the working set to the accuracy fp64 offers -- accepted if the residual gradient is
                // small (1e-5 relative), which a wrong factorisation would not produce.
                const bool vis = __any_sync(FULL, visible), unst = __any_sync(FULL, unstationary);
                if (!vis) {
                    stable = certified = true;
                    break;
                }
                if (du_last >= 0.0 && du_last <= 1e-9 * fmax(1.0, warp_max(umax)) && !__any_sync(FULL, rough)) {
                    stable = certified = true;
                    break;
                }
                if (rf == 6) {
                    stable = true;
                    certified = !unst;
                    break;
                }
                du_last = riccati_solve<CF, FUSED, true>(sr, qp_in, 0.0, SWEEP_REFINE, true, lane);
                x_nonfinite = du_last < 0.0;
                if (x_nonfinite) {
                    stable = true;
                    break;
                }
                cnt.admm += 2;   // one correction sweep + one adjoint sweep
                gmax = qp.q_diag ? riccati_solve<CF, FUSED>(sr, qp_in, 0.0, SWEEP_ADJOINT, false, lane)
                                 : adjoint_gradient<CF, FUSED>(sr, qp_in, lane);
            }
            if (stable) {
                numeric = !certified;
                break;
            }
        }
        if (certified) {
            // warm start of the next solve: z = u*, y = the (scaled) multipliers of the pinned controls
            const double inv_rho = 1.0 / set.rho;
#pragma unroll 1
            for (int e = lane; e < HM; e += 32) {
                const int t = e / M, i = e % M;
                s.z[e] = fmin(fmax(s.Uo[e], box_lo(s, qp.sat, t, i)), box_hi(s, qp.sat, t, i));
                s.y[e] = s.mask[e] ? -s.kk[e] * inv_rho : 0.0;
                if (eps <= 1e-6) s.Uo[e] = s.z[e];   // relaxed certificate: a free control may sit 1e-8 outside its bound
            }
            __syncwarp();
            break;
        }
        // not certified: (re)seed with an ADMM block at a tighter tolerance
        if (run_admm) eps *= 0.1;
        run_admm = true;
        // The pivoted KKT solve takes over before the certificate would be relaxed, and (kkt_mode 2) as soon as the Riccati path
        // breaks down NUMERICALLY -- a settled working set whose solve is not stationary or not finite: the cost-to-go
        // has left the fp64 range (order-1 model at H = 100).  A working set that merely keeps moving is the ADMM
        // re-seeding's business.
        bool unstable = false;
        if (kkt_ok && set.kkt_mode >= 2 && !numeric) {
            // ... or the rollout shows that the linearised dynamics are unstable over the horizon (|x_t| grows by more
            // than 1e3: a cost-to-go 1e6 times its O(1) part); the order-2 model at the same horizon stays O(1) and
            // keeps the (much cheaper) ADMM re-seeding
            const double *Xr = ws_Xo<CF>(sr);
            double x0m = 0.0, xm = 0.0;
            bool nf = false;
#pragma unroll 1
            for (int e = lane; e < (H + 1) * N; e += 32) {
                const double v = fabs(Xr[e]);
                nf |= !isfinite(v);
                xm = fmax(xm, v);
                if (e < N) x0m = fmax(x0m, v);
            }
            unstable = __any_sync(FULL, nf) || warp_max(xm) > 1e3 * fmax(warp_max(x0m), 1e-3);
        }
        // (with the KKT solve available the relaxed certificate below is never needed: four ADMM re-seedings, then KKT)
        if (kkt_ok && ((set.kkt_mode >= 2 && (numeric || unstable)) || eps < 3e-6)) {
            if (set.kkt_mode >= 2 && (numeric || unstable)) cnt.sticky = 1;
            status = kkt_active_set<CF, FUSED>(sr, qp_in, set, lane, cnt);
            x_nonfinite = false;
            break;
        }
        if (eps < 1e-10) {
            status = 2;   // could not certify: report the ADMM iterate (reference: solver warning -> exit code 2)
#pragma unroll 1
            for (int e = lane; e < HM; e += 32) s.Uo[e] = s.z[e];
            __syncwarp();
            break;
        }
    }
    // non-finite result -> reference exit code 3 (mpc.py:200-203)
    bool nonfinite = false;
#pragma unroll 1
    for (int e = lane; e < HM; e += 32) nonfinite |= !isfinite(s.Uo[e]);
    if (__any_sync(FULL, nonfinite) || x_nonfinite) status = 3;
    return status;
}

// objective value sum (x-r)^T Q (x-r) + (u-ub)^T R (u-ub)  (optimize.py:34-35, :54; no 1/2)
template <class CF>
__device__ double qp_objective(const SlabRef &sr, const QPData &qp, int lane) {
    constexpr int N = CF::N, M = CF::M;
    const Slab<CF> s = slab_view<CF>(sr);
    const int H = sr.H;
    const double *Xo = ws_Xo<CF>(sr);
    double acc = 0.0;
#pragma unroll 1
    for (int t = 0; t <= H; ++t) {
        __syncwarp();
        if (lane < N) s.vb[lane] = Xo[t * N + lane] - qp.r[t * N + lane];
        __syncwarp();
        const double qv = apply_Q<CF>(t == H ? qp.Qf : qp.Q + t * qp.q_stride, qp.q_diag, s.vb, lane);
        if (lane < N) acc = fma(qv, s.vb[lane], acc);
    }
#pragma unroll 1
    for (int e = lane; e < H * M; e += 32) {
        const int t = e / M, i = e % M;
        const double *Rt = qp.R + t * qp.r_stride;
        double rv = 0.0;
        for (int j = 0; j < M; ++j) rv = fma(Rt[i * M + j], s.Uo[t * M + j] - qp.ub[t * M + j], rv);
        acc = fma(rv, s.Uo[e] - qp.ub[e], acc);
    }
    return warp_sum(acc);
}

// ---------------------------------------------------------------------------------------------------------
// Linearisation of the bilinear model along (Xg, Ug): fills phi (slab) and B, D (stage records)
// (linearize.py:50-70).
//   B_t[:, i] = sum_k pow[k][i] * prod_l u_l^(pow[k][l] - [l == i]) * (N_k x_t);  D_t = -B_t u_t.
// x_t comes from the workspace one stage ahead (register prefetch); the vector and the derivative weights are
// double-buffered, so one warp sync per stage.
// ---------------------------------------------------------------------------------------------------------
// hb != nullptr: also checks that Xg is sigma-conjugate-symmetric (x_sigma(k) = conj(x_k), HermBasis) over all H + 1
// stages to 1e-12 of its largest entry -- the premise of the factor in Hermitian coordinates; returns 1 if it is.
template <class CF, bool FUSED>
__device__ __noinline__ int linearize(SlabRef sr, const StageOps &model_in, const int *pow, int lane, const int *hb) {
    constexpr int C = CF::C, N = CF::N, M = CF::M;
    using R_ = Rec<CF>;
    const Slab<CF> s = slab_view<CF>(sr);
    const StageOps model = localize<FUSED>(model_in);
    const int H = sr.H;
    const int p = model.nblk - 1;
    const double *Xg = ws_Xg<CF>(sr);
    const bool act = lane < N;
    const bool im = lane >= C;
    const int r = im ? lane - C : lane;
    const double sgn = im ? 1.0 : -1.0;
    double x_n = act ? Xg[lane] : 0.0;
    // sigma check: the partner lane holds x_sigma(j), equal to x_j (real part) or -x_j (imaginary part)
    const bool chk = hb != nullptr;
    const int pa = (chk && act) ? hb[HermBasis<CF>::PA + lane] : lane;
    const double hs = im ? -1.0 : 1.0;
    double hdev = 0.0, hmax = 0.0;
    bool hnf = false;
    auto herm_stage = [&](double x) {
        const double xp = __shfl_sync(FULL, x, pa);
        hdev = fmax(hdev, fabs(xp - hs * x));
        hmax = fmax(hmax, fabs(x));
        hnf |= !isfinite(x);
    };
    // order-1 library (phi_k = u_k): the derivative weights are the identity and need not be tabulated per stage
    bool first_order = p == M;
    if (first_order) {
#pragma unroll 1
        for (int e = 0; e < M * M; ++e) first_order &= pow[e] == ((e / M == e % M) ? 1 : 0);
    }
#pragma unroll 1
    for (int t = 0; t < H; ++t) {
        double *dco = s.scr + (t & 1) * (p * M);   // [p][M]
        double *vec = (t & 1) ? s.vb : s.va;
        if (chk) herm_stage(x_n);
        if (act) {
            vec[lane] = x_n;
            if (t + 1 < H) x_n = Xg[(t + 1) * N + lane];
        }
        // derivative weights of the monomials: lane k < p computes its own (the monomials themselves are evaluated where
        // they are used, stage_weight())
        if (!first_order && lane < p) {
            double dw[M];
#pragma unroll
            for (int i = 0; i < M; ++i) dw[i] = (double)pow[lane * M + i];
#pragma unroll
            for (int l = 0; l < M; ++l) {
                const int e = pow[lane * M + l];
                const double ul = s.Ug[t * M + l];
                double pw = 1.0, pwm1 = 1.0;   // u^e and u^(e-1)
#pragma unroll 1
                for (int q = 0; q < e; ++q) {
                    pwm1 = pw;
                    pw *= ul;
                }
#pragma unroll
                for (int i = 0; i < M; ++i) dw[i] *= (i == l) ? (e > 0 ? pwm1 : 0.0) : pw;
            }
#pragma unroll
            for (int i = 0; i < M; ++i) dco[lane * M + i] = dw[i];
        }
        __syncwarp();
        if (act) {
            const double *xp = vec + (im ? C : 0), *xq = vec + (im ? 0 : C);
            double pv[C], qv[C];
#pragma unroll
            for (int j = 0; j < C; ++j) {
                pv[j] = xp[j];
                qv[j] = xq[j];
            }
            double b[M];
#pragma unroll
            for (int i = 0; i < M; ++i) b[i] = 0.0;
            // rows of N_k: [r][j] from the blocks, or (c multiple of 8) [j][r] from the transposed copies
            const bool tr = (C % 8 == 0) && FUSED && model.soffT != 0;
            const double2 *blk = tr ? reinterpret_cast<const double2 *>(dyn_smem() + model.soffT) + r : model.blocks + (C + r) * C;
            const int js = tr ? C : 1;
#pragma unroll 1
            for (int kb = 1; kb <= p; ++kb, blk += C * C) {
                double p0 = 0.0, p1 = 0.0, q0 = 0.0, q1 = 0.0;
#pragma unroll
                for (int j = 0; j < C; ++j) {
                    const double2 m = blk[j * js];
                    if (j & 1) {
                        p1 = fma(m.x, pv[j], p1);
                        q1 = fma(m.y, qv[j], q1);
                    } else {
                        p0 = fma(m.x, pv[j], p0);
                        q0 = fma(m.y, qv[j], q0);
                    }
                }
                const double y = fma(sgn, q0 + q1, p0 + p1);
#pragma unroll
                for (int i = 0; i < M; ++i) b[i] = first_order ? (kb - 1 == i ? y : b[i]) : fma(dco[(kb - 1) * M + i], y, b[i]);
            }
            double *rec = ws_rec<CF>(sr, t);
            double d = 0.0;
#pragma unroll
            for (int i = 0; i < M; ++i) {
                rec[R_::B + R_::pair(i, lane)] = b[i];
                d = fma(-b[i], s.Ug[t * M + i], d);
            }
            rec[R_::D + lane] = d;
        }
    }
    __syncwarp();
    if (!chk) return 0;
    herm_stage(act ? Xg[H * N + lane] : 0.0);
    const double tol = 1e-12 * warp_max(hmax);
    return !__any_sync(FULL, hnf || !(hdev <= tol));
}

// ---------------------------------------------------------------------------------------------------------
// Line search (mpc.py:101-125): alpha = -(M (Zg - Zt)) . DZ / (DZ . M DZ), step = |alpha| ||DZ||_2 with
// M = blockdiag(Qbar_0..Qbar_H, [[R,0],[0,R]]_0..) in TIME-major order while Z is the STATE-major flattening
// [Re X.ravel(), Im X.ravel(), Re U.ravel(), Im U.ravel()] of X [c][H+1], U [m][H].  Reproduced as is.
// X arrays here are [t][N] realified (workspace); r = qp.r.  Z index zeta <-> (t, k):
//   part = zeta / (C*(H+1)), rem = zeta % (C*(H+1)), state = rem / (H+1), t = rem % (H+1), k = part*C + state,
// and zeta belongs to metric block tau = zeta / N, row zeta % N.  Diagonal costs: one coalesced pass in memory
// order; full costs: block by block with gathers.
// ---------------------------------------------------------------------------------------------------------
template <class CF, bool FUSED>
__device__ __noinline__ void line_search(SlabRef sr, const QPData &qp_in, int lane, double &alpha, double &step) {
    constexpr int C = CF::C, N = CF::N, M = CF::M;
    const Slab<CF> s = slab_view<CF>(sr);
    const QPData qp = localize<FUSED>(qp_in);
    const int H = sr.H;
    const double *Xg = ws_Xg<CF>(sr), *Xo = ws_Xo<CF>(sr);
    double num = 0.0, den = 0.0, nrm = 0.0;
    const int H1 = H + 1;
    if (qp.q_diag) {
#pragma unroll 4
        for (int e = lane; e < H1 * N; e += 32) {
            const int t = e / N, k = e % N;
            const int part = k / C, st = k % C;
            const int zeta = (part * C + st) * H1 + t;
            const int tau = zeta / N, row = zeta % N;
            const double *Qt = (tau == H) ? qp.Qf : qp.Q + tau * qp.q_stride;
            const double qd = Qt[row * N + row];
            const double xg = Xg[e];
            const double e_k = xg - qp.r[e], d_k = Xo[e] - xg;
            nrm = fma(d_k, d_k, nrm);
            num = fma(qd * e_k, d_k, num);
            den = fma(qd * d_k, d_k, den);
        }
    } else {
#pragma unroll 1
        for (int tau = 0; tau <= H; ++tau) {
            double e_k = 0.0, d_k = 0.0;
            if (lane < N) {
                const int zeta = tau * N + lane;
                const int part = zeta / (C * H1), rem = zeta % (C * H1);
                const int st = rem / H1, t = rem % H1;
                const int idx = t * N + part * C + st;
                const double xg = Xg[idx];
                e_k = xg - qp.r[idx];
                d_k = Xo[idx] - xg;
                nrm = fma(d_k, d_k, nrm);
            }
            const double *Qt = (tau == H) ? qp.Qf : qp.Q + tau * qp.q_stride;
            __syncwarp();
            if (lane < N) {
                s.va[lane] = e_k;
                s.vb[lane] = d_k;
            }
            __syncwarp();
            if (lane < N) {
                double qe = 0.0, qd = 0.0;
                for (int j = 0; j < N; ++j) {
                    const double qv = Qt[lane * N + j];
                    qe = fma(qv, s.va[j], qe);
                    qd = fma(qv, s.vb[j], qd);
                }
                num = fma(qe, d_k, num);
                den = fma(qd, d_k, den);
            }
        }
    }
    // control part: Z_U = [U.ravel() (index i*H + t), zeros(mH)], blocks tau < H of size 2M: [[R,0],[0,R]]
    const int HM = H * M;
#pragma unroll 1
    for (int tau = 0; tau < H; ++tau) {
        const double *Rt = qp.R + tau * qp.r_stride;
        if (lane < 2 * M) {
            const int a = lane;
            const int blk_row = a / M, ia = a % M;   // block row 0: real rows, 1: imaginary rows
            const int za = tau * 2 * M + a;
            double da = 0.0;
            if (za < HM) {
                const int i = za / H, t = za % H;
                da = s.Uo[t * M + i] - s.Ug[t * M + i];
            }
            double re = 0.0, rd = 0.0;
#pragma unroll 1
            for (int jb = 0; jb < M; ++jb) {
                const int zb = tau * 2 * M + blk_row * M + jb;
                if (zb < HM) {
                    const int i = zb / H, t = zb % H;
                    const double ug = s.Ug[t * M + i];
                    re = fma(Rt[ia * M + jb], ug - qp.ub[t * M + i], re);
                    rd = fma(Rt[ia * M + jb], s.Uo[t * M + i] - ug, rd);
                }
            }
            num = fma(re, da, num);
            den = fma(rd, da, den);
        }
    }
#pragma unroll 1
    for (int e = lane; e < HM; e += 32) {
        const double d = s.Uo[e] - s.Ug[e];
        nrm = fma(d, d, nrm);
    }
    num = warp_sum(num);
    den = warp_sum(den);
    nrm = warp_sum(nrm);
    if (den == 0.0) {   // reference would produce 0/0; treat a vanishing direction as converged
        alpha = 0.0;
        step = 0.0;
    } else {
        alpha = -num / den;
        step = fabs(alpha) * sqrt(nrm);
    }
    __syncwarp();
}

// ---------------------------------------------------------------------------------------------------------
// Small complex matrices for the plant: d <= 4, entries distributed one per lane (lane = i*d + j).
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double2 cmul(double2 a, double2 b) {
    return make_double2(fma(a.x, b.x, -a.y * b.y), fma(a.x, b.y, a.y * b.x));
}
__device__ __forceinline__ double2 cfma(double2 a, double2 b, double2 c) {
    return make_double2(fma(a.x, b.x, fma(-a.y, b.y, c.x)), fma(a.x, b.y, fma(a.y, b.x, c.y)));
}

// out(i,j) = sum_k A[i][k] B[k][j] (lane holds out entry); A, B in shared memory as double2 [d*d]
__device__ __forceinline__ double2 cmm(const double2 *A, const double2 *B, int d, int i, int j) {
    double2 acc = make_double2(0.0, 0.0);
#pragma unroll 1
    for (int k = 0; k < d; ++k) acc = cfma(A[i * d + k], B[k * d + j], acc);
    return acc;
}

// U = expm(-i H dt) for Hermitian-or-not H (d x d) by scaling and squaring of a degree-16 Taylor polynomial.
// Hm, T0, T1: shared scratch [d*d] double2 each.  Result left in T0.  All 32 lanes must call.
__device__ __noinline__ void expm_minus_i(const double2 *Hm, double dt, int d, double2 *G, double2 *T0, double2 *T1, int lane) {
    const int dd = d * d;
    const int i = lane / d, j = lane % d;
    const bool act = lane < dd;
    // G = -i H dt ; 1-norm
    double2 g = make_double2(0.0, 0.0);
    if (act) {
        const double2 h = Hm[lane];
        g = make_double2(h.y * dt, -h.x * dt);
    }
    double colsum = act ? hypot(g.x, g.y) : 0.0;
    // column sums: reduce over i for fixed j
    if (act) T1[lane] = make_double2(colsum, 0.0);
    __syncwarp();
    double nrm = 0.0;
    if (act) {
        double cs = 0.0;
#pragma unroll 1
        for (int k = 0; k < d; ++k) cs += T1[k * d + j].x;
        nrm = cs;
    }
    nrm = warp_max(nrm);
    int sq = 0;
    while (nrm > 0.5 && sq < 40) {
        nrm *= 0.5;
        ++sq;
    }
    const double sc = ldexp(1.0, -sq);
    g.x *= sc;
    g.y *= sc;
    __syncwarp();
    if (act) {
        G[lane] = g;
        T0[lane] = make_double2(i == j ? 1.0 : 0.0, 0.0);
    }
    __syncwarp();
    // Horner: T = I + G/1 (I + G/2 (I + ... (I + G/16)))   (||G|| <= 0.5: remainder 0.5^17/17! ~ 2e-20)
    for (int k = 16; k >= 1; --k) {
        double2 v = make_double2(0.0, 0.0);
        if (act) {
            v = cmm(G, T0, d, i, j);
            const double inv = 1.0 / (double)k;
            v.x = fma(v.x, inv, i == j ? 1.0 : 0.0);
            v.y *= inv;
        }
        __syncwarp();
        if (act) T0[lane] = v;
        __syncwarp();
    }
#pragma unroll 1
    for (int q = 0; q < sq; ++q) {
        double2 v = make_double2(0.0, 0.0);
        if (act) v = cmm(T0, T0, d, i, j);
        __syncwarp();
        if (act) T0[lane] = v;
        __syncwarp();
    }
}

// rho <- U rho U^dagger ; rho in shared (double2 [dd]), U in shared; tmp scratch
__device__ __noinline__ void conjugate(double2 *rho, const double2 *U, int d, double2 *tmp, int lane) {
    const int dd = d * d;
    const int i = lane / d, j = lane % d;
    const bool act = lane < dd;
    if (act) tmp[lane] = cmm(U, rho, d, i, j);
    __syncwarp();
    double2 v = make_double2(0.0, 0.0);
    if (act) {
#pragma unroll 1
        for (int k = 0; k < d; ++k) {
            const double2 uc = U[j * d + k];
            v = cfma(tmp[i * d + k], make_double2(uc.x, -uc.y), v);
        }
    }
    __syncwarp();
    if (act) rho[lane] = v;
    __syncwarp();
}

// ---------------------------------------------------------------------------------------------------------
// Exact discretisation of the bilinear generator (SURVEY.md 8f rank 1; replaces the Taylor blocks of
// vectorize.py:8-49 for this model mode):  x+ = expm(G(u) dt) x,  G(u) = L_0 + sum_i u_i L_i.
//   A = expm(G dt)                      scaling and squaring of a degree-16 Taylor polynomial (Horner), C x C complex
//   b_i = (d/du_i expm(G(u) dt)) x      = w_i(1) of  y' = G dt y,  w_i' = G dt w_i + L_i dt y,  y(0) = x, w_i(0) = 0,
//                                       integrated exactly by Taylor series on sub-steps of norm <= 4
// gen [M+1][C][C] (shared or global), u [M], x [C] (shared).  scr: double2 [exact_scratch<CF>()] shared.
// On return A sits in scr[C*C .. 2*C*C) and b_i[r] in scr[exact_b_offset<CF>() + i*C + r].  All lanes must call.
// ---------------------------------------------------------------------------------------------------------
__host__ __device__ constexpr int strip_len(int C) {
    for (int sl = 1; sl <= C; ++sl)
        if (C % sl == 0 && C * C / sl <= 32) return sl;
    return C;
}
template <class CF> __host__ __device__ constexpr int exact_b_offset() { return 2 * CF::C * CF::C + 2 * (1 + CF::M) * CF::C; }
template <class CF> __host__ __device__ constexpr int exact_scratch() { return exact_b_offset<CF>() + CF::M * CF::C; }

template <class CF>
__device__ __noinline__ void exact_stage(const double2 *gen, const double *u, const double2 *x, double dt, double2 *scr,
                                         int lane) {
    constexpr int C = CF::C, M = CF::M, CC = C * C, NE = cdiv(CC, 32), NV = cdiv((1 + M) * C, 32);
    double2 *G = scr, *T = scr + CC, *vec = scr + 2 * CC, *bout = scr + exact_b_offset<CF>();
    // ---- G = dt (L_0 + sum u_i L_i), 1-norm
    double uu[M];
#pragma unroll
    for (int i = 0; i < M; ++i) uu[i] = u[i];
#pragma unroll
    for (int q = 0; q < NE; ++q) {
        const int e = lane + 32 * q;
        if (e < CC) {
            double2 g = gen[e];
#pragma unroll
            for (int i = 0; i < M; ++i) {
                const double2 l = gen[(1 + i) * CC + e];
                g.x = fma(uu[i], l.x, g.x);
                g.y = fma(uu[i], l.y, g.y);
            }
            G[e] = make_double2(g.x * dt, g.y * dt);
        }
    }
    __syncwarp();
    double nrm = 0.0;
    if (lane < C) {
#pragma unroll 1
        for (int i = 0; i < C; ++i) {
            const double2 g = G[i * C + lane];
            nrm += hypot(g.x, g.y);
        }
    }
    nrm = warp_max(nrm);
    const double theta = nrm;
    int sq = 0;
    while (nrm > 0.5 && sq < 40) {
        nrm *= 0.5;
        ++sq;
    }
    const double sc = ldexp(1.0, -sq);
    // strip length: smallest divisor of C with C * C / SL <= 32 lanes
    constexpr int SL = strip_len(C), STRIPS = C * C / SL;
    const int sl = lane < STRIPS ? lane : STRIPS - 1;
    const int si = sl / (C / SL), sj = (sl % (C / SL)) * SL;
    // (A Paterson-Stockmeyer evaluation -- 7 + sq products instead of 16 + sq, +13 % throughput of this mode -- agreed with
    // scipy to 1.4e-15 instead of 8e-16; the closed loop of this mode amplifies such differences by up to 1e12 on badly
    // mismatched plants (DESIGN.md 5a), and the Horner form tracked the CPU oracle 100x closer there, so it stays.)
    // ---- T = expm(G): Horner of degree 16 on G / 2^sq, then sq squarings.
#pragma unroll
    for (int q = 0; q < NE; ++q) {
        const int e = lane + 32 * q;
        if (e < CC) T[e] = make_double2(e / C == e % C ? 1.0 : 0.0, 0.0);
    }
    __syncwarp();
#pragma unroll 1
    for (int k = 16 + sq; k >= 1; --k) {
        const bool horner = k > sq;                      // first 16 passes: T = I + (sc / kk) G T; then T = T T
        const double f = horner ? sc / (double)(k - sq) : 1.0;
        const double2 *Lm = horner ? G : T;
        // each lane owns a strip of SL consecutive entries of one row: one load of Lm[i][kk] serves SL products
        double2 v[SL];
#pragma unroll
        for (int q = 0; q < SL; ++q) v[q] = make_double2(0.0, 0.0);
        const double2 *lrow = Lm + si * C, *tcol = T + sj;
#pragma unroll
        for (int kk = 0; kk < C; ++kk) {
            const double2 l = lrow[kk];
#pragma unroll
            for (int q = 0; q < SL; ++q) v[q] = cfma(l, tcol[kk * C + q], v[q]);
        }
        __syncwarp();
        if (lane < STRIPS) {
#pragma unroll
            for (int q = 0; q < SL; ++q)
                T[si * C + sj + q] = make_double2(fma(v[q].x, f, (horner && si == sj + q) ? 1.0 : 0.0), v[q].y * f);
        }
        __syncwarp();
    }
    // ---- b_i: Taylor series of the augmented vector system on n_sub sub-steps (||G|| / n_sub <= 4)
    int n_sub = (theta < 128.0) ? (int)ceil(theta * 0.25) : 32;    // also catches a non-finite generator
    if (n_sub < 1) n_sub = 1;
    const double h = 1.0 / (double)n_sub;
    // number of terms: (theta h)^K / K! < 1e-19 (sub-step norm <= 4: K <= 36; partial sums stay below e^4)
    int K = 0;
    {
        double term = 1.0;
        const double th = theta * h;
        while (term > 1e-19 && K < 40) {
            ++K;
            term *= th / (double)K;
        }
    }
    // vec: two buffers [(1 + M) C]: term vectors (y-term, w_1-term, ...); lane job e -> (v = e / C, r = e % C)
    double2 acc[NV];
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        const int e = lane + 32 * q;
        acc[q] = (e < C) ? x[e] : make_double2(0.0, 0.0);
        if (e < (1 + M) * C) vec[e] = acc[q];
    }
    __syncwarp();
    // small systems (one job per lane): the lane's rows of G and L_v are the same in every term -- keep them in
    // registers, so a term costs only the loads of the term vectors
    constexpr bool ROWS_IN_REGS = (NV == 1) && (C <= 9);
    double2 grow_r[ROWS_IN_REGS ? C : 1], lrow_r[ROWS_IN_REGS ? C : 1];
    if constexpr (ROWS_IN_REGS) {
        const int ec = lane < (1 + M) * C ? lane : 0;
        const int v = ec / C, r = ec % C;
#pragma unroll
        for (int j = 0; j < C; ++j) {
            grow_r[j] = G[r * C + j];
            const double2 l = gen[(v > 0 ? v : 1) * CC + r * C + j];
            lrow_r[j] = v > 0 ? make_double2(l.x * dt, l.y * dt) : make_double2(0.0, 0.0);
        }
    }
#pragma unroll 1
    for (int sub = 0; sub < n_sub; ++sub) {
        int cur = 0;
#pragma unroll 1
        for (int k = 1; k <= K; ++k) {
            const double f = h / (double)k;
            const double2 *tv = vec + cur * (1 + M) * C;
            double2 *nv = vec + (cur ^ 1) * (1 + M) * C;
            if constexpr (ROWS_IN_REGS) {
                if (lane < (1 + M) * C) {
                    const int v = lane / C;
                    const double2 *tw = tv + v * C;
                    double2 a0 = make_double2(0.0, 0.0), a1 = make_double2(0.0, 0.0);
#pragma unroll
                    for (int j = 0; j < C; ++j) {
                        a0 = cfma(grow_r[j], tw[j], a0);
                        a1 = cfma(lrow_r[j], tv[j], a1);
                    }
                    const double2 t = make_double2((a0.x + a1.x) * f, (a0.y + a1.y) * f);
                    nv[lane] = t;
                    acc[0].x += t.x;
                    acc[0].y += t.y;
                }
            } else {
#pragma unroll
                for (int q = 0; q < NV; ++q) {
                    const int e = lane + 32 * q;
                    if (e < (1 + M) * C) {
                        const int v = e / C, r = e % C;
                        double2 a0 = make_double2(0.0, 0.0), a1 = make_double2(0.0, 0.0);
                        const double2 *grow = G + r * C, *tw = tv + v * C;
#pragma unroll
                        for (int j = 0; j < C; ++j) a0 = cfma(grow[j], tw[j], a0);
                        if (v > 0) {
                            const double2 *lrow = gen + v * CC + r * C;
#pragma unroll
                            for (int j = 0; j < C; ++j) a1 = cfma(lrow[j], tv[j], a1);
                        }
                        const double2 t = make_double2(fma(a1.x, dt, a0.x) * f, fma(a1.y, dt, a0.y) * f);
                        nv[e] = t;
                        acc[q].x += t.x;
                        acc[q].y += t.y;
                    }
                }
            }
            __syncwarp();
            cur ^= 1;
        }
        // restart the series from the state at the end of the sub-step
#pragma unroll
        for (int q = 0; q < NV; ++q) {
            const int e = lane + 32 * q;
            if (e < (1 + M) * C) vec[e] = acc[q];
        }
        __syncwarp();
    }
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        const int e = lane + 32 * q;
        if (e >= C && e < (1 + M) * C) bout[e - C] = acc[q];
    }
    __syncwarp();
}

// U <- T U (gate synthesis: the plant state is the propagator itself, experiment.py:371-401)
__device__ __noinline__ void left_multiply(double2 *U, const double2 *T, int d, double2 *tmp, int lane) {
    const bool act = lane < d * d;
    if (act) tmp[lane] = cmm(T, U, d, lane / d, lane % d);
    __syncwarp();
    if (act) U[lane] = tmp[lane];
    __syncwarp();
}

}  // namespace m4q
