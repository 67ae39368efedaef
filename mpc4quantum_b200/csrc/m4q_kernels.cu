// libm4q: kernels and C ABI of the B200-native MPC4quantum hot path (sm_100a).
//
// One warp owns one ensemble member (or one QP instance); everything a member needs between the first
// linearisation and the last plant step lives in a warp-private slab of shared memory, so the closed loop of
// mpc4quantum/mpc.py:128-304 runs without leaving the SM.  The device building blocks are in m4q_core.cuh; this
// file holds the kernels, the launch geometry and the extern "C" entry points declared in include/m4q.h.
#include "m4q_core.cuh"
#include "../../include/m4q.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

namespace m4q {

static thread_local std::string g_err;

static int fail(const std::string &msg) {
    g_err = msg;
    return -1;
}
#define M4Q_CUDA(call)                                                                                         \
    do {                                                                                                       \
        cudaError_t e_ = (call);                                                                               \
        if (e_ != cudaSuccess)                                                                                 \
            return fail(std::string(#call) + ": " + cudaGetErrorString(e_));                                  \
    } while (0)

// ---------------------------------------------------------------------------------------------------------
// Shared tables of one closed-loop problem (member independent), built once per launch by build_tables.
// Layout in doubles; offsets from TableLayout.
// ---------------------------------------------------------------------------------------------------------
struct TableLayout {
    int Qr, Qfr, Rr, r, qlin, qlinf, ub, Rub, flags, hq, hqf, hb, total;
    __host__ __device__ TableLayout(int N, int M, int n_targ) {
        int o = 0;
        auto take = [&](int cnt) {
            int at = o;
            o += rup(cnt, 2);
            return at;
        };
        Qr = take(N * N);
        Qfr = take(N * N);
        Rr = take(M * M);
        r = take(n_targ * N);
        qlin = take(n_targ * N);
        qlinf = take(n_targ * N);
        ub = take(n_targ * M);
        Rub = take(n_targ * M);
        flags = take(4);   // [0] q_diag, [1] work counter (as int), [2..3] factorisations in Hermitian / realified
                           // coordinates (unsigned 64-bit, summed over the members of the launch)
        // Hermitian coordinates (HermCfg, HermBasis in m4q_core.cuh): reduced costs T^T Q T, T^T Qf T, basis descriptors
        const int NR = rup(N / 2, 2);
        hq = take(NR * NR);
        hqf = take(NR * NR);
        hb = take(cdiv(3 * NR + 3 * N + 1, 2));
        total = o;
    }
};

// realified, symmetrised cost block: M = [[Re, -Im], [Im, Re]], out = (M + M^T) / 2
__device__ __forceinline__ double realified_sym(const double2 *Qc, int C, int i, int j) {
    auto entry = [&](int a, int b) {
        const int ra = a % C, rb = b % C;
        const double2 v = Qc[ra * C + rb];
        if (a < C) return b < C ? v.x : -v.y;
        return b < C ? v.y : v.x;
    };
    return 0.5 * (entry(i, j) + entry(j, i));
}

// sigma of the lift (m4q_mpc_herm_sigma); ok = 0: the factor stays realified
struct HermSigma {
    int ok;
    int sig[32];
};

// Largest deviation of a model block from sigma-conjugate symmetry, N[s(i)][s(j)] = conj(N[i][j]), against the tolerance:
// true if symmetric.  The device Taylor discretisation sums the products of an entry and of its partner in different
// orders (q and s(q)), so the blocks it produces are symmetric to a few ulp, not bit for bit: the tolerance is 16 ulp of
// the block's largest entry.  The same comparisons run for shared (build_tables) and per-member models (mpc_kernel),
// so a member gets the same factor whichever way its model arrives.
__device__ __forceinline__ double herm_block_scale(double2 v) { return fmax(fabs(v.x), fabs(v.y)); }
__device__ __forceinline__ bool herm_entry_ok(const double2 *blk, const int *sig, int C, int e, double scale) {
    const int i = e / C, j = e % C;
    const double2 a = blk[e], b = blk[sig[i] * C + sig[j]];
    const double tol = 16.0 * 2.220446049250313e-16 * scale;
    return fabs(b.x - a.x) <= tol && fabs(b.y + a.y) <= tol;
}

__global__ void build_tables(int C, int M, int n_targ, const double2 *Q, const double2 *Qf, const double *R,
                             const double2 *X_targ, const double *U_targ, double *tab, HermSigma hs,
                             const double2 *A_blocks, int nblk) {
    const int N = 2 * C;
    const TableLayout L(N, M, n_targ);
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int e = tid; e < N * N; e += nt) {
        tab[L.Qr + e] = realified_sym(Q, C, e / N, e % N);
        tab[L.Qfr + e] = realified_sym(Qf, C, e / N, e % N);
    }
    for (int e = tid; e < M * M; e += nt) tab[L.Rr + e] = 0.5 * (R[e] + R[(e % M) * M + e / M]);
#pragma unroll 1
    for (int e = tid; e < n_targ * N; e += nt) {
        const int col = e / N, k = e % N;
        const double2 v = X_targ[(k % C) * n_targ + col];
        tab[L.r + e] = k < C ? v.x : v.y;
    }
#pragma unroll 1
    for (int e = tid; e < n_targ * M; e += nt) {
        const int col = e / M, i = e % M;
        tab[L.ub + e] = col < n_targ - 1 ? U_targ[i * (n_targ - 1) + col] : 0.0;
    }
    __syncthreads();
#pragma unroll 1
    for (int e = tid; e < n_targ * N; e += nt) {
        const int col = e / N, k = e % N;
        double a = 0.0, b = 0.0;
        for (int j = 0; j < N; ++j) {
            const double rv = tab[L.r + col * N + j];
            a = fma(tab[L.Qr + k * N + j], rv, a);
            b = fma(tab[L.Qfr + k * N + j], rv, b);
        }
        tab[L.qlin + e] = a;
        tab[L.qlinf + e] = b;
    }
#pragma unroll 1
    for (int e = tid; e < n_targ * M; e += nt) {
        const int col = e / M, i = e % M;
        double a = 0.0;
        for (int j = 0; j < M; ++j) a = fma(tab[L.Rr + i * M + j], tab[L.ub + col * M + j], a);
        tab[L.Rub + e] = a;
    }
    if (tid == 0) {
        bool diag = true;
        for (int i = 0; i < N; ++i)
            for (int j = 0; j < N; ++j)
                if (i != j && (tab[L.Qr + i * N + j] != 0.0 || tab[L.Qfr + i * N + j] != 0.0)) diag = false;
        tab[L.flags] = diag ? 1.0 : 0.0;
        int *ctr = reinterpret_cast<int *>(tab + L.flags + 1);
        ctr[0] = 0;
        ctr[1] = 0;
        unsigned long long *fc = reinterpret_cast<unsigned long long *>(tab + L.flags + 2);
        fc[0] = 0;
        fc[1] = 0;
        // basis of the Hermitian coordinates (HermBasis): a fixed point k of sigma gives Re x_k; a pair k < s(k) gives
        // (Re x_k + Re x_sk) / 2 and (Im x_k - Im x_sk) / 2
        const int NR = rup(C, 2);
        int *hb = reinterpret_cast<int *>(tab + L.hb);
        int *J1 = hb, *J2 = hb + NR, *SG = hb + 2 * NR, *CO = hb + 3 * NR, *WT = CO + N, *PA = WT + N, *OK = PA + N;
        for (int a = 0; a < NR; ++a) J1[a] = J2[a] = SG[a] = 0;
        int a = 0;
        bool ok = hs.ok != 0;
        for (int k = 0; k < C && ok; ++k) {
            const int sk = hs.sig[k];
            ok &= sk >= 0 && sk < C && hs.sig[sk] == k;
            if (!ok) break;
            PA[k] = sk;
            PA[C + k] = C + sk;
            if (sk == k) {
                J1[a] = J2[a] = k;
                SG[a] = 1;
                CO[k] = CO[C + k] = a;
                WT[k] = 2;
                WT[C + k] = 0;
                ++a;
            } else if (k < sk) {
                J1[a] = k;
                J2[a] = sk;
                SG[a] = 1;
                CO[k] = CO[sk] = a;
                WT[k] = WT[sk] = 1;
                ++a;
                J1[a] = C + k;
                J2[a] = C + sk;
                SG[a] = -1;
                CO[C + k] = CO[C + sk] = a;
                WT[C + k] = 1;
                WT[C + sk] = -1;
                ++a;
            }
        }
        if (!ok)
            for (int j = 0; j < N; ++j) {
                CO[j] = WT[j] = 0;
                PA[j] = j;
            }
        // the premise shared by every QP of the launch: sigma-symmetric costs (exact) and shared model blocks
        for (int i = 0; i < N && ok; ++i)
            for (int j = 0; j < N; ++j) {
                const int pi = PA[i], pj = PA[j];
                const double sg = ((i < C) == (j < C)) ? 1.0 : -1.0;
                ok &= tab[L.Qr + pi * N + pj] * sg == tab[L.Qr + i * N + j] && tab[L.Qfr + pi * N + pj] * sg == tab[L.Qfr + i * N + j];
            }
        for (int kb = 0; kb < nblk && ok && A_blocks; ++kb) {
            const double2 *blk = A_blocks + (size_t)kb * C * C;
            double scale = 0.0;
            for (int e = 0; e < C * C; ++e) scale = fmax(scale, herm_block_scale(blk[e]));
            for (int e = 0; e < C * C; ++e) ok &= herm_entry_ok(blk, hs.sig, C, e, scale);
        }
        *OK = ok ? 1 : 0;
    }
    __syncthreads();
    // reduced costs T^T Q T: coordinate a is x_J1 + SG x_J2 (x_J1 alone for a fixed point); padding rows stay zero
    const int NR = rup(C, 2);
    const int *hb = reinterpret_cast<const int *>(tab + L.hb);
    for (int e = tid; e < NR * NR; e += nt) {
        const int a = e / NR, b = e % NR;
        double q = 0.0, qf = 0.0;
        if (a < C && b < C) {
            const int ja[2] = {hb[a], hb[NR + a]}, jb[2] = {hb[b], hb[NR + b]};
            const double wa[2] = {1.0, ja[0] == ja[1] ? 0.0 : (double)hb[2 * NR + a]};
            const double wb[2] = {1.0, jb[0] == jb[1] ? 0.0 : (double)hb[2 * NR + b]};
            for (int u = 0; u < 2; ++u)
                for (int v = 0; v < 2; ++v) {
                    q = fma(wa[u] * wb[v], tab[L.Qr + ja[u] * N + jb[v]], q);
                    qf = fma(wa[u] * wb[v], tab[L.Qfr + ja[u] * N + jb[v]], qf);
                }
        }
        tab[L.hq + e] = q;
        tab[L.hqf + e] = qf;
    }
}

// ---------------------------------------------------------------------------------------------------------
// Observable maps (experiment.py:29-37, 225-235, 248-306).  plant state: double2 [d*d] in shared memory.
// ---------------------------------------------------------------------------------------------------------
// model state (realified, length 2C) <- lift(plant state)
template <class CF>
__device__ void lift_state(int mode, int d, const double2 *rho, double *out, int lane) {
    constexpr int C = CF::C;
    if (mode == M4Q_LIFT_IDENTITY) {
        if (lane < C) {
            out[lane] = rho[lane].x;
            out[C + lane] = rho[lane].y;
        }
    } else if (mode == M4Q_LIFT_COUPLED) {
        // d = dA*dA; stacked [vec(tr_B rho), vec(tr_A rho)], C = 2*dA*dA
        const int dA = (d == 4) ? 2 : (d == 9 ? 3 : 1);
        const int half = dA * dA;
        if (lane < 2 * half) {
            const int which = lane / half, e = lane % half, a = e / dA, b = e % dA;
            double2 acc = make_double2(0.0, 0.0);
#pragma unroll 1
            for (int k = 0; k < dA; ++k) {
                // which = 0: rhoA[a][b] = sum_k rho[(a,k),(b,k)];  which = 1: rhoB[a][b] = sum_k rho[(k,a),(k,b)]
                const int row = which == 0 ? a * dA + k : k * dA + a;
                const int col = which == 0 ? b * dA + k : k * dA + b;
                const double2 v = rho[row * d + col];
                acc.x += v.x;
                acc.y += v.y;
            }
            out[lane] = acc.x;
            out[C + lane] = acc.y;
        }
    } else if (mode == M4Q_LIFT_PROCESS) {
        // plant state = propagator U [d][d]; model state = vec(U (x) U^*), C = d^4 (experiment.py:357-369):
        // element (i d + k) d^2 + (j d + l) = U[i][j] conj(U[k][l])
        const int d2 = d * d;
        if (lane < C) {
            const int row = lane / d2, col = lane % d2;
            const double2 a = rho[(row / d) * d + col / d], b = rho[(row % d) * d + col % d];
            const double2 v = cmul(a, make_double2(b.x, -b.y));
            out[lane] = v.x;
            out[C + lane] = v.y;
        }
    } else {   // M4Q_LIFT_TRUNC32: qubit block of a qutrit divided by its trace norm (sum of singular values)
        const double2 a = rho[0], b = rho[1], c = rho[3], e = rho[4];
        const double fro = a.x * a.x + a.y * a.y + b.x * b.x + b.y * b.y + c.x * c.x + c.y * c.y + e.x * e.x + e.y * e.y;
        const double2 ae = cmul(a, e), bc = cmul(b, c);
        const double det = hypot(ae.x - bc.x, ae.y - bc.y);
        const double nrm = sqrt(fro + 2.0 * det);
        if (lane < 4) {
            const double2 v = rho[(lane / 2) * 3 + lane % 2];
            out[lane] = v.x / nrm;
            out[C + lane] = v.y / nrm;
        }
    }
    __syncwarp();
}

// plant state <- proj(model state)
template <class CF>
__device__ void proj_state(int mode, int d, const double *x, double2 *rho, int lane) {
    constexpr int C = CF::C;
    if (mode == M4Q_LIFT_COUPLED) {
        const int dA = (d == 4) ? 2 : (d == 9 ? 3 : 1);
        const int half = dA * dA;
        if (lane < d * d) {
            const int row = lane / d, col = lane % d;
            const int a = row / dA, b = row % dA, a2 = col / dA, b2 = col % dA;
            const double2 ra = make_double2(x[a * dA + a2], x[C + a * dA + a2]);
            const double2 rb = make_double2(x[half + b * dA + b2], x[C + half + b * dA + b2]);
            rho[lane] = cmul(ra, rb);
        }
    } else {
        if (lane < C) rho[lane] = make_double2(x[lane], x[C + lane]);
    }
    __syncwarp();
}

// Re <w, observed state>: the plant state itself (<psi|rho|psi> for w = vec(|psi><psi|)), or, for gate synthesis,
// the lifted process vector (|tr(Uf^+ U)|^2 / d^2 for w = vec(Uf (x) Uf^*) / d^2).
template <class CF>
__device__ double fidelity_of(int mode, int d, const double2 *w, const double2 *xcur, double *scratch, int lane) {
    constexpr int C = CF::C;
    double f = 0.0;
    if (mode == M4Q_LIFT_PROCESS) {
        lift_state<CF>(mode, d, xcur, scratch, lane);
        if (lane < C) {
            const double2 wv = w[lane];
            f = wv.x * scratch[lane] + wv.y * scratch[C + lane];
        }
        __syncwarp();
    } else if (lane < d * d) {
        const double2 wv = w[lane], x = xcur[lane];
        f = wv.x * x.x + wv.y * x.y;
    }
    return warp_sum(f);
}

// ---------------------------------------------------------------------------------------------------------
// Measurement noise (experiment.py:193-194, :212): counter-based generator Philox4x32-10, key = the 64-bit seed,
// counter = (member lo, member hi, MPC step, component): one call gives the two N(0,1) deviates of a complex
// component (Box-Muller on two 53-bit uniforms).  Independent of the launch geometry and of the GPU count.
// ---------------------------------------------------------------------------------------------------------
__host__ __device__ inline void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n1 = (uint32_t)p1;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1, n3 = (uint32_t)p0;
        c[0] = n0;
        c[1] = n1;
        c[2] = n2;
        c[3] = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}
__device__ __noinline__ double2 normal_pair(uint64_t seed, long long member, int step, int comp) {
    uint32_t c[4] = {(uint32_t)member, (uint32_t)((unsigned long long)member >> 32), (uint32_t)step, (uint32_t)comp};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    const double u1 = (double)((((uint64_t)c[1] << 32) | c[0]) >> 11) * 0x1.0p-53 + 0x1.0p-54;
    const double u2 = (double)((((uint64_t)c[3] << 32) | c[2]) >> 11) * 0x1.0p-53;
    const double r = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    return make_double2(r * cs, r * sn);
}

// ---------------------------------------------------------------------------------------------------------
// Streaming model of one member (OnlineDMDc, model.py:216-313): A [c][dz], P [dz][dz] complex in global memory,
// dz = c (p + 1); z = [x; phi_1 x; ..; phi_p x] is built in shared memory (zs, dz complex).
//   stream_predict:  out = A z                                         (model.py:81-93 with the member's A)
//   stream_update:   gamma = 1 / (1 + z^T P z);  A += gamma (y - A z)(P z)^T;  P = (P - gamma P z (P z)^T) / discount
// (plain transposes, as the reference writes them).  pz: dz complex of shared scratch.
// ---------------------------------------------------------------------------------------------------------
template <class CF>
__device__ __noinline__ void stream_build_z(const double *x_real, const double *phi, int nblk, double2 *zs, int lane) {
    constexpr int C = CF::C;
#pragma unroll 1
    for (int e = lane; e < nblk * C; e += 32) {
        const int kb = e / C, r = e % C;
        const double ph = kb == 0 ? 1.0 : phi[kb];
        zs[e] = make_double2(ph * x_real[r], ph * x_real[C + r]);
    }
    __syncwarp();
}
template <class CF>
__device__ __noinline__ double2 stream_row_dot(const double2 *row, const double2 *zs, int dz) {
    double2 acc = make_double2(0.0, 0.0);
#pragma unroll 1
    for (int j = 0; j < dz; ++j) acc = cfma(row[j], zs[j], acc);
    return acc;
}
template <class CF>
__device__ __noinline__ void stream_update(double2 *A, double2 *P, const double2 *zs, const double *y_real, int dz, double discount,
                              double2 *pz, double2 *red, int lane) {
    constexpr int C = CF::C;
    // P z (rows over lanes) and z^T P z
    double2 part = make_double2(0.0, 0.0);
#pragma unroll 1
    for (int i = lane; i < dz; i += 32) {
        const double2 v = stream_row_dot<CF>(P + (size_t)i * dz, zs, dz);
        pz[i] = v;
        part = cfma(zs[i], v, part);
    }
    part.x = warp_sum(part.x);
    part.y = warp_sum(part.y);
    // gamma = 1 / (1 + z^T P z), complex
    const double dr = 1.0 + part.x, di = part.y, dn = dr * dr + di * di;
    const double2 gamma = make_double2(dr / dn, -di / dn);
    __syncwarp();
    // A += gamma (y - A z) (P z)^T : lane r < C owns row r
    if (lane < C) {
        double2 *row = A + (size_t)lane * dz;
        const double2 az = stream_row_dot<CF>(row, zs, dz);
        const double2 err = cmul(gamma, make_double2(y_real[lane] - az.x, y_real[C + lane] - az.y));
#pragma unroll 1
        for (int j = 0; j < dz; ++j) row[j] = cfma(err, pz[j], row[j]);
    }
    // P = (P - gamma (P z)(P z)^T) / discount : rows over lanes
    const double inv = 1.0 / discount;
#pragma unroll 1
    for (int i = lane; i < dz; i += 32) {
        double2 *row = P + (size_t)i * dz;
        const double2 gi = cmul(gamma, pz[i]);
#pragma unroll 1
        for (int j = 0; j < dz; ++j) {
            const double2 d = cmul(gi, pz[j]);
            row[j] = make_double2((row[j].x - d.x) * inv, (row[j].y - d.y) * inv);
        }
    }
    (void)red;
    __syncwarp();
}

// ---------------------------------------------------------------------------------------------------------
// The closed loop kernel
// ---------------------------------------------------------------------------------------------------------
struct MpcArgs {
    int H, S, mf, warm_start, max_iter, lift_mode, has_du, n_targ, d, nblk;
    double dt, sat, du, exit_infid;
    QPSet set;
    const double2 *A_blocks;
    const int *powers;
    const double2 *fid_vec;
    double *tab;
    long long n_members;
    const double2 *x0;
    int x0_shared;
    const double2 *H0, *H1;
    int shared_ham;
    int step_begin, step_end, external_plant;
    double2 *xs;
    double *us;
    int *exit_code, *steps_done, *qp_count, *counters;
    double *fidelity;
    double *state;
    double *ws;   // L2-resident workspaces, one per resident warp (ws_doubles<CF>(H) each)
    int slab_doubles, shared_doubles;
    int model_per_member;   // A_blocks is [n_members][nblk][C][C]: every member controls with its own model
    double *ws_exact;       // EXACT: per resident warp, the stage matrices A_t = expm(G(u_t) dt)  [H][C][C] complex
    double noise_sigma;
    unsigned long long noise_seed;
    long long member_offset;   // global index of member 0 of this launch (noise streams do not depend on the sharding)
    int streaming, fidelity_sqrt;
    double stream_discount;
    double2 *stream_A, *stream_P;
};

// ---------------------------------------------------------------------------------------------------------
// Exact-discretisation model mode: linearisation along (Xg, Ug) with the generators [L_0, L_1..L_M] in place of the
// Taylor blocks.  Writes A_t (dense, per stage) to the warp's global array, B_t / Delta_t to the stage records, phi = 1.
// ---------------------------------------------------------------------------------------------------------
template <class CF>
__device__ __noinline__ void linearize_exact(SlabRef sr, const double2 *gen, double dt, double2 *At, int lane) {
    constexpr int C = CF::C, N = CF::N, M = CF::M, CC = C * C;
    using R_ = Rec<CF>;
    static_assert(2 * exact_scratch<CF>() <= CF::KR * (CF::LDP + CF::LDG), "exact-stage scratch must fit the factor scratch");
    const Slab<CF> s = slab_view<CF>(sr);
    const double *Xg = ws_Xg<CF>(sr);
    double2 *scr = reinterpret_cast<double2 *>(s.recring);
    double2 *xs = reinterpret_cast<double2 *>(s.va);
#pragma unroll 1
    for (int t = 0; t < sr.H; ++t) {
        if (lane < C) xs[lane] = make_double2(Xg[t * N + lane], Xg[t * N + C + lane]);
        __syncwarp();
        exact_stage<CF>(gen, s.Ug + t * M, xs, dt, scr, lane);
        const double2 *T = scr + CC, *b = scr + exact_b_offset<CF>();
#pragma unroll 1
        for (int e = lane; e < CC; e += 32) At[(size_t)t * CC + e] = T[e];
        if (lane < N) {
            const int r = lane < C ? lane : lane - C;
            double *rec = ws_rec<CF>(sr, t);
            double d = 0.0;
#pragma unroll
            for (int i = 0; i < M; ++i) {
                const double2 bv = b[i * C + r];
                const double bb = lane < C ? bv.x : bv.y;
                rec[R_::B + R_::pair(i, lane)] = bb;
                d = fma(-bb, s.Ug[t * M + i], d);
            }
            rec[R_::D + lane] = d;
        }
        __syncwarp();
    }
}


template <class CF, bool EXACT>
__global__ void __launch_bounds__(CF::MAXW * 32) mpc_kernel(const MpcArgs a) {
    constexpr int C = CF::C, N = CF::N, M = CF::M;
    extern __shared__ double2 smem2[];
    double *smem = reinterpret_cast<double *>(smem2);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int H = a.H, S = a.S, d = a.d, dd = d * d;
    const int xdim = a.external_plant ? C : dd;   // length of one xs column
    const TableLayout L(N, M, a.n_targ);

    // ---- CTA-shared, read-only: model blocks, monomial exponents, cost matrices
    double2 *blocks = reinterpret_cast<double2 *>(smem);
    double *Qr = smem + 2 * a.nblk * C * C;
    double *Qfr = Qr + N * N;
    double *Rr = Qfr + N * N;
    int *pow = reinterpret_cast<int *>(Rr + rup(M * M, 2));
#pragma unroll 1
    for (int e = threadIdx.x; e < a.nblk * C * C; e += blockDim.x) blocks[e] = a.model_per_member ? make_double2(0.0, 0.0) : a.A_blocks[e];
    for (int e = threadIdx.x; e < N * N; e += blockDim.x) {
        Qr[e] = a.tab[L.Qr + e];
        Qfr[e] = a.tab[L.Qfr + e];
    }
    for (int e = threadIdx.x; e < M * M; e += blockDim.x) Rr[e] = a.tab[L.Rr + e];
#pragma unroll 1
    for (int e = threadIdx.x; e < (a.nblk - 1) * M; e += blockDim.x) pow[e] = a.powers[e];
    // c = 8, 16: rows of a block are a multiple of 128 bytes apart, so the one-row-per-lane loads of linearize() would be
    // an 8-way bank conflict; it reads transposed copies instead (consecutive lanes -> consecutive addresses)
    const int soffT = a.shared_doubles - 2 * (a.nblk - 1) * C * C;
    if (C % 8 == 0 && !a.model_per_member) {
        double2 *blocksT = reinterpret_cast<double2 *>(smem + soffT);
#pragma unroll 1
        for (int e = threadIdx.x; e < (a.nblk - 1) * C * C; e += blockDim.x) {
            const int kb = e / (C * C), rj = e % (C * C);
            blocksT[kb * C * C + (rj % C) * C + rj / C] = a.A_blocks[(kb + 1) * C * C + rj];
        }
    }
    __syncthreads();

    const SlabRef sr = {a.shared_doubles + warp * a.slab_doubles, H, a.nblk, cmax(dd, C),
                        a.ws + (size_t)(blockIdx.x * (blockDim.x >> 5) + warp) * ws_doubles<CF>(H)};
    const Slab<CF> s = slab_view<CF>(sr);
    double *Xg = ws_Xg<CF>(sr);
    const double *Xo = ws_Xo<CF>(sr);
    double2 *xcur = reinterpret_cast<double2 *>(s.xcur);
    double2 *xmeas = reinterpret_cast<double2 *>(s.xmeas);
    double2 *scr2 = reinterpret_cast<double2 *>(s.scr);

    StageOps model;
    model.blocks = blocks;
    model.nblk = a.nblk;
    model.stage_stride = 0;
    model.soff = 0;
    model.soffT = (C % 8 == 0 && !a.model_per_member) ? soffT : 0;
    model.pow = pow;
    model.pow_soff = (int)(reinterpret_cast<double *>(pow) - smem);
    {
        bool fo = a.nblk - 1 == M;
        if (fo)
            for (int e = 0; e < M * M; ++e) fo &= pow[e] == ((e / M == e % M) ? 1 : 0);
        model.first_order = fo;
    }
    if (a.model_per_member) {
        // perturbed MODELS: the member's own blocks sit behind its slab (the slab stride includes them)
        model.soff = sr.off + a.slab_doubles - 2 * a.nblk * C * C;
        model.blocks = reinterpret_cast<const double2 *>(smem + model.soff);
    }

    int *work = reinterpret_cast<int *>(a.tab + L.flags + 1);
    const int q_diag = a.tab[L.flags] != 0.0;
    // factor in Hermitian coordinates: instantiation, launch-wide premise (build_tables), then per member and per QP
    const int *hb = reinterpret_cast<const int *>(a.tab + L.hb);
    const bool herm_launch = CF::HERM && !EXACT && hb[HermBasis<CF>::OK] != 0;
    const int persist = Slab<CF>::persistent_doubles(H, cmax(dd, C));

    for (;;) {
        long long k = 0;
        if (lane == 0) k = atomicAdd(work, 1);
        k = __shfl_sync(FULL, k, 0);
        if (k >= a.n_members) break;

        Counters cnt = {};
        bool herm_member = herm_launch;
        int exit_code = 0;
        double2 *xs_k = a.xs + (size_t)k * xdim * (S + 1);
        double *us_k = a.us + (size_t)k * M * S;
        const double2 *H0k = a.H0 ? a.H0 + (a.shared_ham ? 0 : (size_t)k * dd) : nullptr;
        const double2 *H1k = a.H1 ? a.H1 + (a.shared_ham ? 0 : (size_t)k * M * dd) : nullptr;
        if (a.model_per_member) {
            double2 *mine = reinterpret_cast<double2 *>(smem + model.soff);
            const double2 *src = a.A_blocks + (size_t)k * a.nblk * C * C;
#pragma unroll 1
            for (int e = lane; e < a.nblk * C * C; e += 32) mine[e] = src[e];
            __syncwarp();
            if (herm_member) {
                // the member's own blocks must be sigma-symmetric too (same test as build_tables)
                const int *sig = hb + HermBasis<CF>::PA;   // sigma on the real parts
                bool ok = true;
#pragma unroll 1
                for (int kb = 0; kb < a.nblk; ++kb) {
                    const double2 *blk = mine + kb * C * C;
                    double scale = 0.0;
#pragma unroll 1
                    for (int e = lane; e < C * C; e += 32) scale = fmax(scale, herm_block_scale(blk[e]));
                    scale = warp_max(scale);
#pragma unroll 1
                    for (int e = lane; e < C * C; e += 32) ok &= herm_entry_ok(blk, sig, C, e, scale);
                }
                herm_member = __all_sync(FULL, ok);
            }
        }

        // ---- initial or restored loop state
        if (a.step_begin == 0) {
            const double2 *x0k = a.x0 + (a.x0_shared ? 0 : (size_t)k * xdim);
            if (lane < xdim) {
                const double2 v = x0k[lane];
                xcur[lane] = v;
                xmeas[lane] = v;
                xs_k[(size_t)lane * (S + 1)] = v;
            }
            __syncwarp();
            lift_state<CF>(a.external_plant ? M4Q_LIFT_IDENTITY : a.lift_mode, d, xcur, s.x0, lane);
#pragma unroll 1
            for (int e = lane; e < (H + 1) * N; e += 32) Xg[e] = s.x0[e % N];     // mpc.py:141
#pragma unroll 1
            for (int e = lane; e < H * M; e += 32) {                              // mpc.py:142
                s.Ug[e] = 0.0;
                s.z[e] = 0.0;
                s.y[e] = 0.0;
            }
        } else {
            const double *st = a.state + (size_t)k * persist;
            int o = 0;
#pragma unroll 1
            for (int e = lane; e < (H + 1) * N; e += 32) Xg[e] = st[o + e];
            o += (H + 1) * N;
#pragma unroll 1
            for (int e = lane; e < H * M; e += 32) {
                s.Ug[e] = st[o + e];
                s.z[e] = st[o + H * M + e];
                s.y[e] = st[o + 2 * H * M + e];
            }
            o += 3 * H * M;
            if (lane < xdim) {
                // the caller may have written xs[:, step_begin] (external plant); the measured state is read from xs
                xcur[lane] = xs_k[(size_t)lane * (S + 1) + a.step_begin];
                xmeas[lane] = make_double2(st[o + 2 * lane], st[o + 2 * lane + 1]);
            }
            exit_code = a.exit_code[k];
        }
        __syncwarp();

        int step = a.step_begin;
        if (exit_code == 0) {
            for (; step < a.step_end; ++step) {
                // reference windows lag by one step (mpc.py:145-146, :276-277)
                const int w0 = step == 0 ? 0 : step - 1;
                QPData qp;
                qp.Q = Qr;
                qp.q_stride = 0;
                qp.Qf = Qfr;
                qp.R = Rr;
                qp.r_stride = 0;
                qp.r = a.tab + L.r + (size_t)w0 * N;
                qp.qlin = a.tab + L.qlin + (size_t)w0 * N;
                qp.qlinf = a.tab + L.qlinf + (size_t)(w0 + H) * N;
                qp.ub = a.tab + L.ub + (size_t)w0 * M;
                qp.Rub = a.tab + L.Rub + (size_t)w0 * M;
                qp.sat = a.sat;
                qp.q_diag = q_diag;
                qp.Q_soff = 2 * a.nblk * C * C;
                qp.Qf_soff = qp.Q_soff + N * N;
                qp.R_soff = qp.Qf_soff + N * N;
                qp.Qh = a.tab + L.hq;
                qp.Qfh = a.tab + L.hqf;
                qp.hb = hb;
                qp.herm = 0;

                // measured state -> model space: the QP's initial condition (mpc.py:187)
                lift_state<CF>(a.external_plant ? M4Q_LIFT_IDENTITY : a.lift_mode, d, xcur, s.x0, lane);
                // rate bound centred on us[step-1], or on the reference control for step <= 1 (mpc.py:185)
                if (lane < M) {
                    double lo = -a.sat, hi = a.sat;
                    if (a.has_du) {
                        const double up = step > 1 ? us_k[lane * S + step - 1] : qp.ub[lane];
                        lo = fmax(lo, up - a.du);
                        hi = fmin(hi, up + a.du);
                    }
                    s.lo0[lane] = lo;
                    s.hi0[lane] = hi;
                }
                __syncwarp();
                // an empty stage-0 box (reference control outside the saturation range by more than du): the reference's
                // solver reports the problem infeasible and mpc() leaves with exit code 3 (mpc.py:200-203)
                if (__any_sync(FULL, lane < M && s.lo0[lane < M ? lane : 0] > s.hi0[lane < M ? lane : 0])) {
                    exit_code = 3;
                    break;
                }

                int n_iter = 0;
                bool done = false;
                while (!done && n_iter < a.max_iter) {
                    int status;
                    if constexpr (EXACT) {
                        double2 *At = reinterpret_cast<double2 *>(a.ws_exact) +
                                      (size_t)(blockIdx.x * (blockDim.x >> 5) + warp) * H * C * C;
                        linearize_exact<CF>(sr, model.blocks, a.dt, At, lane);
                        StageOps dense;
                        dense.blocks = At;
                        dense.nblk = 1;
                        dense.stage_stride = C * C;
                        dense.soff = 0;
                        dense.soffT = 0;
                        dense.pow = nullptr;
                        dense.pow_soff = 0;
                        dense.first_order = 0;
                        status = qp_solve<CF, false>(sr, dense, qp, a.set, lane, cnt);
                    } else {
                        // mpc.py:175; the premise of the Hermitian factor is checked on this QP's guess trajectory
                        qp.herm = linearize<CF, true>(sr, model, pow, lane, herm_member ? hb : nullptr);
                        status = qp_solve<CF, true>(sr, model, qp, a.set, lane, cnt);   // mpc.py:189
                    }
                    if (status != 0) {
                        exit_code = status;
                        break;
                    }
                    double alpha = 1.0;
                    if (step > 1 && a.warm_start) {                             // mpc.py:208-212
                        done = true;
                    } else {
                        double stp;
                        line_search<CF, true>(sr, qp, lane, alpha, stp);        // mpc.py:215
                        done = stp < 1e-4;                                      // mpc.py:224
                    }
                    // guess update, four independent elements in flight (the arrays live in L2)
#pragma unroll 1
                    for (int e0 = lane; e0 < (H + 1) * N; e0 += 128) {
                        double xg[4], xo[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int e = e0 + 32 * q;
                            xg[q] = e < (H + 1) * N ? Xg[e] : 0.0;
                            xo[q] = e < (H + 1) * N ? Xo[e] : 0.0;
                        }
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int e = e0 + 32 * q;
                            if (e < (H + 1) * N) Xg[e] = fma(alpha, xo[q] - xg[q], xg[q]);
                        }
                    }
#pragma unroll 1
                    for (int e = lane; e < H * M; e += 32) s.Ug[e] = fma(alpha, s.Uo[e] - s.Ug[e], s.Ug[e]);
                    __syncwarp();
                    ++n_iter;
                }
                if (exit_code != 0) break;
                if (lane == 0) a.qp_count[(size_t)k * S + step] = n_iter;

                // apply the first control of the last QP (mpc.py:250)
                if (lane < M) us_k[lane * S + step] = s.Uo[lane];
                __syncwarp();

                if (!a.external_plant) {
                    if ((step + 1) % a.mf == 0) {
                        // plant window, newest control first (mpc.py:257): segment j uses us[step - j]
#pragma unroll 1
                        for (int j = 0; j < a.mf; ++j) {
                            if (lane < dd) {
                                double2 h = H0k[lane];
                                for (int i = 0; i < M; ++i) {
                                    const double u = us_k[i * S + step - j];
                                    const double2 h1 = H1k[i * dd + lane];
                                    h.x = fma(u, h1.x, h.x);
                                    h.y = fma(u, h1.y, h.y);
                                }
                                scr2[lane] = h;
                            }
                            __syncwarp();
                            expm_minus_i(scr2, a.dt, d, scr2 + dd, scr2 + 2 * dd, scr2 + 3 * dd, lane);
                            if (a.lift_mode == M4Q_LIFT_PROCESS) left_multiply(xmeas, scr2 + 2 * dd, d, scr2 + dd, lane);
                            else conjugate(xmeas, scr2 + 2 * dd, d, scr2 + dd, lane);
                        }
                        if (a.noise_sigma > 0.0 && lane < dd) {
                            // measurement noise; the plant goes on from the noisy record, as the reference's does
                            // (experiment.py:212 feeds mpc.py:259)
                            const double2 nz = normal_pair(a.noise_seed, a.member_offset + k, step, lane);
                            xmeas[lane].x = fma(a.noise_sigma, nz.x, xmeas[lane].x);
                            xmeas[lane].y = fma(a.noise_sigma, nz.y, xmeas[lane].y);
                        }
                        if (lane < dd) xcur[lane] = xmeas[lane];
                        __syncwarp();
                    } else {
                        // model step through lift/proj (mpc.py:264-267): x+ = proj(f(lift(x), u))
                        if (lane < a.nblk) {
                            double phi = 1.0;
                            if (lane > 0)
                                for (int l = 0; l < M; ++l) {
                                    const double ul = s.Uo[l];
#pragma unroll 1
                                    for (int q = 0; q < pow[(lane - 1) * M + l]; ++q) phi *= ul;
                                }
                            s.scr[lane] = phi;
                        }
                        __syncwarp();
                        if (a.streaming) {
                            // the member's own, updated model predicts (model.py:81-93 after fit_iteration rebinds A)
                            double2 *zs = reinterpret_cast<double2 *>(s.scr + MAXBLK);
                            const int dz = a.nblk * C;
                            stream_build_z<CF>(s.x0, s.scr, a.nblk, zs, lane);
                            if (lane < C) {
                                const double2 v = stream_row_dot<CF>(a.stream_A + ((size_t)k * C + lane) * dz, zs, dz);
                                s.va[lane] = v.x;
                                s.va[C + lane] = v.y;
                            }
                        } else {
                            const double fx = apply_A<CF>(model, s.scr, 0, s.x0, lane);
                            __syncwarp();
                            if (lane < N) s.va[lane] = fx;
                        }
                        __syncwarp();
                        proj_state<CF>(a.lift_mode, d, s.va, xcur, lane);
                    }
                    if (lane < dd) xs_k[(size_t)lane * (S + 1) + step + 1] = xcur[lane];
                    if (a.streaming) {
                        // online model update with the transition just observed (mpc.py:281-285, model.py:295-313)
                        __syncwarp();
                        if (lane < a.nblk) {
                            double phi = 1.0;
                            if (lane > 0)
                                for (int l = 0; l < M; ++l) {
                                    const double ul = s.Uo[l];
#pragma unroll 1
                                    for (int q = 0; q < pow[(lane - 1) * M + l]; ++q) phi *= ul;
                                }
                            s.scr[lane] = phi;
                        }
                        __syncwarp();
                        const int dz = a.nblk * C;
                        double2 *zs = reinterpret_cast<double2 *>(s.scr + MAXBLK), *pz = zs + dz;
                        stream_build_z<CF>(s.x0, s.scr, a.nblk, zs, lane);
                        lift_state<CF>(a.lift_mode, d, xcur, s.va, lane);
                        stream_update<CF>(a.stream_A + (size_t)k * C * dz, a.stream_P + (size_t)k * dz * dz, zs, s.va, dz,
                                          a.stream_discount, pz, pz + dz, lane);
                    }
                }

                // shift the guesses (mpc.py:271-272) and, with them, the ADMM warm start
                // (each lane moves its own component through time: no cross-lane hazard)
                if (lane < N) {
#pragma unroll 4
                    for (int t = 0; t < H; ++t) Xg[t * N + lane] = Xg[(t + 1) * N + lane];
                }
                if (lane < M)
#pragma unroll 1
                    for (int t = 0; t + 1 < H; ++t) {
                        s.Ug[t * M + lane] = s.Ug[(t + 1) * M + lane];
                        s.z[t * M + lane] = s.z[(t + 1) * M + lane];
                        s.y[t * M + lane] = s.y[(t + 1) * M + lane];
                    }
                __syncwarp();

                // built-in exit condition: infidelity of the new plant state below a threshold (mpc.py:289-292)
                if (!a.external_plant && a.exit_infid > 0.0 && a.fid_vec) {
                    const double f = fidelity_of<CF>(a.lift_mode, d, a.fid_vec, xcur, s.va, lane);
                    if (1.0 - f < a.exit_infid) {
                        exit_code = 1;
                        ++step;
                        break;
                    }
                }
            }
        }

        // ---- results
        if (lane == 0) {
            a.exit_code[k] = exit_code;
            a.steps_done[k] = step;
            if (a.counters) {
                int *c = a.counters + (size_t)k * 4;
                if (a.step_begin == 0) c[0] = c[1] = c[2] = c[3] = 0;
                c[0] += cnt.admm;
                c[1] += cnt.factor;
                c[2] += cnt.polish + cnt.kkt;
                c[3] += cnt.solves;
            }
            unsigned long long *fc = reinterpret_cast<unsigned long long *>(a.tab + L.flags + 2);
            if (cnt.fac_herm) atomicAdd(fc, (unsigned long long)cnt.fac_herm);
            if (cnt.fac_full) atomicAdd(fc + 1, (unsigned long long)cnt.fac_full);
        }
        if (a.fidelity && !a.external_plant && a.fid_vec) {
            const double f = fidelity_of<CF>(a.lift_mode, d, a.fid_vec, xcur, s.va, lane);
            if (lane == 0) a.fidelity[k] = a.fidelity_sqrt ? sqrt(fmax(f, 0.0)) : f;
        }
        if (a.state) {
            double *st = a.state + (size_t)k * persist;
            int o = 0;
#pragma unroll 1
            for (int e = lane; e < (H + 1) * N; e += 32) st[o + e] = Xg[e];
            o += (H + 1) * N;
#pragma unroll 1
            for (int e = lane; e < H * M; e += 32) {
                st[o + e] = s.Ug[e];
                st[o + H * M + e] = s.z[e];
                st[o + 2 * H * M + e] = s.y[e];
            }
            o += 3 * H * M;
            if (lane < xdim) {
                st[o + 2 * lane] = xmeas[lane].x;
                st[o + 2 * lane + 1] = xmeas[lane].y;
            }
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------------------
// Stand-alone horizon QP: one warp per instance, dense per-stage operators read from global memory.
// Workspace per instance (doubles): Q [(H+1) N N] | R [H M M] | r [(H+1) N] | qlin [(H+1) N] | ub [H M] | Rub [H M]
// ---------------------------------------------------------------------------------------------------------
template <class CF> __host__ __device__ inline long long qp_ws_doubles(int H) {
    constexpr int N = CF::N, M = CF::M;
    // every block starts on a 16-byte boundary (the stage records behind it are moved with 16-byte cp.async)
    return (long long)(H + 1) * N * N + rup(H * M * M, 2) + 2LL * (H + 1) * N + 2LL * rup(H * M, 2) + ws_doubles<CF>(H);
}

struct QpArgs {
    long long n_inst;
    int H, has_du, has_uprev;
    double sat, du;
    QPSet set;
    const double2 *x_init, *X_bm, *Q_ls, *A_ls, *B_ls, *D_ls;
    const double *U_bm, *R_ls, *u_prev;
    double2 *X_out;
    double *U_out, *obj_out;
    int *status_out, *iters_out;
    double *ws;
    int slab_doubles;
};

template <class CF>
__global__ void __launch_bounds__(CF::MAXW * 32) qp_kernel(const QpArgs a) {
    constexpr int C = CF::C, N = CF::N, M = CF::M;
    extern __shared__ double2 smem2[];
    double *smem = reinterpret_cast<double *>(smem2);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wpc = blockDim.x >> 5;
    const int H = a.H;
    SlabRef sr = {warp * a.slab_doubles, H, 1, C, nullptr};
    const Slab<CF> s = slab_view<CF>(sr);

    for (long long k = (long long)blockIdx.x * wpc + warp; k < a.n_inst; k += (long long)gridDim.x * wpc) {
        double *ws = a.ws + k * qp_ws_doubles<CF>(H);
        double *wQ = ws, *wR = wQ + (size_t)(H + 1) * N * N, *wr = wR + rup(H * M * M, 2), *wql = wr + (H + 1) * N,
               *wub = wql + (H + 1) * N, *wRub = wub + rup(H * M, 2);
        sr.ws = wRub + rup(H * M, 2);
        const double2 *Qk = a.Q_ls + (size_t)k * (H + 1) * C * C;
        const double *Rk = a.R_ls + (size_t)k * H * M * M;
        const double2 *Xb = a.X_bm + (size_t)k * C * (H + 1);
        const double *Ub = a.U_bm + (size_t)k * M * H;
        // ---- realify the instance (optimize.py:21-35)
#pragma unroll 1
        for (int e = lane; e < (H + 1) * N * N; e += 32) {
            const int t = e / (N * N), ij = e % (N * N);
            wQ[e] = realified_sym(Qk + (size_t)t * C * C, C, ij / N, ij % N);
        }
#pragma unroll 1
        for (int e = lane; e < H * M * M; e += 32) {
            const int t = e / (M * M), ij = e % (M * M);
            wR[e] = 0.5 * (Rk[t * M * M + ij] + Rk[t * M * M + (ij % M) * M + ij / M]);
        }
#pragma unroll 1
        for (int e = lane; e < (H + 1) * N; e += 32) {
            const int t = e / N, kk = e % N;
            const double2 v = Xb[(kk % C) * (H + 1) + t];
            wr[e] = kk < C ? v.x : v.y;
        }
#pragma unroll 1
        for (int e = lane; e < H * M; e += 32) wub[e] = Ub[(e % M) * H + e / M];
        __syncwarp();
#pragma unroll 1
        for (int e = lane; e < (H + 1) * N; e += 32) {
            const int t = e / N, kk = e % N;
            double acc = 0.0;
            for (int j = 0; j < N; ++j) acc = fma(wQ[(size_t)t * N * N + kk * N + j], wr[t * N + j], acc);
            wql[e] = acc;
        }
#pragma unroll 1
        for (int e = lane; e < H * M; e += 32) {
            const int t = e / M, i = e % M;
            double acc = 0.0;
            for (int j = 0; j < M; ++j) acc = fma(wR[t * M * M + i * M + j], wub[t * M + j], acc);
            wRub[e] = acc;
        }
        // ---- slab: B, D, x0, bounds, cold ADMM start
        const double2 *Bk = a.B_ls + (size_t)k * H * C * M;
        const double2 *Dk = a.D_ls + (size_t)k * H * C;
#pragma unroll 1
        for (int e = lane; e < H * N * M; e += 32) {
            const int t = e / (N * M), rem = e % (N * M), kk = rem / M, i = rem % M;
            const double2 v = Bk[((size_t)t * C + kk % C) * M + i];
            ws_rec<CF>(sr, t)[Rec<CF>::B + Rec<CF>::pair(i, kk)] = kk < C ? v.x : v.y;
        }
#pragma unroll 1
        for (int e = lane; e < H * N; e += 32) {
            const int t = e / N, kk = e % N;
            const double2 v = Dk[(size_t)t * C + kk % C];
            ws_rec<CF>(sr, t)[Rec<CF>::D + kk] = kk < C ? v.x : v.y;
        }
#pragma unroll 1
        for (int e = lane; e < H * M; e += 32) {
            s.z[e] = 0.0;
            s.y[e] = 0.0;
        }
        if (lane < C) {
            const double2 v = a.x_init[(size_t)k * C + lane];
            s.x0[lane] = v.x;
            s.x0[C + lane] = v.y;
        }
        if (lane < M) {
            double lo = -a.sat, hi = a.sat;
            if (a.has_du && a.has_uprev) {   // optimize.py:29-30
                const double up = a.u_prev[(size_t)k * M + lane];
                lo = fmax(lo, up - a.du);
                hi = fmin(hi, up + a.du);
            }
            s.lo0[lane] = lo;
            s.hi0[lane] = hi;
        }
        __syncwarp();

        StageOps ops;
        ops.blocks = a.A_ls + (size_t)k * H * C * C;
        ops.nblk = 1;
        ops.stage_stride = C * C;
        ops.soff = 0;
        ops.soffT = 0;
        ops.pow = nullptr;
        ops.pow_soff = 0;
        ops.first_order = 0;
        QPData qp;
        qp.Q = wQ;
        qp.q_stride = N * N;
        qp.Qf = wQ + (size_t)H * N * N;
        qp.R = wR;
        qp.r_stride = M * M;
        qp.r = wr;
        qp.qlin = wql;
        qp.qlinf = wql + H * N;
        qp.ub = wub;
        qp.Rub = wRub;
        qp.sat = a.sat;
        qp.q_diag = 0;
        qp.Q_soff = qp.Qf_soff = qp.R_soff = 0;
        Counters cnt = {0, 0, 0, 0};
        int status = qp_solve<CF, false>(sr, ops, qp, a.set, lane, cnt);
        const double obj = qp_objective<CF>(sr, qp, lane);
        if (!isfinite(obj)) status = 3;   // mpc.py:200
        // empty stage-0 box (u_prev further than du outside the saturation range): infeasible, as the reference's solver says
        if (__any_sync(FULL, lane < M && s.lo0[lane < M ? lane : 0] > s.hi0[lane < M ? lane : 0])) status = 3;
        double2 *Xo = a.X_out + (size_t)k * C * (H + 1);
        double *Uo = a.U_out + (size_t)k * M * H;
        const double *wXo = ws_Xo<CF>(sr);
#pragma unroll 1
        for (int e = lane; e < C * (H + 1); e += 32) {
            const int kk = e / (H + 1), t = e % (H + 1);
            Xo[e] = make_double2(wXo[t * N + kk], wXo[t * N + C + kk]);
        }
#pragma unroll 1
        for (int e = lane; e < M * H; e += 32) Uo[e] = s.Uo[(e % H) * M + e / H];
        if (lane == 0) {
            a.obj_out[k] = obj;
            a.status_out[k] = status;
            if (a.iters_out) {
                a.iters_out[2 * k] = cnt.admm;
                a.iters_out[2 * k + 1] = cnt.factor;
            }
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------------------
// Stand-alone linearisation (linearize.py:61-70)
// ---------------------------------------------------------------------------------------------------------
struct LinArgs {
    long long n_inst;
    int H, nblk;
    const double2 *A_blocks;
    const int *powers;
    const double2 *Xg;
    const double *Ug;
    double2 *A_out, *B_out, *D_out;
    int slab_doubles;
};

// One warp per (instance, stage): the stages of the stand-alone call are independent, so nothing is kept per
// instance -- the model blocks sit in shared memory once per CTA, x_t / u_t / the monomial weights in a few words per
// warp, and the outputs are written straight to HBM with coalesced 16-byte stores.  The row products y_k = N_k x_t
// are spread over the lanes as (k, row) pairs; B_t[:, i] = sum_k dphi_k/du_i y_k and Delta_t = -B_t u_t are then
// assembled per output element.
template <class CF>
__host__ __device__ inline int lin_warp_doubles(int nblk) {
    const int p = nblk - 1;
    return rup(2 * CF::C + CF::M + nblk + p * CF::M + p + 2 * p * CF::C, 2);
}

template <class CF>
__global__ void __launch_bounds__(256) linearize_stage_kernel(const LinArgs a) {
    constexpr int C = CF::C, M = CF::M, CC = C * C;
    extern __shared__ double2 smem2[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    const int H = a.H, nblk = a.nblk, p = nblk - 1;
    double2 *blk = smem2;   // [nblk][C][C]
    double *wbase = reinterpret_cast<double *>(smem2 + (size_t)nblk * CC) + (size_t)warp * lin_warp_doubles<CF>(nblk);
    double2 *xs = reinterpret_cast<double2 *>(wbase);    // x_t [C]
    double2 *ys = xs + C;                                // y_k [p][C]
    double *ut = reinterpret_cast<double *>(ys + p * C); // u_t [M]
    double *phi = ut + M, *dw = phi + nblk, *gk = dw + p * M;   // phi [nblk], dphi [p][M], g_k = sum_i u_i dphi_k/du_i
#pragma unroll 1
    for (int e = threadIdx.x; e < nblk * CC; e += blockDim.x) blk[e] = a.A_blocks[e];
    bool first_order = p == M;
    if (first_order) {
#pragma unroll 1
        for (int e = 0; e < M * M; ++e) first_order &= a.powers[e] == ((e / M == e % M) ? 1 : 0);
    }
    __syncthreads();
    const long long total = a.n_inst * H;
    const long long stride = (long long)gridDim.x * wpc;
    long long item = (long long)blockIdx.x * wpc + warp;
    long long k = item / H;
    int t = (int)(item - k * H);
    const long long sk = stride / H;
    const int st = (int)(stride - sk * H);
    // x_t and u_t of the NEXT item are fetched into registers while the current one is processed
    double2 x_n = make_double2(0.0, 0.0);
    double u_n = 0.0;
    if (item < total) {
        if (lane < C) x_n = a.Xg[(size_t)k * C * (H + 1) + lane * (H + 1) + t];
        if (lane < M) u_n = a.Ug[(size_t)k * M * H + lane * H + t];
    }
#pragma unroll 1
    for (; item < total; item += stride) {
        if (lane < C) xs[lane] = x_n;
        if (lane < M) ut[lane] = u_n;
        {
            int t2 = t + st;
            long long k2 = k + sk;
            if (t2 >= H) {
                t2 -= H;
                ++k2;
            }
            if (item + stride < total) {
                if (lane < C) x_n = a.Xg[(size_t)k2 * C * (H + 1) + lane * (H + 1) + t2];
                if (lane < M) u_n = a.Ug[(size_t)k2 * M * H + lane * H + t2];
            }
        }
        __syncwarp();
        // monomials phi_k(u_t), their derivative weights (linearize.py:37-58) and g_k
        if (first_order) {
            if (lane < M) phi[1 + lane] = ut[lane];
        } else {
#pragma unroll 1
            for (int kb = lane; kb < p; kb += 32) {
                double ph = 1.0, dwl[M];
#pragma unroll
                for (int i = 0; i < M; ++i) dwl[i] = (double)a.powers[kb * M + i];
#pragma unroll
                for (int l = 0; l < M; ++l) {
                    const int e = a.powers[kb * M + l];
                    const double ul = ut[l];
                    double pw = 1.0, pwm1 = 1.0;
#pragma unroll 1
                    for (int q = 0; q < e; ++q) {
                        pwm1 = pw;
                        pw *= ul;
                    }
                    ph *= pw;
#pragma unroll
                    for (int i = 0; i < M; ++i) dwl[i] *= (i == l) ? (e > 0 ? pwm1 : 0.0) : pw;
                }
                double g = 0.0;
#pragma unroll
                for (int i = 0; i < M; ++i) {
                    dw[kb * M + i] = dwl[i];
                    g = fma(dwl[i], ut[i], g);
                }
                phi[1 + kb] = ph;
                gk[kb] = g;
            }
        }
        if (lane == 0) phi[0] = 1.0;
        // y_k[r] = (N_k x_t)[r], one (k, r) pair per lane
        double2 x[C];
#pragma unroll
        for (int j = 0; j < C; ++j) x[j] = xs[j];
#pragma unroll 1
        for (int e = lane; e < p * C; e += 32) {
            const double2 *row = blk + CC + e * C;   // block 1 + e / C, row e % C
            double2 y0 = make_double2(0.0, 0.0), y1 = make_double2(0.0, 0.0);
#pragma unroll
            for (int j = 0; j < C; ++j) {
                if (j & 1) y1 = cfma(row[j], x[j], y1);
                else y0 = cfma(row[j], x[j], y0);
            }
            ys[e] = make_double2(y0.x + y1.x, y0.y + y1.y);
        }
        __syncwarp();
        double2 *Ao = a.A_out + (size_t)item * CC;
#pragma unroll
        for (int q = 0; q < (CC + 31) / 32; ++q) {
            const int e = lane + 32 * q;
            if (e < CC) {
                double2 acc = blk[e];
#pragma unroll 2
                for (int kb = 1; kb < nblk; ++kb) {
                    const double2 v = blk[kb * CC + e];
                    const double w = phi[kb];
                    acc.x = fma(w, v.x, acc.x);
                    acc.y = fma(w, v.y, acc.y);
                }
                Ao[e] = acc;
            }
        }
        double2 *Bo = a.B_out + (size_t)item * C * M;
#pragma unroll
        for (int q = 0; q < (C * M + 31) / 32; ++q) {
            const int e = lane + 32 * q;
            if (e < C * M) {
                const int r = e / M, i = e % M;
                double2 b;
                if (first_order) {
                    b = ys[i * C + r];
                } else {
                    b = make_double2(0.0, 0.0);
#pragma unroll 1
                    for (int kb = 0; kb < p; ++kb) {
                        const double w = dw[kb * M + i];
                        const double2 y = ys[kb * C + r];
                        b.x = fma(w, y.x, b.x);
                        b.y = fma(w, y.y, b.y);
                    }
                }
                Bo[e] = b;
            }
        }
        if (lane < C) {
            double2 d = make_double2(0.0, 0.0);
#pragma unroll 1
            for (int kb = 0; kb < p; ++kb) {
                const double g = first_order ? ut[kb] : gk[kb];
                const double2 y = ys[kb * C + lane];
                d.x = fma(-g, y.x, d.x);
                d.y = fma(-g, y.y, d.y);
            }
            a.D_out[(size_t)item * C + lane] = d;
        }
        __syncwarp();
        t += st;
        k += sk;
        if (t >= H) {
            t -= H;
            ++k;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Stand-alone EXACT linearisation (model mode of SURVEY 8f rank 1): A_t = expm(G(u_t) dt), B_t = d/du [expm(G dt)] x_t,
// Delta_t = -B_t u_t.  One warp per (instance, stage); generators shared by the CTA.
// ---------------------------------------------------------------------------------------------------------
struct ExactArgs {
    long long n_inst;
    int H;
    double dt;
    const double2 *gen;   // [M+1][C][C]
    const double2 *Xg;
    const double *Ug;
    double2 *A_out, *B_out, *D_out;
};

template <class CF> __host__ __device__ inline int exact_warp_complex() { return exact_scratch<CF>() + CF::C + cdiv(CF::M, 2); }

template <class CF>
__global__ void __launch_bounds__(128) exact_linearize_kernel(const ExactArgs a) {
    constexpr int C = CF::C, M = CF::M, CC = C * C;
    extern __shared__ double2 smem2[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    const int H = a.H;
    double2 *gen = smem2;
    double2 *scr = smem2 + (M + 1) * CC + (size_t)warp * exact_warp_complex<CF>();
    double2 *xs = scr + exact_scratch<CF>();
    double *ut = reinterpret_cast<double *>(xs + C);
#pragma unroll 1
    for (int e = threadIdx.x; e < (M + 1) * CC; e += blockDim.x) gen[e] = a.gen[e];
    __syncthreads();
    const long long total = a.n_inst * H;
#pragma unroll 1
    for (long long item = (long long)blockIdx.x * wpc + warp; item < total; item += (long long)gridDim.x * wpc) {
        const long long k = item / H;
        const int t = (int)(item - k * H);
        if (lane < C) xs[lane] = a.Xg[(size_t)k * C * (H + 1) + lane * (H + 1) + t];
        if (lane < M) ut[lane] = a.Ug[(size_t)k * M * H + lane * H + t];
        __syncwarp();
        exact_stage<CF>(gen, ut, xs, a.dt, scr, lane);
        const double2 *T = scr + CC, *b = scr + exact_b_offset<CF>();
#pragma unroll 1
        for (int e = lane; e < CC; e += 32) a.A_out[(size_t)item * CC + e] = T[e];
#pragma unroll 1
        for (int e = lane; e < C * M; e += 32) a.B_out[(size_t)item * C * M + e] = b[(e % M) * C + e / M];
        if (lane < C) {
            double2 d = make_double2(0.0, 0.0);
#pragma unroll
            for (int i = 0; i < M; ++i) {
                d.x = fma(-b[i * C + lane].x, ut[i], d.x);
                d.y = fma(-b[i * C + lane].y, ut[i], d.y);
            }
            a.D_out[(size_t)item * C + lane] = d;
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------------------
// Stand-alone line search (mpc.py:101-125); costs and references shared by all instances.
// Workspace (doubles): Q [(H+1) N N] | R [H M M] | r [(H+1) N] | ub [H M]
// ---------------------------------------------------------------------------------------------------------
__global__ void line_search_prep(int C, int M, int H, const double2 *Q_ls, const double *R_ls, const double2 *X_ref,
                                 const double *U_ref, double *ws) {
    const int N = 2 * C;
    double *wQ = ws, *wR = wQ + (size_t)(H + 1) * N * N, *wr = wR + H * M * M, *wub = wr + (H + 1) * N;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
    for (int e = tid; e < (H + 1) * N * N; e += nt) {
        const int t = e / (N * N), ij = e % (N * N);
        wQ[e] = realified_sym(Q_ls + (size_t)t * C * C, C, ij / N, ij % N);
    }
#pragma unroll 1
    for (int e = tid; e < H * M * M; e += nt) {
        const int t = e / (M * M), ij = e % (M * M);
        wR[e] = 0.5 * (R_ls[t * M * M + ij] + R_ls[t * M * M + (ij % M) * M + ij / M]);
    }
    for (int e = tid; e < (H + 1) * N; e += nt) {
        const int t = e / N, kk = e % N;
        const double2 v = X_ref[(kk % C) * (H + 1) + t];
        wr[e] = kk < C ? v.x : v.y;
    }
#pragma unroll 1
    for (int e = tid; e < H * M; e += nt) wub[e] = U_ref[(e % M) * H + e / M];
}

struct LsArgs {
    long long n_inst;
    int H;
    const double2 *Xg, *Xo;
    const double *Ug, *Uo;
    double *alpha_out, *step_out;
    const double *ws;
    int slab_doubles;
};

template <class CF>
__global__ void __launch_bounds__(CF::MAXW * 32) line_search_kernel(const LsArgs a) {
    constexpr int C = CF::C, N = CF::N, M = CF::M;
    extern __shared__ double2 smem2[];
    double *smem = reinterpret_cast<double *>(smem2);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wpc = blockDim.x >> 5;
    const int H = a.H;
    const int slab_only = rup(Slab<CF>::doubles(H, 1, C), 2);
    const SlabRef sr = {warp * a.slab_doubles, H, 1, C, smem + (size_t)warp * a.slab_doubles + slab_only};
    const Slab<CF> s = slab_view<CF>(sr);
    double *wXg = ws_Xg<CF>(sr), *wXo = ws_Xo<CF>(sr);
    QPData qp;
    qp.Q = a.ws;
    qp.q_stride = N * N;
    qp.Qf = a.ws + (size_t)H * N * N;
    qp.R = a.ws + (size_t)(H + 1) * N * N;
    qp.r_stride = M * M;
    qp.r = qp.R + H * M * M;
    qp.ub = qp.r + (H + 1) * N;
    qp.qlin = qp.qlinf = qp.Rub = nullptr;
    qp.sat = 0.0;
    qp.q_diag = 0;
    qp.Q_soff = qp.Qf_soff = qp.R_soff = 0;
    for (long long k = (long long)blockIdx.x * wpc + warp; k < a.n_inst; k += (long long)gridDim.x * wpc) {
        const double2 *Xgk = a.Xg + (size_t)k * C * (H + 1), *Xok = a.Xo + (size_t)k * C * (H + 1);
        const double *Ugk = a.Ug + (size_t)k * M * H, *Uok = a.Uo + (size_t)k * M * H;
#pragma unroll 1
        for (int e = lane; e < (H + 1) * N; e += 32) {
            const int t = e / N, kk = e % N;
            const double2 g = Xgk[(kk % C) * (H + 1) + t], o = Xok[(kk % C) * (H + 1) + t];
            wXg[e] = kk < C ? g.x : g.y;
            wXo[e] = kk < C ? o.x : o.y;
        }
#pragma unroll 1
        for (int e = lane; e < H * M; e += 32) {
            s.Ug[e] = Ugk[(e % M) * H + e / M];
            s.Uo[e] = Uok[(e % M) * H + e / M];
        }
        __syncwarp();
        double alpha, stp;
        line_search<CF, false>(sr, qp, lane, alpha, stp);
        if (lane == 0) {
            a.alpha_out[k] = alpha;
            a.step_out[k] = stp;
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------------------
// Plant step(s) (experiment.py:202-212): one warp per member, d <= 5
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) expm_step_kernel(long long n, int d, int m, int n_seg, double dt, const double2 *H0,
                                                        const double2 *H1, int shared_ham, const double *u,
                                                        const double2 *rho_in, double2 *rho_out, double2 *prop_out) {
    extern __shared__ double2 smem2[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    const int dd = d * d;
    double2 *base = smem2 + (size_t)warp * 5 * dd;
    double2 *rho = base, *Hm = base + dd, *G = base + 2 * dd, *T0 = base + 3 * dd, *T1 = base + 4 * dd;
    for (long long k = (long long)blockIdx.x * wpc + warp; k < n; k += (long long)gridDim.x * wpc) {
        const double2 *H0k = H0 + (shared_ham ? 0 : (size_t)k * dd);
        const double2 *H1k = H1 + (shared_ham ? 0 : (size_t)k * m * dd);
        if (lane < dd) rho[lane] = rho_in[(size_t)k * dd + lane];
        __syncwarp();
        for (int sgm = 0; sgm < n_seg; ++sgm) {
            if (lane < dd) {
                double2 h = H0k[lane];
                for (int i = 0; i < m; ++i) {
                    const double uu = u[((size_t)k * n_seg + sgm) * m + i];
                    const double2 h1 = H1k[i * dd + lane];
                    h.x = fma(uu, h1.x, h.x);
                    h.y = fma(uu, h1.y, h.y);
                }
                Hm[lane] = h;
            }
            __syncwarp();
            expm_minus_i(Hm, dt, d, G, T0, T1, lane);
            if (prop_out && lane < dd) prop_out[((size_t)k * n_seg + sgm) * dd + lane] = T0[lane];
            conjugate(rho, T0, d, G, lane);
            if (lane < dd) rho_out[((size_t)k * n_seg + sgm) * dd + lane] = rho[lane];
            __syncwarp();
        }
    }
}

// Same computation with ONE THREAD per member and the matrices in registers (d <= 4): no shared memory, no warp
// syncs, every lane busy.  The warp-per-member version above keeps 32 - d*d lanes idle and is latency bound
// (5 % of HBM on 3x3 matrices); this one streams parameters and states near the HBM / fp64 limits.
template <int D>
__global__ void __launch_bounds__(128) expm_step_kernel_t(long long n, int m, int n_seg, double dt, const double2 *H0,
                                                          const double2 *H1, int shared_ham, const double *u,
                                                          const double2 *rho_in, double2 *rho_out, double2 *prop_out) {
    constexpr int DD = D * D;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        const double2 *H0k = H0 + (shared_ham ? 0 : (size_t)k * DD);
        const double2 *H1k = H1 + (shared_ham ? 0 : (size_t)k * m * DD);
        double2 rho[DD];
#pragma unroll
        for (int e = 0; e < DD; ++e) rho[e] = rho_in[(size_t)k * DD + e];
        for (int sgm = 0; sgm < n_seg; ++sgm) {
            double2 G[DD], T[DD];
#pragma unroll
            for (int e = 0; e < DD; ++e) G[e] = H0k[e];
            for (int i = 0; i < m; ++i) {
                const double uu = u[((size_t)k * n_seg + sgm) * m + i];
#pragma unroll
                for (int e = 0; e < DD; ++e) {
                    const double2 h1 = H1k[i * DD + e];
                    G[e].x = fma(uu, h1.x, G[e].x);
                    G[e].y = fma(uu, h1.y, G[e].y);
                }
            }
            // G = -i H dt, 1-norm, scaling by a power of two to ||G||_1 <= 1/2 (same schedule as expm_minus_i)
            double nrm = 0.0;
#pragma unroll
            for (int j = 0; j < D; ++j) {
                double cs = 0.0;
#pragma unroll
                for (int i = 0; i < D; ++i) {
                    const double2 h = G[i * D + j];
                    G[i * D + j] = make_double2(h.y * dt, -h.x * dt);
                    cs += hypot(h.y * dt, h.x * dt);
                }
                nrm = fmax(nrm, cs);
            }
            int sq = 0;
            while (nrm > 0.5 && sq < 40) {
                nrm *= 0.5;
                ++sq;
            }
            const double sc = ldexp(1.0, -sq);
#pragma unroll
            for (int e = 0; e < DD; ++e) {
                G[e].x *= sc;
                G[e].y *= sc;
                T[e] = make_double2((e / D == e % D) ? 1.0 : 0.0, 0.0);
            }
            if constexpr (D <= 3) {
                // degree-17 Taylor polynomial in Paterson-Stockmeyer form: 2 products for G^2, G^3, then 5 Horner steps in
                // G^3 with T_j = T_{j+1} G^3 + (c_{3j} I + c_{3j+1} G + c_{3j+2} G^2), c_k = 1/k!  (16 products as a Horner)
                double2 G2[DD], G3[DD];
#pragma unroll
                for (int i = 0; i < D; ++i)
#pragma unroll
                    for (int j = 0; j < D; ++j) {
                        double2 acc = make_double2(0.0, 0.0);
#pragma unroll
                        for (int q = 0; q < D; ++q) acc = cfma(G[i * D + q], G[q * D + j], acc);
                        G2[i * D + j] = acc;
                    }
#pragma unroll
                for (int i = 0; i < D; ++i)
#pragma unroll
                    for (int j = 0; j < D; ++j) {
                        double2 acc = make_double2(0.0, 0.0);
#pragma unroll
                        for (int q = 0; q < D; ++q) acc = cfma(G2[i * D + q], G[q * D + j], acc);
                        G3[i * D + j] = acc;
                    }
                double c2 = 1.0 / 355687428096000.0;   // 1/17!
                double c1 = c2 * 17.0, c0 = c1 * 16.0;
#pragma unroll
                for (int e = 0; e < DD; ++e)
                    T[e] = make_double2(fma(c2, G2[e].x, fma(c1, G[e].x, (e / D == e % D) ? c0 : 0.0)),
                                        fma(c2, G2[e].y, c1 * G[e].y));
#pragma unroll 1
                for (int jb = 4; jb >= 0; --jb) {
                    c2 = c0 * (double)(3 * jb + 3);
                    c1 = c2 * (double)(3 * jb + 2);
                    c0 = c1 * (double)(3 * jb + 1);
                    double2 V[DD];
#pragma unroll
                    for (int i = 0; i < D; ++i)
#pragma unroll
                        for (int j = 0; j < D; ++j) {
                            double2 acc = make_double2(fma(c2, G2[i * D + j].x, fma(c1, G[i * D + j].x, i == j ? c0 : 0.0)),
                                                       fma(c2, G2[i * D + j].y, c1 * G[i * D + j].y));
#pragma unroll
                            for (int q = 0; q < D; ++q) acc = cfma(T[i * D + q], G3[q * D + j], acc);
                            V[i * D + j] = acc;
                        }
#pragma unroll
                    for (int e = 0; e < DD; ++e) T[e] = V[e];
                }
            } else {
                // Horner: T = I + G/1 (I + G/2 (I + ... (I + G/16)))
#pragma unroll 1
                for (int kk = 16; kk >= 1; --kk) {
                    const double inv = 1.0 / (double)kk;
                    double2 V[DD];
#pragma unroll
                    for (int i = 0; i < D; ++i)
#pragma unroll
                        for (int j = 0; j < D; ++j) {
                            double2 acc = make_double2(0.0, 0.0);
#pragma unroll
                            for (int q = 0; q < D; ++q) acc = cfma(G[i * D + q], T[q * D + j], acc);
                            V[i * D + j] = make_double2(fma(acc.x, inv, i == j ? 1.0 : 0.0), acc.y * inv);
                        }
#pragma unroll
                    for (int e = 0; e < DD; ++e) T[e] = V[e];
                }
            }
#pragma unroll 1
            for (int q2 = 0; q2 < sq; ++q2) {
                double2 V[DD];
#pragma unroll
                for (int i = 0; i < D; ++i)
#pragma unroll
                    for (int j = 0; j < D; ++j) {
                        double2 acc = make_double2(0.0, 0.0);
#pragma unroll
                        for (int q = 0; q < D; ++q) acc = cfma(T[i * D + q], T[q * D + j], acc);
                        V[i * D + j] = acc;
                    }
#pragma unroll
                for (int e = 0; e < DD; ++e) T[e] = V[e];
            }
            if (prop_out) {
#pragma unroll
                for (int e = 0; e < DD; ++e) prop_out[((size_t)k * n_seg + sgm) * DD + e] = T[e];
            }
            // rho <- T rho T^dagger
            double2 V[DD];
#pragma unroll
            for (int i = 0; i < D; ++i)
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    double2 acc = make_double2(0.0, 0.0);
#pragma unroll
                    for (int q = 0; q < D; ++q) acc = cfma(T[i * D + q], rho[q * D + j], acc);
                    V[i * D + j] = acc;
                }
#pragma unroll
            for (int i = 0; i < D; ++i)
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    double2 acc = make_double2(0.0, 0.0);
#pragma unroll
                    for (int q = 0; q < D; ++q) {
                        const double2 tc = T[j * D + q];
                        acc = cfma(V[i * D + q], make_double2(tc.x, -tc.y), acc);
                    }
                    rho[i * D + j] = acc;
                }
#pragma unroll
            for (int e = 0; e < DD; ++e) rho_out[((size_t)k * n_seg + sgm) * DD + e] = rho[e];
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Taylor discretisation (vectorize.py:8-49): one CTA per member.  Recurrence on word length: the sum of all
// words of length k with control-exponent tuple e is W_k[e] = sum_j W_{k-1}[e - 1_j] L_j  (1_0 = 0).
// smem: cur [p1][c*c] | nxt [p1][c*c] | acc [p1][c*c] complex, succ [p1][m+1] int
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) taylor_kernel(long long n, int c, int m, int order, int p1, double dt, const double2 *L,
                                                     const int *powers, double2 *out) {
    extern __shared__ double2 smem2[];
    const int cc = c * c;
    double2 *cur = smem2, *nxt = cur + (size_t)p1 * cc, *acc = nxt + (size_t)p1 * cc;
    int *succ = reinterpret_cast<int *>(acc + (size_t)p1 * cc);   // succ[e][j]: index of powers[e] + 1_j, or -1
    const int tid = threadIdx.x, nt = blockDim.x;
#pragma unroll 1
    for (int e = tid; e < p1 * (m + 1); e += nt) {
        const int src = e / (m + 1), j = e % (m + 1);
        int found = -1;
        if (j == 0) found = src;
        else
#pragma unroll 1
            for (int q = 0; q < p1 && found < 0; ++q) {
                bool same = true;
                for (int l = 0; l < m; ++l) same &= powers[q * m + l] == powers[src * m + l] + (l == j - 1 ? 1 : 0);
                if (same) found = q;
            }
        succ[e] = found;
    }
    __syncthreads();
    for (long long k = blockIdx.x; k < n; k += gridDim.x) {
        const double2 *Lk = L + (size_t)k * (m + 1) * cc;
        // constant row is the all-zero exponent tuple: find it (row 0 in the reference's ordering)
#pragma unroll 1
        for (int e = tid; e < p1 * cc; e += nt) {
            const int blk = e / cc, ij = e % cc;
            bool zero = true;
            for (int l = 0; l < m; ++l) zero &= powers[blk * m + l] == 0;
            const double2 v = make_double2((zero && ij / c == ij % c) ? 1.0 : 0.0, 0.0);
            cur[e] = v;
            acc[e] = v;
        }
        __syncthreads();
        double pref = 1.0;
        for (int ord = 1; ord <= order; ++ord) {
            pref *= dt / (double)ord;
#pragma unroll 1
            for (int e = tid; e < p1 * cc; e += nt) {
                const int dst = e / cc, ij = e % cc, i = ij / c, jcol = ij % c;
                double2 sum = make_double2(0.0, 0.0);
                for (int src = 0; src < p1; ++src)
                    for (int j = 0; j <= m; ++j) {
                        if (succ[src * (m + 1) + j] != dst) continue;
                        const double2 *W = cur + (size_t)src * cc + i * c;
                        const double2 *Lj = Lk + (size_t)j * cc + jcol;
                        for (int q = 0; q < c; ++q) sum = cfma(W[q], Lj[q * c], sum);
                    }
                nxt[e] = sum;
            }
            __syncthreads();
#pragma unroll 1
            for (int e = tid; e < p1 * cc; e += nt) {
                const double2 v = nxt[e];
                cur[e] = v;
                acc[e].x = fma(pref, v.x, acc[e].x);
                acc[e].y = fma(pref, v.y, acc[e].y);
            }
            __syncthreads();
        }
        // hstack layout: out[i][blk*c + j]
        double2 *ok = out + (size_t)k * c * c * p1;
#pragma unroll 1
        for (int e = tid; e < p1 * cc; e += nt) {
            const int blk = e / cc, ij = e % cc, i = ij / c, j = ij % c;
            ok[(size_t)i * c * p1 + blk * c + j] = acc[e];
        }
        __syncthreads();
    }
}

__global__ void hist_kernel(long long n, const double *f, double lo, double hi, int nbins, unsigned long long *counts) {
    const double scale = nbins / (hi - lo);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const double v = f[i];
        if (!(v == v)) continue;
        int b = (int)floor((v - lo) * scale);
        b = b < 0 ? 0 : (b >= nbins ? nbins - 1 : b);
        atomicAdd(&counts[b], 1ULL);
    }
}

// register-resident fp64 FMA chains: the denominator of the fp64 roofline, measured on the same part
__global__ void __launch_bounds__(256) fp64_fma_kernel(long long iters, double seed, double *out) {
    double a[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = seed + i + threadIdx.x * 1e-9;
    const double m = 1.0 - 1e-12, c = 1e-13;
    for (long long it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) a[i] = fma(a[i], m, c);
    }
    double sum = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) sum += a[i];
    if (sum == 123.456) out[0] = sum;
}

// fp64 tensor-core probe: mma.sync m8n8k4 f64 chains (DMMA), 8 independent accumulators per warp
__global__ void __launch_bounds__(256) fp64_dmma_kernel(long long iters, double seed, double *out) {
    double c[8][2];
#pragma unroll
    for (int i = 0; i < 8; ++i) c[i][0] = c[i][1] = seed + i;
    const double a = 1.0 - 1e-12 + threadIdx.x * 1e-15, b = 0.25;
    for (long long it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                         : "+d"(c[i][0]), "+d"(c[i][1])
                         : "d"(a), "d"(b));
    }
    double sum = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) sum += c[i][0] + c[i][1];
    if (sum == 123.456) out[0] = sum;
}

// ---------------------------------------------------------------------------------------------------------
// Launch geometry
// ---------------------------------------------------------------------------------------------------------
struct Geometry {
    int warps, ctas, smem, slab_doubles, shared_doubles;
};

static int device_props(int *sms, int *max_smem) {
    int dev = 0;
    M4Q_CUDA(cudaGetDevice(&dev));
    M4Q_CUDA(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
    M4Q_CUDA(cudaDeviceGetAttribute(max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    return 0;
}

// warps per CTA: as many slabs as fit in shared memory (<= 16), grid = SMs * resident CTAs
template <class KernelT>
static int plan(KernelT kernel, int max_warps, int slab_doubles, int shared_doubles, long long n_units, bool have_device,
                Geometry *g) {
    int sms = 148, max_smem = 232448;
    if (have_device && device_props(&sms, &max_smem) != 0) return -1;
    const long long slab_b = (long long)slab_doubles * 8, shared_b = (long long)shared_doubles * 8;
    if (shared_b + slab_b > max_smem) return fail("horizon too long for the shared-memory slab of this (c, m) instantiation");
    int warps = (int)((max_smem - shared_b) / slab_b);
    if (warps > max_warps) warps = max_warps;
    if (const char *ov = getenv("M4Q_MAX_WARPS")) {   // measurement aid: cap the members per CTA
        const int w = atoi(ov);
        if (w >= 1 && w < warps) warps = w;
    }
    // Less than one round of resident warps: spread the members over all SMs (narrower CTAs) instead of filling some SMs
    // and leaving the others empty -- a member's speed depends on how many warps share its SM's pipes and caches
    // (592 order-1 H = 100 members: 148 CTAs x 4 warps instead of 60 x 10; 4,096 qubits: 148 x 28 instead of 128 x 32)
    if (!getenv("M4Q_MAX_WARPS") && n_units > 0 && n_units < (long long)sms * warps) {
        const int w = (int)((n_units + sms - 1) / sms);
        warps = w < 1 ? 1 : w;
    }
    g->slab_doubles = slab_doubles;
    g->shared_doubles = shared_doubles;
    int per_sm = 1;
    auto residency = [&](int w, int *out) -> int {
        g->warps = w;
        g->smem = (int)(shared_b + (long long)w * slab_b);
        if (have_device) {
            M4Q_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, g->smem));
            M4Q_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(out, kernel, w * 32, g->smem));
            if (*out < 1) return fail("kernel does not fit on an SM (registers x threads)");
        } else {
            *out = (int)(max_smem / (g->smem + 1024));
            if (*out < 1) *out = 1;
        }
        return 0;
    };
    if (residency(warps, &per_sm) != 0) return -1;
    // Few waves (strong scaling: a fixed ensemble split over several GPUs leaves each one a handful of rounds of
    // resident warps): the last, partly filled round costs as much as a full one, so pick the CTA width that fills it.
    // Members take about the same time each and a round of w resident warps per SM about t0 + w (measured on the
    // transmon, 10..16 warps: 13.9 .. 18.7 ms, i.e. t0 = 7.4 in units of the per-warp slope); minimise
    // ceil(n / (SMs w)) (t0 + w) over the widths that still run one CTA per SM.  8,192 transmons on one B200:
    // 16 warps 113.3 k trajectories/s, 14 warps 115.1 k (3.95 rounds instead of 3.46).  M4Q_TAIL_AWARE=0 disables.
    {
        const char *ta = getenv("M4Q_TAIL_AWARE");
        const long long full = (long long)sms * warps;
        if ((!ta || atoi(ta) != 0) && !getenv("M4Q_MAX_WARPS") && per_sm == 1 && n_units > full && n_units < 8 * full) {
            double best = 0.0;
            int best_w = warps;
            for (int w = warps; 2 * w > warps; --w) {
                const long long rounds = (n_units + (long long)sms * w - 1) / ((long long)sms * w);
                const double cost = (double)rounds * (7.4 + w);
                if (best == 0.0 || cost < best * 0.995) {
                    best = cost;
                    best_w = w;
                }
            }
            if (best_w != warps) {
                warps = best_w;
                if (residency(warps, &per_sm) != 0) return -1;
            }
        }
    }
    long long ctas = (long long)sms * per_sm;
    const long long need = (n_units + warps - 1) / warps;
    if (need < ctas) ctas = need < 1 ? 1 : need;
    g->ctas = (int)ctas;
    return 0;
}

static QPSet qp_settings(const m4q_qp_settings *s) {
    QPSet q;
    q.rho = (s && s->rho > 0) ? s->rho : 0.1;
    q.alpha = (s && s->alpha > 0) ? s->alpha : 1.6;
    q.polish = s ? s->polish : 1;
    q.eps = (s && s->eps > 0) ? s->eps : (q.polish ? 1e-2 : 1e-5);
    q.max_admm = (s && s->max_admm > 0) ? s->max_admm : 400;
    q.max_polish = (s && s->max_polish > 0) ? s->max_polish : 8;
    q.admm_first = s ? s->admm_first : 0;
    q.adaptive_rho = (s && s->adaptive_rho < 0) ? 0 : 1;
    q.kkt_mode = (s && s->kkt_fallback > 0 && q.polish) ? s->kkt_fallback : 0;
    q.kkt = nullptr;   // set by the launchers when kkt_mode != 0
    return q;
}

template <class CF> static int mpc_shared_doubles(int nblk) {
    // model blocks | Q | Qf | R | monomial exponents | (c multiple of 8) transposed copies of N_1..N_p for linearize()
    return rup(2 * nblk * CF::C * CF::C + 2 * CF::N * CF::N + rup(CF::M * CF::M, 2) + rup(cdiv(nblk * CF::M, 2) + 1, 2) +
               (CF::C % 8 == 0 ? 2 * (nblk - 1) * CF::C * CF::C : 0), 16);   // slabs start on 128-byte boundaries
}

template <class CF> static int mpc_geometry(const m4q_mpc_problem *p, long long n, bool have_device, Geometry *g) {
    const int dd = p->d * p->d;
    if (!Slab<CF>::scratch_fits(p->p + 1, cmax(dd, CF::C))) return fail("model / plant too large for the slab scratch");
    if (p->streaming && MAXBLK + 4 * (p->p + 1) * CF::C > Slab<CF>::scratch_doubles())
        return fail("streaming model too large for the slab scratch (z and P z, 2 x c (p + 1) complex)");
    const int slab = rup(rup(Slab<CF>::doubles(p->horizon, p->p + 1, cmax(dd, CF::C)), 2) +
                             (p->model_per_member ? 2 * (p->p + 1) * CF::C * CF::C : 0), 16);
    if (p->model_mode == M4Q_MODEL_EXACT)
        return plan(mpc_kernel<CF, true>, CF::MAXW, slab, mpc_shared_doubles<CF>(p->p + 1), n, have_device, g);
    return plan(mpc_kernel<CF, false>, CF::MAXW, slab, mpc_shared_doubles<CF>(p->p + 1), n, have_device, g);
}

// The index involution sigma of the lift: the model state of a Hermitian plant state satisfies x_sigma(k) = conj(x_k).
//   identity lift, vec(rho) of a dA x dA matrix (external plant: c must be a square): transpose
//   trunc32: the 2 x 2 block, transpose;  coupled: transpose inside each stacked dA x dA block
//   process, vec(U (x) U^*): swap of the two tensor factors, (i d + k) d^2 + (j d + l) <-> (k d + i) d^2 + (l d + j)
// Returns false when there is none to use (exact model mode: the factor stays realified).
static bool herm_sigma(const m4q_mpc_problem *p, int *sig) {
    const int c = p->c, d = p->d;
    if (p->model_mode != M4Q_MODEL_TAYLOR || c < 1 || c > 32) return false;
    auto transpose = [&](int off, int n) {
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j) sig[off + i * n + j] = off + j * n + i;
    };
    if (p->lift_mode == M4Q_LIFT_IDENTITY) {
        int n = 0;
        while ((n + 1) * (n + 1) <= c) ++n;
        if (n * n != c) return false;
        transpose(0, n);
    } else if (p->lift_mode == M4Q_LIFT_TRUNC32) {
        if (c != 4) return false;
        transpose(0, 2);
    } else if (p->lift_mode == M4Q_LIFT_COUPLED) {
        int n = 0;
        while (2 * (n + 1) * (n + 1) <= c) ++n;
        if (2 * n * n != c) return false;
        transpose(0, n);
        transpose(n * n, n);
    } else if (p->lift_mode == M4Q_LIFT_PROCESS) {
        if (d < 1 || d * d * d * d != c) return false;
        const int d2 = d * d;
        for (int row = 0; row < d2; ++row)
            for (int col = 0; col < d2; ++col) {
                const int i = row / d, k = row % d, j = col / d, l = col % d;
                sig[row * d2 + col] = (k * d + i) * d2 + (l * d + j);
            }
    } else {
        return false;
    }
    return true;
}

template <class CF>
static int launch_mpc(const m4q_mpc_problem *p, long long n, const MpcArgs &base, cudaStream_t st) {
    Geometry g;
    if (mpc_geometry<CF>(p, n, true, &g) != 0) return -1;
    MpcArgs a = base;
    a.slab_doubles = g.slab_doubles;
    a.shared_doubles = g.shared_doubles;
    // per-warp workspaces follow the shared tables (sized by m4q_mpc_table_bytes for the widest launch)
    a.ws = a.tab + rup(TableLayout(CF::N, CF::M, p->n_targ).total, 2);
    // M4Q_HERM_FACTOR=0 keeps every factorisation realified (measurement aid, read per launch)
    HermSigma hs;
    memset(&hs, 0, sizeof(hs));
    const char *hv = getenv("M4Q_HERM_FACTOR");
    hs.ok = CF::HERM && (!hv || atoi(hv) != 0) && herm_sigma(p, hs.sig);
    build_tables<<<1, 256, 0, st>>>(CF::C, CF::M, p->n_targ, reinterpret_cast<const double2 *>(p->Q),
                                    reinterpret_cast<const double2 *>(p->Qf), p->R,
                                    reinterpret_cast<const double2 *>(p->X_targ), p->U_targ, a.tab, hs,
                                    p->model_per_member ? nullptr : reinterpret_cast<const double2 *>(p->A_blocks),
                                    p->p + 1);
    M4Q_CUDA(cudaGetLastError());
    // The workspaces are rewritten every QP; ask L2 to keep them (persisting lines) instead of writing them back to
    // HBM.  Best effort: M4Q_L2_PERSIST=0 switches it off, failures are ignored.
    bool window = false;
    const char *pv = getenv("M4Q_L2_PERSIST");
    if (!pv || atoi(pv) != 0) {
        int dev = 0, max_persist = 0, max_window = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev);
        cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, dev);
        size_t ws_bytes = (size_t)g.ctas * g.warps * ws_doubles<CF>(p->horizon) * sizeof(double);
        if (max_persist > 0 && max_window > 0) {
            const size_t want = ws_bytes < (size_t)max_persist ? ws_bytes : (size_t)max_persist;
            static size_t reserved_per_device[64] = {0};     // the limit is a per-device setting
            size_t &reserved = reserved_per_device[dev & 63];
            if (want > reserved && cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess) reserved = want;
            cudaStreamAttrValue attr;
            memset(&attr, 0, sizeof(attr));
            attr.accessPolicyWindow.base_ptr = a.ws;
            attr.accessPolicyWindow.num_bytes = ws_bytes < (size_t)max_window ? ws_bytes : (size_t)max_window;
            attr.accessPolicyWindow.hitRatio = reserved >= ws_bytes ? 1.0f : (float)reserved / (float)ws_bytes;
            attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
            // the part of the window that does not get the persisting property: "normal" lets it compete for the rest of
            // L2 (with 16 warps per SM the workspaces are 100 MB, more than the persisting carve-out), "streaming" would
            // evict it first and re-read it from HBM on every sweep
            const char *mp = getenv("M4Q_L2_MISS");
            attr.accessPolicyWindow.missProp = (mp && mp[0] == 's') ? cudaAccessPropertyStreaming : cudaAccessPropertyNormal;
            window = cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &attr) == cudaSuccess;
        }
        cudaGetLastError();
    }
    // the pivoted-KKT workspaces (one per resident warp, m4q_kkt.cuh) follow the other per-warp arrays
    if (a.set.kkt_mode)
        a.set.kkt = a.ws + (size_t)g.ctas * g.warps *
                               (ws_doubles<CF>(p->horizon) + (p->model_mode == M4Q_MODEL_EXACT ? 2 * p->horizon * CF::C * CF::C : 0));
    if (p->model_mode == M4Q_MODEL_EXACT) {
        a.ws_exact = a.ws + (size_t)g.ctas * g.warps * ws_doubles<CF>(p->horizon);
        mpc_kernel<CF, true><<<g.ctas, g.warps * 32, g.smem, st>>>(a);
    } else {
        a.ws_exact = nullptr;
        mpc_kernel<CF, false><<<g.ctas, g.warps * 32, g.smem, st>>>(a);
    }
    M4Q_CUDA(cudaGetLastError());
    if (window) {   // do not leave the window on the caller's stream
        cudaStreamAttrValue attr;
        memset(&attr, 0, sizeof(attr));
        attr.accessPolicyWindow.num_bytes = 0;
        cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &attr);
        cudaGetLastError();
    }
    return 0;
}

// The compiled (c, m) instantiations: c in {4, 8, 9, 16} (qubit, stacked two-qubit, qutrit and two-qubit or process
// vectors), one to four controls.  X(c, m, args...) is applied to each; the dispatch, m4q_supported and the workspace
// sizes are generated from this one list.
#define M4Q_SHAPES(X, ...)                                                                                             \
    X(4, 1, __VA_ARGS__) X(4, 2, __VA_ARGS__) X(4, 3, __VA_ARGS__) X(4, 4, __VA_ARGS__)                                \
    X(8, 1, __VA_ARGS__) X(8, 2, __VA_ARGS__) X(8, 3, __VA_ARGS__) X(8, 4, __VA_ARGS__)                                \
    X(9, 1, __VA_ARGS__) X(9, 2, __VA_ARGS__) X(9, 3, __VA_ARGS__) X(9, 4, __VA_ARGS__)                                \
    X(16, 1, __VA_ARGS__) X(16, 2, __VA_ARGS__) X(16, 3, __VA_ARGS__) X(16, 4, __VA_ARGS__)

// runs the statements with CF = Cfg<c, m>, or returns the error of an unsupported pair
#define M4Q_DISPATCH_CASE(C_, M_, c, m, ...) if ((c) == C_ && (m) == M_) { using CF = Cfg<C_, M_>; __VA_ARGS__; } else
#define M4Q_DISPATCH(c, m, ...)                                                       \
    do {                                                                              \
        M4Q_SHAPES(M4Q_DISPATCH_CASE, c, m, __VA_ARGS__)                              \
        return fail("unsupported (c, m): no compiled instantiation");                 \
    } while (0)

#define M4Q_SUPPORTED_CASE(C_, M_, c, m) || ((c) == C_ && (m) == M_)
static bool supported(int c, int m) { return false M4Q_SHAPES(M4Q_SUPPORTED_CASE, c, m); }

static int check_problem(const m4q_mpc_problem *p) {
    if (!p) return fail("null problem");
    if (!supported(p->c, p->m)) return fail("unsupported (c, m): no compiled instantiation");
    if (p->p < 1 || p->p + 1 > MAXBLK) return fail("number of monomial blocks out of range");
    if (p->horizon < 1 || p->n_steps < 1 || p->measure_freq < 1) return fail("horizon, n_steps and measure_freq must be >= 1");
    if (p->n_targ < p->n_steps + p->horizon) return fail("X_targ needs at least n_steps + horizon columns");
    if (p->d < 0 || p->d * p->d > 32) return fail("plant dimension out of range (d*d <= 32)");
    if (p->d == 0 && p->lift_mode != M4Q_LIFT_IDENTITY) return fail("d = 0 (external plant) goes with the identity lift");
    if (p->d > 0 && p->lift_mode == M4Q_LIFT_IDENTITY && p->d * p->d != p->c) return fail("identity lift needs d*d == c");
    if (p->lift_mode == M4Q_LIFT_COUPLED && !(p->d == 4 && p->c == 8))
        return fail("coupled lift: two qubits (d = 4, c = 8) is the compiled case");
    if (p->lift_mode == M4Q_LIFT_TRUNC32 && !(p->d == 3 && p->c == 4)) return fail("trunc32 lift needs d = 3, c = 4");
    if (p->model_mode != M4Q_MODEL_TAYLOR && p->model_mode != M4Q_MODEL_EXACT) return fail("unknown model_mode");
    if (p->model_mode == M4Q_MODEL_EXACT && p->p != p->m)
        return fail("exact model mode: A_blocks holds the m + 1 generators, p must equal m");
    if (p->model_mode == M4Q_MODEL_EXACT && p->measure_freq != 1)
        return fail("exact model mode: model steps between measurements are not built, measure_freq must be 1");
    if (p->lift_mode == M4Q_LIFT_PROCESS && !(p->d == 2 && p->c == 16)) return fail("process lift needs d = 2, c = d^4 = 16");
    if (p->lift_mode == M4Q_LIFT_PROCESS && p->measure_freq != 1)
        return fail("process lift: the propagator cannot be recovered from a model step, measure_freq must be 1");
    if (p->lift_mode == M4Q_LIFT_TRUNC32 && p->measure_freq != 1)
        return fail("QExperiment32.proj is not a map back to the plant space (experiment.py:232-235); measure_freq must be 1");
    if (!(p->sat > 0)) return fail("sat is mandatory (optimize.py:43)");
    return 0;
}

}  // namespace m4q

using namespace m4q;

// =========================================================================================================
// C ABI
// =========================================================================================================
extern "C" {

int m4q_version(void) { return M4Q_VERSION; }

const char *m4q_last_error(void) { return g_err.c_str(); }

int m4q_supported(int32_t c, int32_t m) { return supported(c, m) ? 1 : 0; }

int m4q_expm_step_batched(int64_t N, int32_t d, int32_t m, int32_t n_seg, double dt, const double *H0, const double *H1,
                          int32_t shared_hamiltonian, const double *u, const double *rho_in, double *rho_out,
                          double *prop_out, void *stream) {
    if (N <= 0) return 0;
    if (d < 1 || d * d > 32) return fail("plant dimension out of range (d*d <= 32)");
    if (!H0 || !H1 || !u || !rho_in || !rho_out) return fail("null pointer");
    if (d <= 4 && N >= 4096) {   // thread-per-member kernel once there are enough members to fill the GPU
        long long tctas = (N + 127) / 128;
        if (tctas > 148 * 16) tctas = 148 * 16;
#define M4Q_EXPM_T(D_)                                                                                                  \
    expm_step_kernel_t<D_><<<(int)tctas, 128, 0, (cudaStream_t)stream>>>(                                               \
        N, m, n_seg, dt, (const double2 *)H0, (const double2 *)H1, shared_hamiltonian, u, (const double2 *)rho_in,      \
        (double2 *)rho_out, (double2 *)prop_out)
        if (d == 1) M4Q_EXPM_T(1);
        else if (d == 2) M4Q_EXPM_T(2);
        else if (d == 3) M4Q_EXPM_T(3);
        else M4Q_EXPM_T(4);
#undef M4Q_EXPM_T
        M4Q_CUDA(cudaGetLastError());
        return 0;
    }
    const int wpc = 8;
    long long ctas = (N + wpc - 1) / wpc;
    if (ctas > 148 * 8) ctas = 148 * 8;
    const size_t smem = (size_t)wpc * 5 * d * d * sizeof(double2);
    expm_step_kernel<<<(int)ctas, wpc * 32, smem, (cudaStream_t)stream>>>(
        N, d, m, n_seg, dt, (const double2 *)H0, (const double2 *)H1, shared_hamiltonian, u, (const double2 *)rho_in,
        (double2 *)rho_out, (double2 *)prop_out);
    M4Q_CUDA(cudaGetLastError());
    return 0;
}

int m4q_taylor_discretize_batched(int64_t N, int32_t c, int32_t m, int32_t order, int32_t p1, double dt, const double *L,
                                  const int32_t *powers, double *out, void *stream) {
    if (N <= 0) return 0;
    if (!L || !powers || !out) return fail("null pointer");
    const size_t smem = (size_t)3 * p1 * c * c * sizeof(double2) + (size_t)p1 * (m + 1) * sizeof(int);
    if (smem > 227 * 1024) return fail("model too large for the shared-memory discretisation kernel");
    M4Q_CUDA(cudaFuncSetAttribute(taylor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    long long ctas = N > 148 * 4 ? 148 * 4 : N;
    taylor_kernel<<<(int)ctas, 128, smem, (cudaStream_t)stream>>>(N, c, m, order, p1, dt, (const double2 *)L, powers,
                                                                 (double2 *)out);
    M4Q_CUDA(cudaGetLastError());
    return 0;
}

int m4q_linearize_batched(int64_t N, int32_t c, int32_t m, int32_t p, int32_t H, const double *A_blocks,
                          const int32_t *powers, const double *Xg, const double *Ug, double *A_out, double *B_out,
                          double *D_out, void *stream) {
    if (N <= 0) return 0;
    if (p < 1 || p + 1 > MAXBLK) return fail("number of monomial blocks out of range");
    LinArgs a;
    a.n_inst = N;
    a.H = H;
    a.nblk = p + 1;
    a.A_blocks = (const double2 *)A_blocks;
    a.powers = powers;
    a.Xg = (const double2 *)Xg;
    a.Ug = Ug;
    a.A_out = (double2 *)A_out;
    a.B_out = (double2 *)B_out;
    a.D_out = (double2 *)D_out;
    if (H < 1) return fail("linearize: horizon out of range");
    M4Q_DISPATCH(c, m, {
        const int wpc = 8;
        const size_t smem = (size_t)(p + 1) * c * c * sizeof(double2) + (size_t)wpc * lin_warp_doubles<CF>(p + 1) * sizeof(double);
        if (smem > 200 * 1024) return fail("model too large for the shared-memory linearisation kernel");
        M4Q_CUDA(cudaFuncSetAttribute(linearize_stage_kernel<CF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 1;
        M4Q_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, linearize_stage_kernel<CF>, wpc * 32, smem));
        if (per_sm < 1) per_sm = 1;
        long long ctas = (N * H + wpc - 1) / wpc;
        if (ctas > 148LL * per_sm) ctas = 148LL * per_sm;
        linearize_stage_kernel<CF><<<(int)ctas, wpc * 32, smem, (cudaStream_t)stream>>>(a);
    });
    M4Q_CUDA(cudaGetLastError());
    return 0;
}

int m4q_exact_linearize_batched(int64_t N, int32_t c, int32_t m, int32_t H, double dt, const double *generators,
                                const double *Xg, const double *Ug, double *A_out, double *B_out, double *D_out,
                                void *stream) {
    if (N <= 0) return 0;
    if (H < 1) return fail("exact linearize: horizon out of range");
    if (!generators || !Xg || !Ug || !A_out || !B_out || !D_out) return fail("null pointer");
    ExactArgs a;
    a.n_inst = N;
    a.H = H;
    a.dt = dt;
    a.gen = (const double2 *)generators;
    a.Xg = (const double2 *)Xg;
    a.Ug = Ug;
    a.A_out = (double2 *)A_out;
    a.B_out = (double2 *)B_out;
    a.D_out = (double2 *)D_out;
    M4Q_DISPATCH(c, m, {
        const int wpc = 4;
        const size_t smem = ((size_t)(m + 1) * c * c + (size_t)wpc * exact_warp_complex<CF>()) * sizeof(double2);
        M4Q_CUDA(cudaFuncSetAttribute(exact_linearize_kernel<CF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 1;
        M4Q_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, exact_linearize_kernel<CF>, wpc * 32, smem));
        if (per_sm < 1) per_sm = 1;
        long long ctas = (N * H + wpc - 1) / wpc;
        if (ctas > 148LL * per_sm) ctas = 148LL * per_sm;
        exact_linearize_kernel<CF><<<(int)ctas, wpc * 32, smem, (cudaStream_t)stream>>>(a);
    });
    M4Q_CUDA(cudaGetLastError());
    return 0;
}

int64_t m4q_qp_workspace_bytes(int64_t N, int32_t c, int32_t m, int32_t H) {
    M4Q_DISPATCH(c, m, return (int64_t)sizeof(double) * N * qp_ws_doubles<CF>(H));
}

// with room for the pivoted-KKT workspaces of the resident warps (settings.kkt_fallback != 0)
int64_t m4q_qp_workspace_bytes_kkt(int64_t N, int32_t c, int32_t m, int32_t H) {
    const int64_t base = m4q_qp_workspace_bytes(N, c, m, H);
    if (base < 0) return -1;
    long long kkt = 0;
    M4Q_DISPATCH(c, m, {
        Geometry g;
        const int slab = rup(Slab<CF>::doubles(H, 1, CF::C), 2);
        int count = 0;
        const bool have_device = cudaGetDeviceCount(&count) == cudaSuccess && count > 0;
        if (!have_device) cudaGetLastError();
        if (plan(qp_kernel<CF>, CF::MAXW, slab, 0, 1LL << 40, have_device, &g) != 0) return -1;
        kkt = (long long)g.ctas * g.warps * Kkt<CF>::doubles(H);
    });
    return base + (int64_t)sizeof(double) * kkt;
}

int m4q_qp_admm_batched(int64_t N, int32_t c, int32_t m, int32_t H, const double *x_init, const double *X_bm,
                        const double *U_bm, const double *Q_ls, const double *R_ls, const double *A_ls, const double *B_ls,
                        const double *D_ls, const double *u_prev, double sat, double du, int32_t has_du,
                        const m4q_qp_settings *settings_host, double *X_out, double *U_out, double *obj_out,
                        int32_t *status_out, int32_t *iters_out, void *workspace, void *stream) {
    if (N <= 0) return 0;
    if (!(sat > 0)) return fail("sat is mandatory (optimize.py:43)");
    if (!workspace) return fail("null workspace");
    QpArgs a;
    a.n_inst = N;
    a.H = H;
    a.has_du = has_du;
    a.has_uprev = u_prev != nullptr;
    a.sat = sat;
    a.du = du;
    a.set = qp_settings(settings_host);
    a.x_init = (const double2 *)x_init;
    a.X_bm = (const double2 *)X_bm;
    a.Q_ls = (const double2 *)Q_ls;
    a.A_ls = (const double2 *)A_ls;
    a.B_ls = (const double2 *)B_ls;
    a.D_ls = (const double2 *)D_ls;
    a.U_bm = U_bm;
    a.R_ls = R_ls;
    a.u_prev = u_prev;
    a.X_out = (double2 *)X_out;
    a.U_out = U_out;
    a.obj_out = obj_out;
    a.status_out = status_out;
    a.iters_out = iters_out;
    a.ws = (double *)workspace;
    M4Q_DISPATCH(c, m, {
        Geometry g;
        const int slab = rup(Slab<CF>::doubles(H, 1, CF::C), 2);
        if (plan(qp_kernel<CF>, CF::MAXW, slab, 0, N, true, &g) != 0) return -1;
        a.slab_doubles = slab;
        if (a.set.kkt_mode) a.set.kkt = a.ws + (size_t)N * qp_ws_doubles<CF>(H);   // sized by m4q_qp_workspace_bytes_kkt
        qp_kernel<CF><<<g.ctas, g.warps * 32, g.smem, (cudaStream_t)stream>>>(a);
    });
    M4Q_CUDA(cudaGetLastError());
    return 0;
}

int64_t m4q_line_search_workspace_bytes(int32_t c, int32_t m, int32_t H) {
    const int N = 2 * c;
    return (int64_t)sizeof(double) * ((int64_t)(H + 1) * N * N + (int64_t)H * m * m + (int64_t)(H + 1) * N + (int64_t)H * m);
}

int m4q_line_search_batched(int64_t N, int32_t c, int32_t m, int32_t H, const double *Q_ls, const double *R_ls,
                            const double *X_ref, const double *U_ref, const double *Xg, const double *Ug, const double *Xo,
                            const double *Uo, double *alpha_out, double *step_out, void *workspace, void *stream) {
    if (N <= 0) return 0;
    if (!workspace) return fail("null workspace");
    line_search_prep<<<32, 256, 0, (cudaStream_t)stream>>>(c, m, H, (const double2 *)Q_ls, R_ls, (const double2 *)X_ref, U_ref,
                                                          (double *)workspace);
    M4Q_CUDA(cudaGetLastError());
    LsArgs a;
    a.n_inst = N;
    a.H = H;
    a.Xg = (const double2 *)Xg;
    a.Xo = (const double2 *)Xo;
    a.Ug = Ug;
    a.Uo = Uo;
    a.alpha_out = alpha_out;
    a.step_out = step_out;
    a.ws = (const double *)workspace;
    M4Q_DISPATCH(c, m, {
        Geometry g;
        const int slab = rup(Slab<CF>::doubles(H, 1, CF::C), 2) + rup(ws_doubles<CF>(H), 2);
        if (plan(line_search_kernel<CF>, CF::MAXW, slab, 0, N, true, &g) != 0) return -1;
        a.slab_doubles = slab;
        line_search_kernel<CF><<<g.ctas, g.warps * 32, g.smem, (cudaStream_t)stream>>>(a);
    });
    M4Q_CUDA(cudaGetLastError());
    return 0;
}

int64_t m4q_mpc_state_bytes(const m4q_mpc_problem *p, int64_t N) {
    if (check_problem(p) != 0) return -1;
    int persist = 0;
    const int dd = p->d * p->d;
    M4Q_DISPATCH(p->c, p->m, { persist = Slab<CF>::persistent_doubles(p->horizon, cmax(dd, CF::C)); });
    return (int64_t)sizeof(double) * N * persist;
}

int64_t m4q_mpc_table_bytes(const m4q_mpc_problem *p) {
    if (check_problem(p) != 0) return -1;
    Geometry g;
    int count = 0;
    const bool have_device = cudaGetDeviceCount(&count) == cudaSuccess && count > 0;
    if (!have_device) cudaGetLastError();
    long long ws = 0;
    M4Q_DISPATCH(p->c, p->m, {
        if (mpc_geometry<CF>(p, 1LL << 40, have_device, &g) != 0) return -1;
        ws = (long long)g.ctas * g.warps * ws_doubles<CF>(p->horizon);
        if (p->model_mode == M4Q_MODEL_EXACT) ws += (long long)g.ctas * g.warps * 2 * p->horizon * CF::C * CF::C;
        if (p->qp.kkt_fallback > 0 && p->qp.polish) ws += (long long)g.ctas * g.warps * Kkt<CF>::doubles(p->horizon);
    });
    return (int64_t)sizeof(double) * (rup(TableLayout(2 * p->c, p->m, p->n_targ).total, 2) + ws);
}

int m4q_mpc_herm_sigma(const m4q_mpc_problem *p, int32_t *sigma) {
    if (check_problem(p) != 0) return -1;
    int sig[32];
    if (!herm_sigma(p, sig)) return 0;
    if (sigma)
        for (int k = 0; k < p->c; ++k) sigma[k] = sig[k];
    return 1;
}

int64_t m4q_mpc_factor_counts_offset(const m4q_mpc_problem *p) {
    if (check_problem(p) != 0) return -1;
    return (int64_t)sizeof(double) * (TableLayout(2 * p->c, p->m, p->n_targ).flags + 2);
}

int m4q_mpc_launch_info(const m4q_mpc_problem *p, int64_t N, int32_t *warps_per_cta, int32_t *ctas, int32_t *smem_bytes) {
    if (check_problem(p) != 0) return -1;
    Geometry g;
    int count = 0;
    const bool have_device = cudaGetDeviceCount(&count) == cudaSuccess && count > 0;
    if (!have_device) cudaGetLastError();
    M4Q_DISPATCH(p->c, p->m, {
        if (mpc_geometry<CF>(p, N > 0 ? (long long)N : 1LL << 40, have_device, &g) != 0) return -1;
    });
    if (warps_per_cta) *warps_per_cta = g.warps;
    if (ctas) *ctas = g.ctas;
    if (smem_bytes) *smem_bytes = g.smem;
    return 0;
}

int m4q_mpc_closed_loop(const m4q_mpc_problem *p, int64_t N, const double *x0, int32_t x0_shared, const double *H0,
                        const double *H1, int32_t shared_hamiltonian, int32_t step_begin, int32_t step_end,
                        int32_t external_plant, double *xs, double *us, int32_t *exit_code, int32_t *steps_done,
                        int32_t *qp_count, int32_t *counters, double *fidelity, void *state, void *tables, void *stream) {
    if (check_problem(p) != 0) return -1;
    if (N <= 0) return 0;
    if (!x0 || !xs || !us || !exit_code || !steps_done || !qp_count || !tables) return fail("null pointer");
    if (!external_plant && (!H0 || !H1)) return fail("plant Hamiltonians are required unless external_plant is set");
    if (!external_plant && p->d == 0) return fail("d = 0 is only valid with external_plant");
    if (step_begin < 0 || step_end > p->n_steps || step_begin >= step_end) return fail("bad step range");
    if ((step_begin > 0 || step_end < p->n_steps) && !state) return fail("a partial step range needs the state buffer");
    MpcArgs a;
    memset(&a, 0, sizeof(a));
    a.H = p->horizon;
    a.S = p->n_steps;
    a.mf = p->measure_freq;
    a.warm_start = p->warm_start;
    a.max_iter = p->max_iter > 0 ? p->max_iter : 100;
    a.lift_mode = p->lift_mode;
    a.has_du = p->has_du;
    a.n_targ = p->n_targ;
    a.d = p->d;
    a.nblk = p->p + 1;
    a.dt = p->dt;
    a.sat = p->sat;
    a.du = p->du;
    a.exit_infid = p->exit_infidelity;
    a.set = qp_settings(&p->qp);
    a.A_blocks = (const double2 *)p->A_blocks;
    a.model_per_member = p->model_per_member != 0;
    a.powers = p->powers;
    a.fid_vec = (const double2 *)p->fid_vec;
    a.tab = (double *)tables;
    a.n_members = N;
    a.x0 = (const double2 *)x0;
    a.x0_shared = x0_shared;
    a.H0 = (const double2 *)H0;
    a.H1 = (const double2 *)H1;
    a.shared_ham = shared_hamiltonian;
    a.step_begin = step_begin;
    a.step_end = step_end;
    a.external_plant = external_plant;
    a.xs = (double2 *)xs;
    a.us = us;
    a.exit_code = exit_code;
    a.steps_done = steps_done;
    a.qp_count = qp_count;
    a.counters = counters;
    a.fidelity = fidelity;
    a.state = (double *)state;
    a.noise_sigma = external_plant ? 0.0 : p->noise_sigma;
    a.noise_seed = p->noise_seed;
    a.member_offset = p->member_offset;
    a.streaming = external_plant ? 0 : p->streaming;
    a.fidelity_sqrt = p->fidelity_sqrt;
    a.stream_discount = p->stream_discount > 0 ? p->stream_discount : 1.0;
    a.stream_A = (double2 *)p->stream_A;
    a.stream_P = (double2 *)p->stream_P;
    if (a.streaming && (!a.stream_A || !a.stream_P)) return fail("streaming needs the per-member stream_A / stream_P buffers");
    if (a.streaming && p->model_mode == M4Q_MODEL_EXACT) return fail("streaming updates belong to the Taylor (DMDc) model");
    M4Q_DISPATCH(p->c, p->m, { return launch_mpc<CF>(p, N, a, (cudaStream_t)stream); });
    return 0;
}

int m4q_hist_fidelity(int64_t N, const double *fidelity, double lo, double hi, int32_t nbins, int64_t *counts, void *stream) {
    if (N <= 0) return 0;
    if (!(hi > lo) || nbins < 1) return fail("bad histogram range");
    long long ctas = (N + 255) / 256;
    if (ctas > 148 * 8) ctas = 148 * 8;
    hist_kernel<<<(int)ctas, 256, 0, (cudaStream_t)stream>>>(N, fidelity, lo, hi, nbins, (unsigned long long *)counts);
    M4Q_CUDA(cudaGetLastError());
    return 0;
}

int m4q_fp64_fma_probe(int32_t ctas, int64_t iters, double *scratch, void *stream) {
    fp64_fma_kernel<<<ctas, 256, 0, (cudaStream_t)stream>>>(iters, 0.5, scratch);
    M4Q_CUDA(cudaGetLastError());
    return 0;
}

int m4q_fp64_dmma_probe(int32_t ctas, int64_t iters, double *scratch, void *stream) {
    fp64_dmma_kernel<<<ctas, 256, 0, (cudaStream_t)stream>>>(iters, 0.5, scratch);
    M4Q_CUDA(cudaGetLastError());
    return 0;
}

}  // extern "C"
