// Five-point essential-matrix RANSAC (replaces cv2.findEssentialMat(p1, p2, K, method=RANSAC, prob,
// threshold) at reference VisualOdometryPipeLine.py:308; spec SURVEY.md A.6/A.7 and the header of
// oracle/emat_oracle.c).
//
// All maxIters 5-subsets are drawn (bit-exact cv::RNG stream) and solved at once; scoring goes in chunks:
//   emat_normalize_kernel   pixels -> normalised double coordinates
//   ransac_samples_kernel<5> (ransac.cuh)
//   emat_solve_kernel       one WARP per sample: Nister five-point in FP64 (Householder null
//                           space, cubic constraints with one monomial per lane, Gauss-Jordan
//                           with one column per lane, det B(z), Aberth roots with one root per
//                           lane, back-substitution) -> up to 10 models
//   emat_score_kernel       (256 points) x (8 samples x <=10 models): Sampson error in double ->
//                           float32, ballot+popc counts, one atomicAdd per warp
//   emat_update_kernel      sequential replay of cv2's loop over (sample, model) counts with the
//                           adaptive iteration bound; hypotheses go through in chunks of 64, 128, 256, ... and a
//                           chunk beyond the bound exits at once (cv2 stops after 10-60 samples)
//   emat_finish_kernel      the winner's E and mask
// Every kernel runs for a batch of independent point sets (sequences) at once, the sequence taken from the grid; each one
// replays cv2's RNG stream and adaptive stop on its own.  One call is the batch of one.
#include "emat.cuh"
#include "mathdev.cuh"
#include "ransac.cuh"

using namespace vo;

#define EM_MAXM 10

// ------------------------------------------------------------------------------------------
// Warp-cooperative Nister five-point solver: ONE WARP per 5-point sample.
//   1. null space of the 5x9 epipolar matrix: Householder QR of its transpose in registers
//      (every lane redundantly, statically indexed); lane c < 4 expands basis vector c.
//   2. the 10 cubic constraints det(E) = 0, 2 E E^T E - tr(E E^T) E = 0 in the 20 monomials of
//      (x, y, z, 1): lane m owns monomial m and sums the trilinear forms over the distinct
//      orderings of its basis triple -> column m of the 10 x 20 coefficient matrix, in registers.
//   3. Gauss-Jordan with partial pivoting: lane = column, pivot column broadcast by shuffles.
//   4. B(z) and the degree-10 determinant polynomial (every lane, registers).
//   5. Aberth-Ehrlich iteration: lane k owns root k, the other roots arrive by shuffles.
//   6. lane k polishes a real root (Newton), back-substitutes x, y and writes its E at the slot
//      given by the ascending-z rank among the valid candidates.
// Monomial order [x3 y3 x2y xy2 x2z x2 y2z y2 xyz xy | xz2 xz x yz2 yz y z3 z2 z 1]; basis index
// x = 0, y = 1, z = 2, 1 = 3.
// ------------------------------------------------------------------------------------------
#define EMW_WARPS 4
struct EmwShared { double N[4][9]; double T[6][10]; };

__constant__ unsigned char EMW_TRI[20][3] = {
    {0, 0, 0}, {1, 1, 1}, {0, 0, 1}, {0, 1, 1}, {0, 0, 2}, {0, 0, 3}, {1, 1, 2}, {1, 1, 3}, {0, 1, 2}, {0, 1, 3},
    {0, 2, 2}, {0, 2, 3}, {0, 3, 3}, {1, 2, 2}, {1, 2, 3}, {1, 3, 3}, {2, 2, 2}, {2, 2, 3}, {2, 3, 3}, {3, 3, 3}};

__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }
__device__ __forceinline__ double warp_max_d(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// reciprocal to ~1 ulp for normal-range arguments: hardware seed + two Newton steps (no slow path)
__device__ __forceinline__ double fast_rcp(double x)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(r, fma(-x, r, 1.0), r);
    r = fma(r, fma(-x, r, 1.0), r);
    return isfinite(r) && r != 0 ? r : 1.0 / x;
}

template <int NA, int NB>
__device__ __forceinline__ void poly1_mul(const double* a, const double* b, double* o)
{
#pragma unroll
    for (int i = 0; i <= NA + NB; ++i) o[i] = 0;
#pragma unroll
    for (int i = 0; i <= NA; ++i)
#pragma unroll
        for (int j = 0; j <= NB; ++j) o[i + j] += a[i] * b[j];
}

// step 1; returns false for a rank-deficient sample (warp-uniform)
__device__ __forceinline__ bool emw_null_space(const double* s1, const double* s2, int lane, double (*Nsm)[9])
{
    double A[9][5], V[5][9], beta[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        const double a = s1[2 * i], b = s1[2 * i + 1], c = s2[2 * i], d = s2[2 * i + 1];
        const double r[9] = {c * a, c * b, c, d * a, d * b, d, a, b, 1.0};
#pragma unroll
        for (int j = 0; j < 9; ++j) A[j][i] = r[j];
    }
    bool ok = true;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        double nrm = 0;
#pragma unroll
        for (int i = k; i < 9; ++i) nrm += A[i][k] * A[i][k];
        nrm = sqrt(nrm);
        if (nrm < 1e-300) ok = false;
        const double alpha = A[k][k] > 0 ? -nrm : nrm;
#pragma unroll
        for (int i = k; i < 9; ++i) V[k][i] = A[i][k];
        V[k][k] -= alpha;
        double vn = 0;
#pragma unroll
        for (int i = k; i < 9; ++i) vn += V[k][i] * V[k][i];
        beta[k] = vn > 0 ? 2 / vn : 0;
#pragma unroll
        for (int j = k; j < 5; ++j) {
            double sdot = 0;
#pragma unroll
            for (int i = k; i < 9; ++i) sdot += V[k][i] * A[i][j];
            sdot *= beta[k];
#pragma unroll
            for (int i = k; i < 9; ++i) A[i][j] -= sdot * V[k][i];
        }
    }
    double e[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) e[i] = (i == 5 + (lane & 3)) ? 1.0 : 0.0;
#pragma unroll
    for (int k = 4; k >= 0; --k) {
        double sdot = 0;
#pragma unroll
        for (int i = k; i < 9; ++i) sdot += V[k][i] * e[i];
        sdot *= beta[k];
#pragma unroll
        for (int i = k; i < 9; ++i) e[i] -= sdot * V[k][i];
    }
    if (lane < 4) {
#pragma unroll
        for (int i = 0; i < 9; ++i) Nsm[lane][i] = e[i];
    }
    return ok;
}

// whole solver; every lane of the warp calls it.  Writes up to 10 unit-norm models (row-major) to
// `models` in ascending-z order and returns their number (warp-uniform).
__device__ int five_point_warp(const double* s1, const double* s2, EmwShared& S, int lane, double* models)
{
    if (!emw_null_space(s1, s2, lane, S.N)) return 0;
    __syncwarp();
    // ---- 2. this lane's column of the constraint matrix ----
    double col[10];
#pragma unroll
    for (int r = 0; r < 10; ++r) col[r] = 0;
    {
        const int m = lane < 20 ? lane : 19;
        const int t[3] = {EMW_TRI[m][0], EMW_TRI[m][1], EMW_TRI[m][2]};
        const int P[6][3] = {{0, 1, 2}, {0, 2, 1}, {1, 0, 2}, {1, 2, 0}, {2, 0, 1}, {2, 1, 0}};
        int pa[6], pb[6], pc[6];
        bool inc[6];
#pragma unroll
        for (int p = 0; p < 6; ++p) {
            pa[p] = t[P[p][0]]; pb[p] = t[P[p][1]]; pc[p] = t[P[p][2]];
            inc[p] = true;
#pragma unroll
            for (int q = 0; q < p; ++q) if (pa[q] == pa[p] && pb[q] == pb[p] && pc[q] == pc[p]) inc[p] = false;
        }
#pragma unroll 1
        for (int p = 0; p < 6; ++p) {
            int ia = pa[0], ib = pb[0], ic = pc[0];
            bool on = inc[0];
#pragma unroll
            for (int q = 1; q < 6; ++q) if (p == q) { ia = pa[q]; ib = pb[q]; ic = pc[q]; on = inc[q]; }
            const double* A = S.N[ia];
            const double* B = S.N[ib];
            const double* C = S.N[ic];
            double a[9], b[9], c[9], M[9];
#pragma unroll
            for (int i = 0; i < 9; ++i) { a[i] = A[i]; b[i] = B[i]; c[i] = C[i]; }
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int q = 0; q < 3; ++q) M[3 * r + q] = a[3 * r] * b[3 * q] + a[3 * r + 1] * b[3 * q + 1] + a[3 * r + 2] * b[3 * q + 2];
            const double tr = M[0] + M[4] + M[8];
            const double w = on ? 1.0 : 0.0;
            // det: row 0 of A . (row 1 of B x row 2 of C)
            const double cx = b[4] * c[8] - b[5] * c[7], cy = b[5] * c[6] - b[3] * c[8], cz = b[3] * c[7] - b[4] * c[6];
            col[0] += w * (a[0] * cx + a[1] * cy + a[2] * cz);
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    const double mc = M[3 * r] * c[q] + M[3 * r + 1] * c[3 + q] + M[3 * r + 2] * c[6 + q];
                    col[1 + 3 * r + q] += w * (2.0 * mc - tr * c[3 * r + q]);
                }
        }
    }
    // ---- 3. Gauss-Jordan, lane = column ----
    bool ok = true;
#pragma unroll
    for (int c = 0; c < 10; ++c) {
        double f[10];
#pragma unroll
        for (int r = 0; r < 10; ++r) f[r] = shfl_d(col[r], c);
        int piv = c;
        double best = fabs(f[c]);
#pragma unroll
        for (int r = c + 1; r < 10; ++r) if (fabs(f[r]) > best) { best = fabs(f[r]); piv = r; }
        if (best < 1e-300) ok = false;
#pragma unroll
        for (int r = c + 1; r < 10; ++r)
            if (piv == r) {
                const double t0 = col[c]; col[c] = col[r]; col[r] = t0;
                const double t1 = f[c]; f[c] = f[r]; f[r] = t1;
            }
        const double inv = 1.0 / f[c];
        col[c] *= inv;
#pragma unroll
        for (int r = 0; r < 10; ++r)
            if (r != c) col[r] -= f[r] * col[c];
    }
    if (!ok) return 0;
    // ---- 4. B(z), det B(z) ----
    __syncwarp();
    if (lane >= 10 && lane < 20) {
#pragma unroll
        for (int r = 0; r < 6; ++r) S.T[r][lane - 10] = col[4 + r];
    }
    __syncwarp();
    double Bx[3][4], By[3][4], Bc[3][5];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const double* r1 = S.T[2 * i];
        const double* r2 = S.T[2 * i + 1];
        Bx[i][3] = -r2[0]; Bx[i][2] = r1[0] - r2[1]; Bx[i][1] = r1[1] - r2[2]; Bx[i][0] = r1[2];
        By[i][3] = -r2[3]; By[i][2] = r1[3] - r2[4]; By[i][1] = r1[4] - r2[5]; By[i][0] = r1[5];
        Bc[i][4] = -r2[6]; Bc[i][3] = r1[6] - r2[7]; Bc[i][2] = r1[7] - r2[8]; Bc[i][1] = r1[8] - r2[9]; Bc[i][0] = r1[9];
    }
    double det[11];
    {
        double m1[8], m2[8], m3[11], m4[7], m5[7];
#pragma unroll
        for (int k = 0; k < 11; ++k) det[k] = 0;
        poly1_mul<3, 4>(By[1], Bc[2], m1); poly1_mul<4, 3>(Bc[1], By[2], m2);
#pragma unroll
        for (int k = 0; k < 8; ++k) m1[k] -= m2[k];
        poly1_mul<3, 7>(Bx[0], m1, m3);
#pragma unroll
        for (int k = 0; k < 11; ++k) det[k] += m3[k];
        poly1_mul<3, 4>(Bx[1], Bc[2], m1); poly1_mul<4, 3>(Bc[1], Bx[2], m2);
#pragma unroll
        for (int k = 0; k < 8; ++k) m1[k] -= m2[k];
        poly1_mul<3, 7>(By[0], m1, m3);
#pragma unroll
        for (int k = 0; k < 11; ++k) det[k] -= m3[k];
        poly1_mul<3, 3>(Bx[1], By[2], m4); poly1_mul<3, 3>(By[1], Bx[2], m5);
#pragma unroll
        for (int k = 0; k < 7; ++k) m4[k] -= m5[k];
        poly1_mul<4, 6>(Bc[0], m4, m3);
#pragma unroll
        for (int k = 0; k < 11; ++k) det[k] += m3[k];
    }
    // ---- 5. all complex roots: Aberth-Ehrlich, lane k = root k ----
    int n = 10;
#pragma unroll
    for (int i = 10; i >= 1; --i) if (n == i && det[i] == 0) n = i - 1;
    if (n <= 0) return 0;
    double lead = det[10];
#pragma unroll
    for (int i = 9; i >= 1; --i) if (n == i) lead = det[i];
    double am[10];   // monic coefficients a_0 .. a_{n-1}
#pragma unroll
    for (int i = 0; i < 10; ++i) am[i] = det[i] / lead;
    double mine = 0;
#pragma unroll
    for (int i = 0; i < 10; ++i) if (lane == i) mine = am[i];
    double rad = (lane < n && mine != 0) ? pow(fabs(mine), 1.0 / (n - lane)) : 0.0;
    {
        const bool bad = __any_sync(0xffffffffu, !isfinite(rad));
        if (bad) return 0;
    }
    rad = warp_max_d(rad);
    rad = rad > 0 ? 0.7 * rad : 1.0;
    double zr, zi;
    {
        const int k = lane < n ? lane : 0;
        const double ang = 6.283185307179586476925286766559 * k / n + 0.4, r = rad * (1 + 0.1 * k / n);
        zr = r * cos(ang); zi = r * sin(ang);
    }
    const bool mineroot = lane < n;
    // (fused multiply-adds and Newton reciprocals in this loop: the iterates are self-correcting, and
    // the real roots are polished against the exact coefficients afterwards)
    for (int it = 0; it < 200; ++it) {
        double pr = 1, pi = 0, dr = 0, di = 0, sb = 1;
        const double az = sqrt(fma(zr, zr, zi * zi));
#pragma unroll
        for (int i = 9; i >= 0; --i) {
            if (i < n) {
                const double ndr = fma(dr, zr, fma(-di, zi, pr)), ndi = fma(dr, zi, fma(di, zr, pi));
                const double npr = fma(pr, zr, fma(-pi, zi, am[i])), npi = fma(pr, zi, pi * zr);
                dr = ndr; di = ndi; pr = npr; pi = npi;
                sb = fma(sb, az, fabs(am[i]));          // sum |a_i| |z|^i: scale of the rounding error of p(z)
            }
        }
        double sr = 0, si = 0;
#pragma unroll
        for (int j = 0; j < 10; ++j) {
            const double ojr = shfl_d(zr, j), oji = shfl_d(zi, j);
            if (j < n && j != lane) {
                const double er = zr - ojr, ei = zi - oji, d2 = fma(er, er, ei * ei);
                if (d2 != 0) { const double id2 = fast_rcp(d2); sr = fma(er, id2, sr); si = fma(-ei, id2, si); }
            }
        }
        double rel = 0;
        const double den = fma(dr, dr, di * di);
        if (mineroot && den != 0) {
            const double iden = fast_rcp(den);
            const double wr = fma(pr, dr, pi * di) * iden, wi = fma(pi, dr, -pr * di) * iden;
            const double qr = 1 - fma(wr, sr, -wi * si), qi = -fma(wr, si, wi * sr);
            const double qd = fma(qr, qr, qi * qi);
            if (qd != 0) {
                const double iqd = fast_rcp(qd);
                const double stepr = fma(wr, qr, wi * qi) * iqd, stepi = fma(wi, qr, -wr * qi) * iqd;
                zr -= stepr; zi -= stepi;
                rel = (fabs(stepr) + fabs(stepi)) / (fabs(zr) + fabs(zi) + 1e-300);
            }
        }
        // A root is settled when its step is below 1e-12 (relative); when |p(z)| has reached the
        // rounding noise of its own evaluation (an ill-conditioned root cannot get closer); or --
        // only real roots become models -- when it is unmistakably complex and within 1e-6 of its
        // limit (close complex clusters converge linearly and would keep the whole warp iterating).
        const double mag = fabs(zr) + fabs(zi);
        const bool noise = fabs(pr) + fabs(pi) <= 2e-14 * sb;
        const bool settled = !mineroot || rel < 1e-12 || noise ||
                             (it >= 8 && rel < 1e-6 && fabs(zi) > 1e-4 * mag && fabs(zi) > 1e-7);
        if (__all_sync(0xffffffffu, settled)) break;   // real roots are Newton-polished below
    }
    // ---- 6. real roots -> models ----
    bool cand = mineroot && fabs(zi) <= 1e-10;
    double z = zr;
    if (cand) {
#pragma unroll 1
        for (int itn = 0; itn < 2; ++itn) {
            double p = det[10], dp = 0;
#pragma unroll
            for (int i = 9; i >= 0; --i) { dp = dp * z + p; p = p * z + det[i]; }
            if (dp != 0 && isfinite(p / dp)) z -= p / dp;
        }
    }
    double Ev[9];
    bool valid = false;
    if (cand) {
        double Bz[3][3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            Bz[i][0] = ((Bx[i][3] * z + Bx[i][2]) * z + Bx[i][1]) * z + Bx[i][0];
            Bz[i][1] = ((By[i][3] * z + By[i][2]) * z + By[i][1]) * z + By[i][0];
            Bz[i][2] = (((Bc[i][4] * z + Bc[i][3]) * z + Bc[i][2]) * z + Bc[i][1]) * z + Bc[i][0];
        }
        double best[3] = {0, 0, 0}, bn = -1;
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = a + 1; b < 3; ++b) {
                const double c0 = Bz[a][1] * Bz[b][2] - Bz[a][2] * Bz[b][1], c1 = Bz[a][2] * Bz[b][0] - Bz[a][0] * Bz[b][2],
                             c2 = Bz[a][0] * Bz[b][1] - Bz[a][1] * Bz[b][0];
                const double n2 = c0 * c0 + c1 * c1 + c2 * c2;
                if (n2 > bn) { bn = n2; best[0] = c0; best[1] = c1; best[2] = c2; }
            }
        if (bn > 0 && !(fabs(best[2] / sqrt(bn)) < 1e-10)) {
            const double x = best[0] / best[2], y = best[1] / best[2];
            double nrm = 0;
#pragma unroll
            for (int i = 0; i < 9; ++i) { Ev[i] = x * S.N[0][i] + y * S.N[1][i] + z * S.N[2][i] + S.N[3][i]; nrm += Ev[i] * Ev[i]; }
            nrm = sqrt(nrm);
            if (nrm > 0 && isfinite(nrm)) {
                valid = true;
#pragma unroll
                for (int i = 0; i < 9; ++i) Ev[i] /= nrm;
            }
        }
    }
    // ascending z among the valid candidates (ties: lower root index first)
    const unsigned vmask = __ballot_sync(0xffffffffu, valid);
    int slot = 0;
#pragma unroll
    for (int j = 0; j < 10; ++j) {
        const double zj = shfl_d(z, j);
        if (((vmask >> j) & 1u) && (zj < z || (zj == z && j < lane))) ++slot;
    }
    if (valid) {
#pragma unroll
        for (int i = 0; i < 9; ++i) models[slot * 9 + i] = Ev[i];
    }
    return __popc(vmask);
}

struct EmatArgs {
    int n, iters;                          // n < 0: each sequence's count is n_dev[s] (emat_seq reads it)
    int cap;                               // point slots per sequence
    const float* p1; const float* p2;     // [n][2] pixels
    const VoIntrinsics* intr;              // [nseq] camera and Sampson threshold of each set
    double conf;
    double* x1; double* x2;               // [n][2] normalised
    int* n_dev;                            // [1] = n
    int* samples;                          // [iters][5]
    double* models;                        // [iters][10][9]
    int* nmodels;                          // [iters]
    int* counts;                           // [iters][10]
    int* flags;
    // outputs
    double* E; uint8_t* mask; int* result; // result[0] = found, [1] = iterations run, [2] = winner flat index
    int* state;                            // [0] current iteration bound (niters), [1] max_good, [2] winner, [3] iterations replayed
    int chunk_start, chunk_len;
    int full;                              // 1: score every sample (the caller reads counts[]); the replay still honours the bound
};

// the view of sequence s: its slices of every per-sequence array ([cap] points, [iters] samples, 9 doubles of E, 4 ints of
// result / state, one n and one flag word)
__device__ __forceinline__ EmatArgs emat_seq(const EmatArgs& A, int s)
{
    EmatArgs a = A;
    const size_t pc = (size_t)s * A.cap, ic = (size_t)s * A.iters;
    a.p1 += 2 * pc; a.p2 += 2 * pc; a.x1 += 2 * pc; a.x2 += 2 * pc; a.mask += pc;
    a.samples += 5 * ic; a.models += ic * EM_MAXM * 9; a.nmodels += ic; a.counts += ic * EM_MAXM;
    a.E += 9 * s; a.result += 4 * s; a.state += 4 * s; a.n_dev += s; a.flags += s; a.intr += s;
    if (A.n < 0) a.n = *a.n_dev;
    return a;
}

__global__ void __launch_bounds__(256)
emat_normalize_kernel(EmatArgs A)
{
    const EmatArgs a = emat_seq(A, blockIdx.y);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {   // state: bound, max_good, winner, replayed
        a.state[0] = a.iters; a.state[1] = 0; a.state[2] = -1; a.state[3] = 0;
        *a.flags = 0;
    }
    if (i >= a.n) return;
    const VoIntrinsics& c = *a.intr;
    a.x1[2 * i] = ((double)a.p1[2 * i] - c.cx) / c.fx; a.x1[2 * i + 1] = ((double)a.p1[2 * i + 1] - c.cy) / c.fy;
    a.x2[2 * i] = ((double)a.p2[2 * i] - c.cx) / c.fx; a.x2[2 * i + 1] = ((double)a.p2[2 * i + 1] - c.cy) / c.fy;
}

__global__ void __launch_bounds__(EMW_WARPS * 32)
emat_solve_kernel(EmatArgs A)
{
    __shared__ EmwShared sh[EMW_WARPS];
    const EmatArgs a = emat_seq(A, blockIdx.y);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int it = blockIdx.x * EMW_WARPS + warp;
    if (it >= a.iters) return;
    if (lane < EM_MAXM) a.counts[it * EM_MAXM + lane] = 0;
    const int* smp = a.samples + 5 * it;
    if (smp[0] < 0) { if (lane == 0) a.nmodels[it] = 0; return; }
    double s1[10], s2[10];
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        const int s = smp[k];
        s1[2 * k] = a.x1[2 * s]; s1[2 * k + 1] = a.x1[2 * s + 1];
        s2[2 * k] = a.x2[2 * s]; s2[2 * k + 1] = a.x2[2 * s + 1];
    }
    const int nm = five_point_warp(s1, s2, sh[warp], lane, a.models + (size_t)it * EM_MAXM * 9);
    if (lane == 0) a.nmodels[it] = nm;
}

__device__ __forceinline__ bool sampson_inlier(const double* E, double ax, double ay, double bx, double by, float thr_sq)
{
    const double Ex0 = E[0] * ax + E[1] * ay + E[2] * 1., Ex1 = E[3] * ax + E[4] * ay + E[5] * 1., Ex2 = E[6] * ax + E[7] * ay + E[8] * 1.;
    const double Et0 = E[0] * bx + E[3] * by + E[6] * 1., Et1 = E[1] * bx + E[4] * by + E[7] * 1.;
    const double s = bx * Ex0 + by * Ex1 + 1. * Ex2;
    const double aa = Ex0 * Ex0, bb = Ex1 * Ex1, cc = Et0 * Et0, dd = Et1 * Et1;
    const float e = (float)(s * s / (aa + bb + cc + dd));
    return e <= thr_sq;
}

#define EM_ST 8   // samples per scoring block
__global__ void __launch_bounds__(256)
emat_score_kernel(EmatArgs A)
{
    __shared__ double s_E[EM_ST * EM_MAXM * 9];
    __shared__ int s_nm[EM_ST];
    const EmatArgs a = emat_seq(A, blockIdx.z);
    if (!a.full && a.chunk_start >= a.state[0]) return;
    const int it0 = a.chunk_start + blockIdx.y * EM_ST;
    const int ns = min(EM_ST, min(a.iters, a.chunk_start + a.chunk_len) - it0);
    if (ns <= 0) return;
    for (int k = threadIdx.x; k < ns * EM_MAXM * 9; k += blockDim.x) s_E[k] = a.models[(size_t)it0 * EM_MAXM * 9 + k];
    if (threadIdx.x < ns) s_nm[threadIdx.x] = a.nmodels[it0 + threadIdx.x];
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < a.n;
    double ax = 0, ay = 0, bx = 0, by = 0;
    if (live) { ax = a.x1[2 * i]; ay = a.x1[2 * i + 1]; bx = a.x2[2 * i]; by = a.x2[2 * i + 1]; }
    const int lane = threadIdx.x & 31;
    const float thr_sq = a.intr->emat_thr_sq;
    for (int s = 0; s < ns; ++s)
        for (int m = 0; m < s_nm[s]; ++m) {
            const bool in = live && sampson_inlier(s_E + (s * EM_MAXM + m) * 9, ax, ay, bx, by, thr_sq);
            const unsigned bm = __ballot_sync(0xffffffffu, in);
            if (lane == 0 && bm) atomicAdd(a.counts + (it0 + s) * EM_MAXM + m, __popc(bm));
        }
}

// replay of cv2's sequential loop over this chunk's (sample, model) counts; shrinks the bound
__global__ void emat_update_kernel(EmatArgs A)
{
    if (threadIdx.x != 0) return;
    const EmatArgs a = emat_seq(A, blockIdx.x);
    int niters = a.state[0], max_good = a.state[1], win = a.state[2];
    if (a.chunk_start >= niters) return;
    const int N = a.n;
    int it = a.chunk_start;
    if (N == 5) {
        if (it == 0) { win = a.nmodels[0] > 0 ? 0 : -1; a.state[2] = win; a.state[3] = 1; a.state[0] = 1; }
        return;
    }
    const int end = min(a.chunk_start + a.chunk_len, a.iters);
    for (; it < end && it < niters; ++it) {
        const int nm = a.nmodels[it];
        for (int m = 0; m < nm; ++m) {
            const int good = a.counts[it * EM_MAXM + m];
            if (good > (max_good > 4 ? max_good : 4)) {
                win = it * EM_MAXM + m; max_good = good;
                niters = ransac_update_num_iters(a.conf, (double)(N - good) / N, 5, niters);
            }
        }
    }
    a.state[0] = niters; a.state[1] = max_good; a.state[2] = win; a.state[3] = it;
}

__global__ void __launch_bounds__(256)
emat_finish_kernel(EmatArgs A)
{
    __shared__ double s_E[9];
    const EmatArgs a = emat_seq(A, blockIdx.x);
    const int win = a.state[2];
    if (threadIdx.x == 0) { a.result[0] = win >= 0; a.result[1] = a.state[3]; a.result[2] = win; }
    if (win < 0) {
        for (int i = threadIdx.x; i < a.n; i += blockDim.x) a.mask[i] = 0;
        return;
    }
    if (threadIdx.x < 9) { s_E[threadIdx.x] = a.models[(size_t)win * 9 + threadIdx.x]; a.E[threadIdx.x] = s_E[threadIdx.x]; }
    __syncthreads();
    const float thr_sq = a.intr->emat_thr_sq;
    for (int i = threadIdx.x; i < a.n; i += blockDim.x)
        a.mask[i] = (a.n == 5) ? 1 : (sampson_inlier(s_E, a.x1[2 * i], a.x1[2 * i + 1], a.x2[2 * i], a.x2[2 * i + 1], thr_sq) ? 1 : 0);
}

int vo_rng_table(b200vo_ctx* ctx, int n, const uint32_t** d_table);

// dev_io != nullptr: p1 / p2 are DEVICE pointers and the results go to dev_io (device) instead of E / mask / found
struct EmatDevIO { double* E; uint8_t* mask; int32_t* found; };

__global__ void emat_export_kernel(EmatArgs A, EmatDevIO io)
{
    const EmatArgs a = emat_seq(A, 0);
    const int ok = a.result[0];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += gridDim.x * blockDim.x) io.mask[i] = ok ? a.mask[i] : 0;
    if (blockIdx.x == 0 && threadIdx.x < 9) io.E[threadIdx.x] = ok ? a.E[threadIdx.x] : 0.0;
    if (blockIdx.x == 0 && threadIdx.x == 0) *io.found = ok;
}

// Enqueues the RANSAC of `nseq` point sets on the ctx stream; the device arrays of `a` are set, a.n_dev holds each set's
// point count (at most max_n <= a.cap).  draw: the samples come from cv2's RNG stream (else a.samples is the caller's).
static int emat_launch(b200vo_ctx* ctx, EmatArgs& a, int nseq, int max_n, bool draw)
{
    const int iters = a.iters;
    const int n_raw = 10 * iters + 256;
    const int pb = (max_n + 255) / 256 > 0 ? (max_n + 255) / 256 : 1;
    emat_normalize_kernel<<<dim3(pb, nseq), 256, 0, ctx->stream>>>(a);
    ctx->launches++;
    if (draw) {
        const uint32_t* rng = nullptr;
        VO_TRY(vo_rng_table(ctx, n_raw, &rng));
        const size_t smem = (size_t)n_raw * sizeof(int);
        if (smem > 48 * 1024)
            VO_CUDA(ctx, cudaFuncSetAttribute(ransac_samples_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ransac_samples_kernel<5><<<nseq, 128, smem, ctx->stream>>>(rng, n_raw, a.n_dev, iters, a.samples, a.flags);
        ctx->launches++;
    }
    // every sample is solved up front: one warp each, so the launch is one wave of latency-bound warps
    // whether it carries 128 samples or all of them
    emat_solve_kernel<<<dim3((iters + EMW_WARPS - 1) / EMW_WARPS, nseq), EMW_WARPS * 32, 0, ctx->stream>>>(a);
    ctx->launches += 1;
    // scoring chunks of 64, 128, 256, ... samples: cv2 usually stops within the first (10-60 samples), and every
    // chunk beyond the bound (known on the device after the previous chunk) costs two empty launches
    for (int c0 = 0, len = 64; c0 < iters; c0 += len, len *= 2) {
        a.chunk_start = c0; a.chunk_len = len;
        emat_score_kernel<<<dim3(pb, (len + EM_ST - 1) / EM_ST, nseq), 256, 0, ctx->stream>>>(a);
        emat_update_kernel<<<nseq, 32, 0, ctx->stream>>>(a);
        ctx->launches += 2;
    }
    emat_finish_kernel<<<nseq, 256, 0, ctx->stream>>>(a);
    ctx->launches += 1;
    VO_CUDA(ctx, cudaGetLastError());
    return 0;
}

int vo_emat_batch(b200vo_ctx* ctx, const float* p1, const float* p2, int cap, const int* n_dev, int max_n, int nseq,
                  const VoIntrinsics* intr_dev, double prob, int max_iters, double* E_dev, uint8_t* mask_dev, int* result_dev,
                  int* flags_dev)
{
    const int iters = max_iters > 1 ? max_iters : 1;
    EmatArgs a{};
    a.n = -1; a.iters = iters; a.cap = cap;
    a.intr = intr_dev;
    a.conf = prob;
    const size_t ns = nseq;
    const size_t b_x = vo_align(ns * cap * 16, 256), b_s = vo_align(ns * iters * 5 * 4, 256), b_m = vo_align(ns * iters * EM_MAXM * 9 * 8, 256);
    const size_t b_nm = vo_align(ns * iters * 4, 256), b_c = vo_align(ns * iters * EM_MAXM * 4, 256), b_st = vo_align(ns * 16, 256);
    VO_TRY(vo_reserve(ctx, ctx->d_scratch[5], 2 * b_x + b_s + b_m + b_nm + b_c + b_st));
    uint8_t* d = (uint8_t*)ctx->d_scratch[5].p;
    a.p1 = p1; a.p2 = p2; a.n_dev = const_cast<int*>(n_dev);
    a.x1 = (double*)d; a.x2 = (double*)(d + b_x); d += 2 * b_x;
    a.samples = (int*)d; d += b_s;
    a.models = (double*)d; d += b_m;
    a.nmodels = (int*)d; d += b_nm;
    a.counts = (int*)d; d += b_c;
    a.state = (int*)d; a.flags = flags_dev;
    a.E = E_dev; a.mask = mask_dev; a.result = result_dev;
    return emat_launch(ctx, a, nseq, max_n, true);
}

static int emat_run(b200vo_ctx* ctx, const float* p1, const float* p2, int n, const double K[9], const int32_t* samples,
                    double prob, double thr, int max_iters, double E[9], uint8_t* mask, int* found, int32_t* nmodels_out,
                    int32_t* counts_out, double* models_out, int* winner_out, int* iters_run, const EmatDevIO* dev_io = nullptr)
{
    if (!ctx || !p1 || !p2 || !K) return B200VO_E_BADARG;
    if (!dev_io && (!E || !mask || !found)) return B200VO_E_BADARG;
    if (found) *found = 0;
    if (n < 0) return vo_set_err(ctx, B200VO_E_BADARG, "npoints >= 0 && points2.checkVector(2) == npoints");
    if (n < 5) {   // cv2 returns an empty matrix
        if (dev_io) { VO_CUDA(ctx, cudaSetDevice(ctx->device)); VO_CUDA(ctx, cudaMemsetAsync(dev_io->found, 0, 4, ctx->stream)); }
        return 0;
    }
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    const int iters = max_iters > 1 ? max_iters : 1;
    EmatArgs a{};
    a.n = n; a.iters = iters; a.cap = n;
    VO_TRY(vo_intrinsics_uniform(ctx, K, thr, 1, &a.intr));   // the batch of one
    a.conf = prob;
    a.full = samples != nullptr;
    const size_t b_p = vo_align((size_t)n * 8, 256), b_x = vo_align((size_t)n * 16, 256);
    const size_t b_s = vo_align((size_t)iters * 5 * 4, 256), b_m = vo_align((size_t)iters * EM_MAXM * 9 * 8, 256);
    const size_t b_nm = vo_align((size_t)iters * 4, 256), b_c = vo_align((size_t)iters * EM_MAXM * 4, 256);
    const size_t b_mask = vo_align((size_t)n, 256);
    VO_TRY(vo_reserve(ctx, ctx->d_scratch[5], 2 * b_p + 2 * b_x + b_s + b_m + b_nm + b_c + b_mask + 1024));
    uint8_t* d = (uint8_t*)ctx->d_scratch[5].p;
    a.p1 = (const float*)d; a.p2 = (const float*)(d + b_p); d += 2 * b_p;
    a.x1 = (double*)d; a.x2 = (double*)(d + b_x); d += 2 * b_x;
    a.samples = (int*)d; d += b_s;
    a.models = (double*)d; d += b_m;
    a.nmodels = (int*)d; d += b_nm;
    a.counts = (int*)d; d += b_c;
    a.mask = d; d += b_mask;
    uint8_t* d_small = d;                       // E[9] | result[3] | n | flags
    a.E = (double*)d_small; a.result = (int*)(d_small + 128); a.n_dev = (int*)(d_small + 192); a.flags = (int*)(d_small + 256);
    a.state = (int*)(d_small + 320);
    const size_t b_dbg = samples ? b_s + b_nm + b_c + (models_out ? b_m : 0) : 0;
    VO_TRY(vo_reserve_pinned(ctx, 2 * b_p + b_mask + 1024 + b_dbg));
    uint8_t* hp = (uint8_t*)ctx->h_pin;
    if (dev_io) {
        a.p1 = p1; a.p2 = p2;     // already resident
    } else {
        memcpy(hp, p1, (size_t)n * 8);
        memcpy(hp + b_p, p2, (size_t)n * 8);
        VO_CUDA(ctx, cudaMemcpyAsync((void*)a.p1, hp, 2 * b_p, cudaMemcpyHostToDevice, ctx->stream));
    }
    VO_CUDA(ctx, cudaMemsetAsync(d_small, 0, 512, ctx->stream));
    int* h_small = (int*)(hp + 2 * b_p + b_mask);
    h_small[0] = n;
    VO_CUDA(ctx, cudaMemcpyAsync(a.n_dev, h_small, 4, cudaMemcpyHostToDevice, ctx->stream));
    uint8_t* h_dbg = hp + 2 * b_p + b_mask + 1024;
    if (samples) {   // the caller's sample set (parity runs: same hypotheses as the oracle / as cv2's RNG replay)
        memcpy(h_dbg, samples, (size_t)iters * 5 * 4);
        VO_CUDA(ctx, cudaMemcpyAsync(a.samples, h_dbg, (size_t)iters * 5 * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    VO_TRY(emat_launch(ctx, a, 1, n, samples == nullptr));
    VO_CUDA(ctx, cudaGetLastError());
    if (dev_io) {   // results stay on the device; nothing to wait for
        emat_export_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(a, *dev_io);
        ctx->launches += 1;
        VO_CUDA(ctx, cudaGetLastError());
        return 0;
    }
    VO_CUDA(ctx, cudaMemcpyAsync(hp, a.mask, b_mask, cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaMemcpyAsync(hp + b_mask, d_small, 512, cudaMemcpyDeviceToHost, ctx->stream));
    if (samples) {
        if (nmodels_out) VO_CUDA(ctx, cudaMemcpyAsync(h_dbg + b_s, a.nmodels, (size_t)iters * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (counts_out) VO_CUDA(ctx, cudaMemcpyAsync(h_dbg + b_s + b_nm, a.counts, (size_t)iters * EM_MAXM * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (models_out) VO_CUDA(ctx, cudaMemcpyAsync(h_dbg + b_s + b_nm + b_c, a.models, (size_t)iters * EM_MAXM * 72, cudaMemcpyDeviceToHost, ctx->stream));
    }
    VO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1);
    const int* res = (const int*)(hp + b_mask + 128);
    const int flg = *(const int*)(hp + b_mask + 256);
    if (flg & 1) return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "RNG table exhausted while drawing subsets (n=%d)", n);
    *found = res[0];
    if (res[0]) {
        memcpy(E, hp + b_mask, 72);
        memcpy(mask, hp, (size_t)n);
    }
    if (winner_out) *winner_out = res[2];
    if (iters_run) *iters_run = res[1];
    if (samples) {
        if (nmodels_out) memcpy(nmodels_out, h_dbg + b_s, (size_t)iters * 4);
        if (counts_out) memcpy(counts_out, h_dbg + b_s + b_nm, (size_t)iters * EM_MAXM * 4);
        if (models_out) memcpy(models_out, h_dbg + b_s + b_nm + b_c, (size_t)iters * EM_MAXM * 72);
    }
    return 0;
}

extern "C" int b200vo_find_essential_mat_ransac(b200vo_ctx* ctx, const float* p1, const float* p2, int n, const double K[9],
                                                double prob, double thr, int max_iters, double E[9], uint8_t* mask, int* found)
{
    return emat_run(ctx, p1, p2, n, K, nullptr, prob, thr, max_iters, E, mask, found, nullptr, nullptr, nullptr, nullptr, nullptr);
}

// Same RANSAC on the CALLER's 5-subsets (north_star: "inlier masks bit-exact given the same hypothesis sample set"):
// every sample is solved and scored (no early exit), the replay of cv2's loop picks the winner; per-sample model
// counts, per-(sample, model) inlier counts and the models themselves come back for comparison with the oracle.
extern "C" int b200vo_find_essential_mat_ransac_samples(b200vo_ctx* ctx, const float* p1, const float* p2, int n, const double K[9],
                                                        const int32_t* samples, int iters, double prob, double thr, double E[9],
                                                        uint8_t* mask, int* found, int32_t* nmodels_out, int32_t* counts_out,
                                                        double* models_out, int* winner_out, int* iters_run)
{
    if (!samples || iters < 1) return B200VO_E_BADARG;
    return emat_run(ctx, p1, p2, n, K, samples, prob, thr, iters, E, mask, found, nmodels_out, counts_out, models_out, winner_out,
                    iters_run);
}

// Device-pointer form (SURVEY 8b `_dev`): p1_dev / p2_dev float32 (n,2) in device memory; E_dev double[9], mask_dev uint8 (n),
// found_dev int32[1] are written on the device (zeros when nothing was found).  Asynchronous on the ctx stream.
extern "C" int b200vo_find_essential_mat_ransac_dev(b200vo_ctx* ctx, const float* p1_dev, const float* p2_dev, int n, const double K[9],
                                                    double prob, double thr, int max_iters, double* E_dev, uint8_t* mask_dev,
                                                    int32_t* found_dev)
{
    if (!E_dev || !mask_dev || !found_dev) return B200VO_E_BADARG;
    const EmatDevIO io{E_dev, mask_dev, found_dev};
    return emat_run(ctx, p1_dev, p2_dev, n, K, nullptr, prob, thr, max_iters, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                    nullptr, nullptr, &io);
}
