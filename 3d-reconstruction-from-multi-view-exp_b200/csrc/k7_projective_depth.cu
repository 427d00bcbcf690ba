// Projective-depth iteration, primary method -- the step BEFORE bundle adjustment in the reference's
// perspective pipeline (SURVEY.md section 8f row 3).
//
// Replaces reference lib/perspective_camera_calibration.py:61-144
// (_compute_projective_depth_primary_method) together with _compute_reprojection_error (:44-58).
// Per iteration the reference forms W = x * z with unit-length point vectors (:86-90), takes the
// four leading left singular vectors U_ of the (3M x N) matrix (:92-96), solves for every point an
// M x M symmetric eigenproblem (:98-125) whose leading eigenvector gives the new depths (:127-131),
// and evaluates the reprojection error of the rank-4 approximation (:133-136).
//
// Here, with the two identities stated in oracle/depth_oracle.py (the point matrices are B B^T with
// B of size M x 4; everything depends on U_ only through the projector U_ U_^T):
//   depth_scale_kernel   warp per point: w = x z / |x z|  ->  Wn [N_pad][ld]  (k-major: row = point)
//   Gram matrix          G = Wn^T Wn (3M x 3M) on the FP64 tensor cores -- the Schur-product SYRK
//                        kernel of K3 (k3_schur_syrk.cu), work items planned on the host
//   subspace_eig_kernel  one CTA: orthogonal iteration Q <- orth(G Q), warm-started from the previous
//                        pass; U4 = an orthonormal basis of the dominant four-dimensional eigenspace
//   jacobi_eig_kernel    fallback when that does not converge (near-degenerate 4th / 5th eigenvalue):
//                        parallel cyclic Jacobi (round-robin pairs) on G, eigenvectors of the four
//                        largest eigenvalues
//   depth_update_kernel  warp per point: B (M x 4), 4 x 4 Gram, its leading eigenvector by Jacobi in
//                        registers, xi = B v / |B v| with the sign rule of :127-128, z = xi / |x|; and
//                        the point's share of the reprojection error (U4 U4^T w against x)
//   depth_error_kernel   fixed-order sum of the partials -> E = f0 sqrt(mean)
// The host reads one double (E) per iteration to apply the stopping rule of :138-142.
#include <cmath>
#include <cstdlib>
#include <vector>

#include "ba_common.cuh"

namespace ba {

// ---- Wn ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
depth_scale_kernel(int64_t N, int M, int ld, const double* __restrict__ x, const double* __restrict__ z,
                   double* __restrict__ Wn) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t j = warp; j < N; j += nwarps) {
    const double* xj = x + (size_t)j * M * 3;
    const double* zj = z + (size_t)j * M;
    double s = 0.0;
    for (int a = lane; a < 3 * M; a += 32) {
      const double w = xj[a] * zj[a / 3];
      s += w * w;
    }
    s = warp_sum(s);
    const double inv = 1.0 / sqrt(s);  // :90  W / ||W_j||
    double* out = Wn + (size_t)j * ld;
    for (int a = lane; a < ld; a += 32) out[a] = a < 3 * M ? (xj[a] * zj[a / 3]) * inv : 0.0;
  }
}

// G (n x n, full symmetric, ld = n) from the lower triangle the SYRK reduce wrote into P (ld = n_pad)
__global__ void gram_symmetrize_kernel(int n, int n_pad, const double* __restrict__ P, double* __restrict__ G) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n * n) return;
  const int r = k / n, c = k - r * n;
  G[k] = r >= c ? P[(size_t)r * n_pad + c] : P[(size_t)c * n_pad + r];
}

// ---- leading four-dimensional eigenspace of the Gram matrix: subspace iteration -----------------
// Everything downstream depends on U4 only through the projector U4 U4^T, so any orthonormal basis
// of the dominant invariant subspace will do.  One CTA iterates Q <- orth(G Q) (Cholesky-QR twice
// per step) from the previous pass's basis (the depths change little between passes), until the
// basis moves by less than 1e-13 in the Frobenius norm, plus two more steps; G is read through L1.
// status[0] = 1 when it converged; otherwise the Jacobi kernel below takes over (near-degenerate
// fourth and fifth eigenvalues).  Fixed order of operations: bit-reproducible.
__global__ void __launch_bounds__(256)
subspace_eig_kernel(int n, const double* __restrict__ G, double* __restrict__ U4, int warm, int max_steps,
                    int* __restrict__ status) {
  extern __shared__ double ssm[];
  double* Q = ssm;           // [n][4]
  double* Y = ssm + 4 * n;   // [n][4]
  __shared__ double S[16], Rinv[16], Mq[16];
  __shared__ double dist2[8];
  __shared__ int s_stop;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;

  // Y <- Y R^-1 with R^T R = Y^T Y  (one Cholesky-QR step; the caller runs it twice)
  auto cholqr = [&]() {
    for (int pr = warp; pr < 10; pr += nw) {  // the 10 entries k <= l of Y^T Y, one warp each
      int k = 0, l = pr;
      while (l >= 4 - k) { l -= 4 - k; ++k; }
      l += k;
      double acc = 0.0;
      for (int a = lane; a < n; a += 32) acc += Y[4 * a + k] * Y[4 * a + l];
      acc = warp_sum(acc);
      if (lane == 0) { S[4 * k + l] = acc; S[4 * l + k] = acc; }
    }
    __syncthreads();
    if (tid == 0) {
      double R[4][4] = {};
      for (int c = 0; c < 4; ++c) {       // upper-triangular R, column by column
        for (int r = 0; r <= c; ++r) {
          double v = S[4 * r + c];
          for (int m = 0; m < r; ++m) v -= R[m][r] * R[m][c];
          R[r][c] = r == c ? sqrt(v) : v / R[r][r];
        }
      }
      double I[4][4] = {};                // R^-1 (upper triangular) by back substitution
      for (int c = 0; c < 4; ++c) {
        I[c][c] = 1.0 / R[c][c];
        for (int r = c - 1; r >= 0; --r) {
          double v = 0.0;
          for (int m = r + 1; m <= c; ++m) v -= R[r][m] * I[m][c];
          I[r][c] = v / R[r][r];
        }
      }
      for (int r = 0; r < 4; ++r)
        for (int c = 0; c < 4; ++c) Rinv[4 * r + c] = I[r][c];
    }
    __syncthreads();
    for (int a = tid; a < n; a += nt) {
      const double y0 = Y[4 * a], y1 = Y[4 * a + 1], y2 = Y[4 * a + 2], y3 = Y[4 * a + 3];
      Y[4 * a] = y0 * Rinv[0];
      Y[4 * a + 1] = y0 * Rinv[1] + y1 * Rinv[5];
      Y[4 * a + 2] = y0 * Rinv[2] + y1 * Rinv[6] + y2 * Rinv[10];
      Y[4 * a + 3] = y0 * Rinv[3] + y1 * Rinv[7] + y2 * Rinv[11] + y3 * Rinv[15];
    }
    __syncthreads();
  };

  if (warm) {
    for (int k = tid; k < 4 * n; k += nt) Y[k] = U4[k];
  } else {
    // cold start: four columns of G spread over the index range
    for (int k = tid; k < 4 * n; k += nt) {
      const int a = k >> 2, c = ((k & 3) * n) / 4 + (k & 3);
      Y[k] = G[(size_t)a * n + (c < n ? c : n - 1)] + ((a == c) ? 1.0 : 0.0);
    }
  }
  __syncthreads();
  cholqr();
  cholqr();
  for (int k = tid; k < 4 * n; k += nt) Q[k] = Y[k];
  __syncthreads();
  int extra = -1;  // thread 0 only; >= 0: steps done after the basis stopped moving
  int step = 0;
  for (; step < max_steps; ++step) {
    for (int w = tid; w < 4 * n; w += nt) {  // Y = G Q
      const int a = w >> 2, k = w & 3;
      const double* g = G + (size_t)a * n;
      double acc0 = 0.0, acc1 = 0.0;
      int b = 0;
      for (; b + 1 < n; b += 2) {
        acc0 = fma(g[b], Q[4 * b + k], acc0);
        acc1 = fma(g[b + 1], Q[4 * (b + 1) + k], acc1);
      }
      if (b < n) acc0 = fma(g[b], Q[4 * b + k], acc0);
      Y[w] = acc0 + acc1;
    }
    __syncthreads();
    cholqr();
    cholqr();
    // how far did the basis move?  D = Y - Q (Q^T Y)
    for (int pr = warp; pr < 16; pr += nw) {
      const int k = pr >> 2, l = pr & 3;
      double acc = 0.0;
      for (int a = lane; a < n; a += 32) acc += Q[4 * a + k] * Y[4 * a + l];
      acc = warp_sum(acc);
      if (lane == 0) Mq[pr] = acc;
    }
    __syncthreads();
    double d2 = 0.0;
    for (int w = tid; w < 4 * n; w += nt) {
      const int a = w >> 2, l = w & 3;
      const double dd = Y[w] - (Q[4 * a] * Mq[l] + Q[4 * a + 1] * Mq[4 + l] + Q[4 * a + 2] * Mq[8 + l] +
                                Q[4 * a + 3] * Mq[12 + l]);
      d2 += dd * dd;
    }
    d2 = warp_sum(d2);
    if (lane == 0) dist2[warp] = d2;
    __syncthreads();
    if (tid == 0) {
      double tot = 0.0;
      for (int w = 0; w < nw; ++w) tot += dist2[w];
      if (extra < 0 && tot <= 1e-26) extra = 0;
      else if (extra >= 0) ++extra;
      s_stop = extra >= 2;
    }
    for (int k = tid; k < 4 * n; k += nt) Q[k] = Y[k];
    __syncthreads();
    if (s_stop) break;
  }
  for (int k = tid; k < 4 * n; k += nt) U4[k] = Q[k];
  if (tid == 0) status[0] = step < max_steps ? 1 : 0;
}

// ---- symmetric eigenproblem of the Gram matrix ---------------------------------------------------
// Parallel cyclic Jacobi in one CTA.  The n indices (padded to an even count with a dummy) are
// paired round-robin, n/2 disjoint rotations per step, n - 1 steps per sweep: each step computes
// the rotation angles, rotates the columns of G and V, then the rows of G.  Fixed order, fixed
// stopping rule: bit-reproducible.  The rotations work on G, a copy of Gin (which the callers still
// need), made after the early return: a converged subspace iteration costs no copy.  G and V live in
// global memory (L1/L2 resident: n <= 192).
__global__ void __launch_bounds__(256)
jacobi_eig_kernel(int n, const double* __restrict__ Gin, double* __restrict__ G, double* __restrict__ V,
                  double* __restrict__ U4, double* __restrict__ evals4, const int* __restrict__ status) {
  if (status && status[0] == 1) return;  // the subspace iteration already delivered U4
  extern __shared__ double jsm[];
  const int ne = n + (n & 1), h = ne / 2;
  double* cs = jsm;                                  // [h][2]
  int* pl = reinterpret_cast<int*>(jsm + 2 * h);     // [ne] players
  int* tmp = pl + ne;                                // [ne]
  __shared__ double scratch[32];
  __shared__ int s_done;
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int k = tid; k < n * n; k += nt) {
    G[k] = Gin[k];
    V[k] = (k / n == k % n) ? 1.0 : 0.0;
  }
  for (int k = tid; k < ne; k += nt) pl[k] = k;
  __syncthreads();
  for (int sweep = 0; sweep < 40; ++sweep) {
    double off = 0.0, dg = 0.0;
    for (int k = tid; k < n * n; k += nt) {
      const double v = G[k];
      if (k / n == k % n) dg += v * v; else off += v * v;
    }
    off = block_sum(off, scratch);
    dg = block_sum(dg, scratch);
    if (tid == 0) s_done = !(off > 1e-31 * dg);
    __syncthreads();
    if (s_done) break;
    for (int step = 0; step < ne - 1; ++step) {
      if (tid < h) {
        int p = pl[tid], q = pl[ne - 1 - tid];
        if (p > q) { const int t = p; p = q; q = t; }
        double c = 1.0, s = 0.0;
        if (q < n) {
          const double apq = G[(size_t)p * n + q];
          if (apq != 0.0) {
            const double tau = (G[(size_t)q * n + q] - G[(size_t)p * n + p]) / (2.0 * apq);
            const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
            c = 1.0 / sqrt(1.0 + t * t);
            s = t * c;
          }
        }
        cs[2 * tid] = c;
        cs[2 * tid + 1] = s;
      }
      __syncthreads();
      // columns p, q of G and V
      for (int w = tid; w < h * n; w += nt) {
        const int k = w / n, r = w - k * n;
        int p = pl[k], q = pl[ne - 1 - k];
        if (p > q) { const int t = p; p = q; q = t; }
        if (q >= n) continue;
        const double c = cs[2 * k], s = cs[2 * k + 1];
        const double gp = G[(size_t)r * n + p], gq = G[(size_t)r * n + q];
        G[(size_t)r * n + p] = c * gp - s * gq;
        G[(size_t)r * n + q] = s * gp + c * gq;
        const double vp = V[(size_t)r * n + p], vq = V[(size_t)r * n + q];
        V[(size_t)r * n + p] = c * vp - s * vq;
        V[(size_t)r * n + q] = s * vp + c * vq;
      }
      __syncthreads();
      // rows p, q of G
      for (int w = tid; w < h * n; w += nt) {
        const int k = w / n, r = w - k * n;
        int p = pl[k], q = pl[ne - 1 - k];
        if (p > q) { const int t = p; p = q; q = t; }
        if (q >= n) continue;
        const double c = cs[2 * k], s = cs[2 * k + 1];
        const double gp = G[(size_t)p * n + r], gq = G[(size_t)q * n + r];
        G[(size_t)p * n + r] = c * gp - s * gq;
        G[(size_t)q * n + r] = s * gp + c * gq;
      }
      __syncthreads();
      // next round of the tournament: player 0 stays, the others move on by one seat
      for (int k = tid; k < ne; k += nt) tmp[k] = k == 0 ? pl[0] : (k == 1 ? pl[ne - 1] : pl[k - 1]);
      __syncthreads();
      for (int k = tid; k < ne; k += nt) pl[k] = tmp[k];
      __syncthreads();
    }
  }
  // the four largest eigenvalues (selection in a fixed order) and their eigenvectors
  __shared__ int top[4];
  if (tid == 0) {
    for (int k = 0; k < 4; ++k) {
      int best = -1;
      for (int a = 0; a < n; ++a) {
        bool used = false;
        for (int m = 0; m < k; ++m) used |= top[m] == a;
        if (!used && (best < 0 || G[(size_t)a * n + a] > G[(size_t)best * n + best])) best = a;
      }
      top[k] = best;
      evals4[k] = G[(size_t)best * n + best];
    }
  }
  __syncthreads();
  for (int w = tid; w < 4 * n; w += nt) {
    const int a = w >> 2, k = w & 3;
    U4[w] = V[(size_t)a * n + top[k]];
  }
}

// ---- per point: new depths and the reprojection error ---------------------------------------------
// Leading eigenvector of a symmetric 4 x 4 matrix by cyclic Jacobi in registers (every lane of the
// warp runs it on identical inputs).
__device__ __forceinline__ void top_eigvec4(double (&a)[4][4], double (&v)[4]) {
  double e[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) e[r][c] = r == c ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 12; ++sweep) {
    // converged?  (all lanes hold the same matrix: the branch is uniform.)  Cyclic Jacobi converges
    // quadratically; a 4 x 4 matrix needs 4-5 sweeps, and each rotation costs two divisions and two
    // square roots in FP64 -- the fixed 12 sweeps were 84 % of the whole pass in the launch list.
    const double off = a[0][1] * a[0][1] + a[0][2] * a[0][2] + a[0][3] * a[0][3] + a[1][2] * a[1][2] +
                       a[1][3] * a[1][3] + a[2][3] * a[2][3];
    const double dg = a[0][0] * a[0][0] + a[1][1] * a[1][1] + a[2][2] * a[2][2] + a[3][3] * a[3][3];
    if (!(off > 1e-33 * dg)) break;
#pragma unroll
    for (int p = 0; p < 3; ++p)
#pragma unroll
      for (int q = p + 1; q < 4; ++q) {
        const double apq = a[p][q];
        if (apq == 0.0) continue;
        const double tau = (a[q][q] - a[p][p]) / (2.0 * apq);
        const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
        const double c = 1.0 / sqrt(1.0 + t * t), s = t * c;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const double gp = a[r][p], gq = a[r][q];
          a[r][p] = c * gp - s * gq;
          a[r][q] = s * gp + c * gq;
          const double vp = e[r][p], vq = e[r][q];
          e[r][p] = c * vp - s * vq;
          e[r][q] = s * vp + c * vq;
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const double gp = a[p][r], gq = a[q][r];
          a[p][r] = c * gp - s * gq;
          a[q][r] = s * gp + c * gq;
        }
      }
  }
  int best = 0;
#pragma unroll
  for (int k = 1; k < 4; ++k)
    if (a[k][k] > a[best][best]) best = k;
#pragma unroll
  for (int r = 0; r < 4; ++r) v[r] = best == 0 ? e[r][0] : (best == 1 ? e[r][1] : (best == 2 ? e[r][2] : e[r][3]));
}

__global__ void __launch_bounds__(256)
depth_update_kernel(int64_t N, int M, int ld, const double* __restrict__ x, const double* __restrict__ Wn,
                    const double* __restrict__ U4, double* __restrict__ z, double* __restrict__ err_part) {
  extern __shared__ double su[];  // U4 [3M][4]
  __shared__ double scratch[32];
  for (int k = threadIdx.x; k < 12 * M; k += blockDim.x) su[k] = U4[k];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  double err = 0.0;
  for (int64_t j = warp; j < N; j += nwarps) {
    const double* xj = x + (size_t)j * M * 3;
    // coefficients of the point in the leading subspace: c = U4^T w   (M S = U4 U4^T W, :133-134)
    double c0 = 0, c1 = 0, c2 = 0, c3 = 0;
    for (int a = lane; a < 3 * M; a += 32) {
      const double w = Wn[(size_t)j * ld + a];
      c0 += w * su[4 * a]; c1 += w * su[4 * a + 1]; c2 += w * su[4 * a + 2]; c3 += w * su[4 * a + 3];
    }
    c0 = warp_sum(c0); c1 = warp_sum(c1); c2 = warp_sum(c2); c3 = warp_sum(c3);
    // 4 x 4 Gram of B (:98-113 in factored form) and the reprojection error of this pass (:44-58)
    double g[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = lane; i < M; i += 32) {
      const double x0 = xj[3 * i], x1 = xj[3 * i + 1], x2 = xj[3 * i + 2];
      const double inv = 1.0 / sqrt(x0 * x0 + x1 * x1 + x2 * x2);
      const double* u = su + 12 * i;  // rows 3i, 3i+1, 3i+2 of U4
      double b[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) b[k] = (x0 * u[k] + x1 * u[4 + k] + x2 * u[8 + k]) * inv;
      int idx = 0;
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int cc = r; cc < 4; ++cc) g[idx++] += b[r] * b[cc];
      const double p0 = u[0] * c0 + u[1] * c1 + u[2] * c2 + u[3] * c3;
      const double p1 = u[4] * c0 + u[5] * c1 + u[6] * c2 + u[7] * c3;
      const double p2 = u[8] * c0 + u[9] * c1 + u[10] * c2 + u[11] * c3;
      const double d0 = x0 - p0 / p2, d1 = x1 - p1 / p2, d2 = x2 - p2 / p2;
      err += d0 * d0 + d1 * d1 + d2 * d2;
    }
#pragma unroll
    for (int k = 0; k < 10; ++k) g[k] = warp_sum(g[k]);
    double a[4][4], v[4];
    {
      int idx = 0;
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int cc = r; cc < 4; ++cc) { a[r][cc] = g[idx]; a[cc][r] = g[idx]; ++idx; }
    }
    top_eigvec4(a, v);
    // xi = B v / |B v|, sign so that sum(xi) >= 0 (:127-128), z = xi / |x| (:131)
    double nrm = 0.0, sum = 0.0;
    for (int i = lane; i < M; i += 32) {
      const double x0 = xj[3 * i], x1 = xj[3 * i + 1], x2 = xj[3 * i + 2];
      const double inv = 1.0 / sqrt(x0 * x0 + x1 * x1 + x2 * x2);
      const double* u = su + 12 * i;
      double xi = 0.0;
#pragma unroll
      for (int k = 0; k < 4; ++k) xi += (x0 * u[k] + x1 * u[4 + k] + x2 * u[8 + k]) * inv * v[k];
      nrm += xi * xi;
      sum += xi;
    }
    nrm = warp_sum(nrm);
    sum = warp_sum(sum);
    const double scale = (sum < 0.0 ? -1.0 : 1.0) / sqrt(nrm);
    for (int i = lane; i < M; i += 32) {
      const double x0 = xj[3 * i], x1 = xj[3 * i + 1], x2 = xj[3 * i + 2];
      const double inv = 1.0 / sqrt(x0 * x0 + x1 * x1 + x2 * x2);
      const double* u = su + 12 * i;
      double xi = 0.0;
#pragma unroll
      for (int k = 0; k < 4; ++k) xi += (x0 * u[k] + x1 * u[4 + k] + x2 * u[8 + k]) * inv * v[k];
      z[(size_t)j * M + i] = xi * scale * inv;
    }
  }
  const double tot = block_sum(err, scratch);
  if (threadIdx.x == 0) err_part[blockIdx.x] = tot;
}

__global__ void depth_error_kernel(const double* __restrict__ part, int n, double count, double f0,
                                   double* __restrict__ out) {
  __shared__ double scratch[32];
  double acc = 0.0;
  for (int k = threadIdx.x; k < n; k += blockDim.x) acc += part[k];
  const double tot = block_sum(acc, scratch);
  if (threadIdx.x == 0) *out = f0 * sqrt(tot / count);  // :56
}


// ==================================================================================================
// Dual method (reference :147-235) and the rank-4 factorisation (lib/factorization.py:5-15)
// ==================================================================================================
// Per pass the reference normalises W per IMAGE (:171-176), takes the four leading RIGHT singular
// vectors V_ (N x 4, :178-181) and solves, per image, the N x N eigenproblem of
//   B_i[j][l] = (v_j . v_l)(x_ij . x_il) / (|x_ij| |x_il|)                       (:183-204)
// -- an (n_images, n_points, n_points) array (:188), the O(M N^2) memory that keeps the method from
// large scenes.  B_i = C_i C_i^T with the N x 12 matrix C_i[j][(a, b)] = v_j[a] xhat_ij[b], so its
// leading eigenvector is C_i w / |C_i w| with w the leading eigenvector of the 12 x 12 matrix
// C_i^T C_i = sum_j (v_j v_j^T) (x) (xhat_ij xhat_ij^T); and V_ enters only through V_ V_^T, so any
// orthonormal basis of the leading right singular subspace will do: V4 = Wn U4 L^-T with
// U4 = basis of the leading eigenspace of G = Wn^T Wn (3M x 3M, tensor-core SYRK) and L L^T =
// U4^T G U4.  Memory is O(M N) throughout.
//   dual_norm_kernel       per-warp partials of the per-image squared norms of x z
//   colsum_finish_kernel   fixed-order sums of per-warp partials (all per-image reductions)
//   dual_scale_kernel      Wn = x z / norm2_i  (k-major, row = point)
//   Gram + subspace_eig    as in the primary method
//   dual_small_kernel      T = U4^T G U4, Cholesky, L^-1
//   dual_v_kernel          warp per point: c = U4^T wn_j, v_j = L^-1 c, reprojection-error share
//   dual_outer_kernel      per image sum_j (v v^T) (x) (xhat xhat^T): 10 x 6 unique products
//   dual_eig12_kernel      warp per image: cyclic Jacobi on the 12 x 12 matrix in shared memory
//   dual_e_kernel          e_ij = sum v_j[a] xhat_ij[b] w_i[a, b]; per-image sum e^2, sum e
//   dual_z_kernel          xi = e / |e_i| with each image's sum made non-negative (the sign LAPACK
//                          leaves open, see oracle/depth_oracle.py), then the reference's row rule
//                          (:212-215) and z = xi / |x|  (:218)
constexpr int kMaxImageSlots = 2;  // images per lane: n_images <= 64

__device__ __forceinline__ int64_t warp_global() { return ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; }
__device__ __forceinline__ int64_t warps_total() { return ((int64_t)gridDim.x * blockDim.x) >> 5; }

__global__ void __launch_bounds__(256)
dual_norm_kernel(int64_t N, int M, const double* __restrict__ x, const double* __restrict__ z,
                 double* __restrict__ part) {
  const int lane = threadIdx.x & 31;
  const int64_t w = warp_global(), nw = warps_total();
  for (int s = 0; s * 32 < M; ++s) {
    const int i = lane + 32 * s;
    double acc = 0.0;
    if (i < M)
      for (int64_t j = w; j < N; j += nw) {
        const double* xv = x + ((size_t)j * M + i) * 3;
        const double zz = z[(size_t)j * M + i];
        const double a = xv[0] * zz, b = xv[1] * zz, c = xv[2] * zz;
        acc += a * a + b * b + c * c;
      }
    if (i < M) part[(size_t)w * M + i] = acc;
  }
}

// out[k] = sum_r part[r][k], r ascending (deterministic), k < width
__global__ void colsum_finish_kernel(const double* __restrict__ part, int64_t rows, int width,
                                     double* __restrict__ out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= width) return;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  int64_t r = 0;
  for (; r + 3 < rows; r += 4) {
    a0 += part[(size_t)r * width + k];
    a1 += part[(size_t)(r + 1) * width + k];
    a2 += part[(size_t)(r + 2) * width + k];
    a3 += part[(size_t)(r + 3) * width + k];
  }
  for (; r < rows; ++r) a0 += part[(size_t)r * width + k];
  out[k] = (a0 + a1) + (a2 + a3);
}

__global__ void __launch_bounds__(256)
dual_scale_kernel(int64_t N, int M, int ld, const double* __restrict__ x, const double* __restrict__ z,
                  const double* __restrict__ norm2, double* __restrict__ Wn) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = warps_total();
  for (int64_t j = warp_global(); j < N; j += nw) {
    const double* xj = x + (size_t)j * M * 3;
    const double* zj = z + (size_t)j * M;
    double* out = Wn + (size_t)j * ld;
    for (int a = lane; a < ld; a += 32) out[a] = a < 3 * M ? (xj[a] * zj[a / 3]) / norm2[a / 3] : 0.0;  // :171-176
  }
}

// Plain copy of W (k-major) into the padded operand of the Gram kernel (factorisation).
__global__ void __launch_bounds__(256)
pad_rows_kernel(int64_t N, int n, int ld, const double* __restrict__ W, double* __restrict__ Wk) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = warps_total();
  for (int64_t j = warp_global(); j < N; j += nw)
    for (int a = lane; a < ld; a += 32) Wk[(size_t)j * ld + a] = a < n ? W[(size_t)j * n + a] : 0.0;
}

// Affine path (reference lib/affine_camera_calibration.py:224-240, _get_observation_matrix): the
// observation matrix is centred per row of W = per column of the k-major array.  Per-warp partial
// column sums in a fixed order (colsum_finish_kernel adds them), then the copy subtracts the means.
__global__ void __launch_bounds__(256)
col_partial_kernel(int64_t N, int n, const double* __restrict__ W, double* __restrict__ part) {
  const int lane = threadIdx.x & 31;
  const int64_t w = warp_global(), nw = warps_total();
  for (int a = lane; a < n; a += 32) {
    double acc = 0.0;
    for (int64_t j = w; j < N; j += nw) acc += W[(size_t)j * n + a];
    part[(size_t)w * n + a] = acc;
  }
}

__global__ void __launch_bounds__(256)
pad_rows_centred_kernel(int64_t N, int n, int ld, const double* __restrict__ W, const double* __restrict__ colsum,
                        double* __restrict__ mean, double* __restrict__ Wk) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = warps_total();
  const double inv = 1.0 / (double)N;
  if (blockIdx.x == 0)
    for (int a = threadIdx.x; a < n; a += blockDim.x) mean[a] = colsum[a] * inv;
  for (int64_t j = warp_global(); j < N; j += nw)
    for (int a = lane; a < ld; a += 32)
      Wk[(size_t)j * ld + a] = a < n ? W[(size_t)j * n + a] - colsum[a] * inv : 0.0;
}

// Cyclic Jacobi on a symmetric K x K matrix held by ONE thread (K <= 12): eigenvalues on the
// diagonal of a, eigenvectors in the columns of e.
template <int K>
__device__ void jacobi_small(double (&a)[K][K], double (&e)[K][K]) {
  for (int r = 0; r < K; ++r)
    for (int c = 0; c < K; ++c) e[r][c] = r == c ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 30; ++sweep) {
    double off = 0.0, dg = 0.0;
    for (int r = 0; r < K; ++r)
      for (int c = 0; c < K; ++c) {
        const double v = a[r][c] * a[r][c];
        if (r == c) dg += v; else off += v;
      }
    if (!(off > 1e-30 * dg)) break;
    for (int p = 0; p < K - 1; ++p)
      for (int q = p + 1; q < K; ++q) {
        const double apq = a[p][q];
        if (apq == 0.0) continue;
        const double tau = (a[q][q] - a[p][p]) / (2.0 * apq);
        const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
        const double c = 1.0 / sqrt(1.0 + t * t), s = t * c;
        for (int r = 0; r < K; ++r) {
          const double gp = a[r][p], gq = a[r][q];
          a[r][p] = c * gp - s * gq;
          a[r][q] = s * gp + c * gq;
          const double vp = e[r][p], vq = e[r][q];
          e[r][p] = c * vp - s * vq;
          e[r][q] = s * vp + c * vq;
        }
        for (int r = 0; r < K; ++r) {
          const double gp = a[p][r], gq = a[q][r];
          a[p][r] = c * gp - s * gq;
          a[q][r] = s * gp + c * gq;
        }
      }
  }
}

// One block.  T = U4^T G U4 (4 x 4).  mode 0 (dual method): T = L L^T, small[0..15] = L^-1 (lower).
// mode 1 (factorisation): T = Z Lambda Z^T with descending eigenvalues, U4 <- U4 Z (the four leading
// left singular vectors of W), small[16..19] = singular values sqrt(Lambda).
__global__ void __launch_bounds__(256)
dual_small_kernel(int n, const double* __restrict__ G, double* __restrict__ U4, double* __restrict__ small,
                  int mode) {
  extern __shared__ double sh[];  // GU [n][4]
  __shared__ double T[16], Zs[16];
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
  for (int w = tid; w < 4 * n; w += nt) {
    const int a = w >> 2, k = w & 3;
    const double* g = G + (size_t)a * n;
    double acc = 0.0;
    for (int b = 0; b < n; ++b) acc = fma(g[b], U4[4 * b + k], acc);
    sh[w] = acc;
  }
  __syncthreads();
  for (int pr = warp; pr < 16; pr += nw) {
    const int k = pr >> 2, l = pr & 3;
    double acc = 0.0;
    for (int a = lane; a < n; a += 32) acc += U4[4 * a + k] * sh[4 * a + l];
    acc = warp_sum(acc);
    if (lane == 0) T[pr] = acc;
  }
  __syncthreads();
  if (tid == 0) {
    double t[4][4];
    for (int r = 0; r < 4; ++r)
      for (int c = 0; c < 4; ++c) t[r][c] = 0.5 * (T[4 * r + c] + T[4 * c + r]);
    if (mode == 0) {
      double L[4][4] = {}, I[4][4] = {};
      for (int c = 0; c < 4; ++c)
        for (int r = c; r < 4; ++r) {
          double v = t[r][c];
          for (int m = 0; m < c; ++m) v -= L[r][m] * L[c][m];
          L[r][c] = r == c ? sqrt(v) : v / L[c][c];
        }
      for (int c = 0; c < 4; ++c) {  // lower-triangular inverse by forward substitution
        I[c][c] = 1.0 / L[c][c];
        for (int r = c + 1; r < 4; ++r) {
          double v = 0.0;
          for (int m = c; m < r; ++m) v -= L[r][m] * I[m][c];
          I[r][c] = v / L[r][r];
        }
      }
      for (int r = 0; r < 4; ++r)
        for (int c = 0; c < 4; ++c) small[4 * r + c] = I[r][c];
    } else {
      double e[4][4];
      jacobi_small<4>(t, e);
      int order[4] = {0, 1, 2, 3};
      for (int a = 0; a < 3; ++a)
        for (int b = a + 1; b < 4; ++b)
          if (t[order[b]][order[b]] > t[order[a]][order[a]]) { const int x = order[a]; order[a] = order[b]; order[b] = x; }
      for (int k = 0; k < 4; ++k) {
        small[16 + k] = sqrt(t[order[k]][order[k]]);
        for (int r = 0; r < 4; ++r) Zs[4 * r + k] = e[r][order[k]];
      }
    }
  }
  __syncthreads();
  if (mode == 1)
    for (int a = tid; a < n; a += nt) {
      const double u0 = U4[4 * a], u1 = U4[4 * a + 1], u2 = U4[4 * a + 2], u3 = U4[4 * a + 3];
#pragma unroll
      for (int k = 0; k < 4; ++k) U4[4 * a + k] = u0 * Zs[k] + u1 * Zs[4 + k] + u2 * Zs[8 + k] + u3 * Zs[12 + k];
    }
}

// warp per point: c = U4^T wn_j; v_j = L^-1 c -> V4[j][4]; reprojection error of this pass (:219-221)
__global__ void __launch_bounds__(256)
dual_v_kernel(int64_t N, int M, int ld, const double* __restrict__ x, const double* __restrict__ Wn,
              const double* __restrict__ U4, const double* __restrict__ small, double* __restrict__ V4,
              double* __restrict__ err_part) {
  extern __shared__ double su[];  // U4 [3M][4]
  __shared__ double scratch[32];
  for (int k = threadIdx.x; k < 12 * M; k += blockDim.x) su[k] = U4[k];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t nw = warps_total();
  double err = 0.0;
  for (int64_t j = warp_global(); j < N; j += nw) {
    const double* xj = x + (size_t)j * M * 3;
    double c0 = 0, c1 = 0, c2 = 0, c3 = 0;
    for (int a = lane; a < 3 * M; a += 32) {
      const double w = Wn[(size_t)j * ld + a];
      c0 += w * su[4 * a]; c1 += w * su[4 * a + 1]; c2 += w * su[4 * a + 2]; c3 += w * su[4 * a + 3];
    }
    c0 = warp_sum(c0); c1 = warp_sum(c1); c2 = warp_sum(c2); c3 = warp_sum(c3);
    if (lane == 0) {
      double* v = V4 + 4 * (size_t)j;
      v[0] = small[0] * c0;
      v[1] = small[4] * c0 + small[5] * c1;
      v[2] = small[8] * c0 + small[9] * c1 + small[10] * c2;
      v[3] = small[12] * c0 + small[13] * c1 + small[14] * c2 + small[15] * c3;
    }
    for (int i = lane; i < M; i += 32) {
      const double x0 = xj[3 * i], x1 = xj[3 * i + 1], x2 = xj[3 * i + 2];
      const double* u = su + 12 * i;
      const double p0 = u[0] * c0 + u[1] * c1 + u[2] * c2 + u[3] * c3;
      const double p1 = u[4] * c0 + u[5] * c1 + u[6] * c2 + u[7] * c3;
      const double p2 = u[8] * c0 + u[9] * c1 + u[10] * c2 + u[11] * c3;
      const double d0 = x0 - p0 / p2, d1 = x1 - p1 / p2, d2 = x2 - p2 / p2;
      err += d0 * d0 + d1 * d1 + d2 * d2;
    }
  }
  const double tot = block_sum(err, scratch);
  if (threadIdx.x == 0) err_part[blockIdx.x] = tot;
}

// per image and warp: sum_j p_j[a] q_ij[b], p = unique entries of v v^T (10), q = of xhat xhat^T (6)
__global__ void __launch_bounds__(256)
dual_outer_kernel(int64_t N, int M, const double* __restrict__ x, const double* __restrict__ V4,
                  double* __restrict__ part /* [warps][M][60] */) {
  const int lane = threadIdx.x & 31;
  const int64_t w = warp_global(), nw = warps_total();
  for (int s = 0; s * 32 < M; ++s) {
    const int i = lane + 32 * s;
    double acc[60];
#pragma unroll
    for (int k = 0; k < 60; ++k) acc[k] = 0.0;
    for (int64_t j = w; j < N; j += nw) {
      const double4 v = *reinterpret_cast<const double4*>(V4 + 4 * (size_t)j);
      double q[6] = {0, 0, 0, 0, 0, 0};
      if (i < M) {
        const double* xv = x + ((size_t)j * M + i) * 3;
        const double x0 = xv[0], x1 = xv[1], x2 = xv[2];
        const double inv2 = 1.0 / (x0 * x0 + x1 * x1 + x2 * x2);
        q[0] = x0 * x0 * inv2; q[1] = x0 * x1 * inv2; q[2] = x0 * x2 * inv2;
        q[3] = x1 * x1 * inv2; q[4] = x1 * x2 * inv2; q[5] = x2 * x2 * inv2;
      }
      const double p[10] = {v.x * v.x, v.x * v.y, v.x * v.z, v.x * v.w, v.y * v.y,
                            v.y * v.z, v.y * v.w, v.z * v.z, v.z * v.w, v.w * v.w};
#pragma unroll
      for (int a = 0; a < 10; ++a)
#pragma unroll
        for (int b = 0; b < 6; ++b) acc[6 * a + b] = fma(p[a], q[b], acc[6 * a + b]);
    }
    if (i < M) {
      double* out = part + ((size_t)w * M + i) * 60;
#pragma unroll
      for (int k = 0; k < 60; ++k) out[k] = acc[k];
    }
  }
}

__device__ __forceinline__ int sym_pair(int a, int b, int n) {  // index of (a, b), a <= b, row-major upper
  if (a > b) { const int t = a; a = b; b = t; }
  return a * n - a * (a - 1) / 2 + (b - a);
}

// Cyclic Jacobi on a symmetric K x K matrix by ONE WARP: A and the eigenvector matrix E live in
// shared memory, lane r owns row r of the column rotation and column r of the row rotation.
// (A single-thread version on local-memory arrays -- the straightforward code, fine on the host -- is
// miscompiled by nvcc 12.9 for sm_100a at K = 12: it stops converging after the first sweep;
// tools/jac_test.cu reproduces it next to this version.)  Returns with the eigenvalues on the
// diagonal of a; fixed order of operations.
template <int K>
__device__ void jacobi_warp(double* a, double* e) {
  const int lane = threadIdx.x & 31;
  for (int k = lane; k < K * K; k += 32) e[k] = (k / K == k % K) ? 1.0 : 0.0;
  __syncwarp();
  for (int sweep = 0; sweep < 30; ++sweep) {
    double off = 0.0, dg = 0.0;
    for (int k = lane; k < K * K; k += 32) {
      const double v = a[k] * a[k];
      if (k / K == k % K) dg += v; else off += v;
    }
    off = warp_sum(off);
    dg = warp_sum(dg);
    if (!(off > 1e-30 * dg)) break;
    for (int p = 0; p < K - 1; ++p)
      for (int q = p + 1; q < K; ++q) {
        const double apq = a[p * K + q];
        double c = 1.0, s = 0.0;
        if (apq != 0.0) {
          const double tau = (a[q * K + q] - a[p * K + p]) / (2.0 * apq);
          const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
          c = 1.0 / sqrt(1.0 + t * t);
          s = t * c;
        }
        __syncwarp();
        if (lane < K) {  // columns p, q of A and E
          const double gp = a[lane * K + p], gq = a[lane * K + q];
          a[lane * K + p] = c * gp - s * gq;
          a[lane * K + q] = s * gp + c * gq;
          const double vp = e[lane * K + p], vq = e[lane * K + q];
          e[lane * K + p] = c * vp - s * vq;
          e[lane * K + q] = s * vp + c * vq;
        }
        __syncwarp();
        if (lane < K) {  // rows p, q of A
          const double gp = a[p * K + lane], gq = a[q * K + lane];
          a[p * K + lane] = c * gp - s * gq;
          a[q * K + lane] = s * gp + c * gq;
        }
        __syncwarp();
      }
  }
}

// warp (= block) per image: 12 x 12 matrix from the 10 x 6 products, leading eigenvector -> W12[i][12]
__global__ void __launch_bounds__(32) dual_eig12_kernel(int M, const double* __restrict__ R60, double* __restrict__ W12) {
  __shared__ double a[144], e[144];
  const int i = blockIdx.x, lane = threadIdx.x;
  if (i >= M) return;
  const double* r = R60 + (size_t)i * 60;
  for (int k = lane; k < 144; k += 32) {
    const int row = k / 12, col = k - 12 * row;
    a[k] = r[6 * sym_pair(row / 3, col / 3, 4) + sym_pair(row % 3, col % 3, 3)];
  }
  __syncwarp();
  jacobi_warp<12>(a, e);
  int best = 0;
  for (int k = 1; k < 12; ++k)
    if (a[k * 12 + k] > a[best * 12 + best]) best = k;
  if (lane < 12) W12[(size_t)i * 12 + lane] = e[lane * 12 + best];
}

// e_ij into ebuf[j][i]; per warp and image: sum e^2, sum e -> part[w][2][M]
__global__ void __launch_bounds__(256)
dual_e_kernel(int64_t N, int M, const double* __restrict__ x, const double* __restrict__ V4,
              const double* __restrict__ W12, double* __restrict__ ebuf, double* __restrict__ part) {
  const int lane = threadIdx.x & 31;
  const int64_t w = warp_global(), nw = warps_total();
  for (int s = 0; s * 32 < M; ++s) {
    const int i = lane + 32 * s;
    double wv[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) wv[k] = i < M ? W12[(size_t)i * 12 + k] : 0.0;
    double s2 = 0.0, s1 = 0.0;
    for (int64_t j = w; j < N; j += nw) {
      if (i >= M) continue;
      const double4 v = *reinterpret_cast<const double4*>(V4 + 4 * (size_t)j);
      const double* xv = x + ((size_t)j * M + i) * 3;
      const double x0 = xv[0], x1 = xv[1], x2 = xv[2];
      const double inv = 1.0 / sqrt(x0 * x0 + x1 * x1 + x2 * x2);
      const double h0 = x0 * inv, h1 = x1 * inv, h2 = x2 * inv;
      const double e = v.x * (h0 * wv[0] + h1 * wv[1] + h2 * wv[2]) + v.y * (h0 * wv[3] + h1 * wv[4] + h2 * wv[5]) +
                       v.z * (h0 * wv[6] + h1 * wv[7] + h2 * wv[8]) + v.w * (h0 * wv[9] + h1 * wv[10] + h2 * wv[11]);
      ebuf[(size_t)j * M + i] = e;
      s2 += e * e;
      s1 += e;
    }
    if (i < M) {
      part[((size_t)w * 2) * M + i] = s2;
      part[((size_t)w * 2 + 1) * M + i] = s1;
    }
  }
}

// sums[0][i] = sum e^2, sums[1][i] = sum e  ->  z
__global__ void __launch_bounds__(256)
dual_z_kernel(int64_t N, int M, const double* __restrict__ x, const double* __restrict__ ebuf,
              const double* __restrict__ sums, double* __restrict__ z) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = warps_total();
  double scale[kMaxImageSlots];
#pragma unroll
  for (int s = 0; s < kMaxImageSlots; ++s) {
    const int i = lane + 32 * s;
    scale[s] = i < M ? (sums[M + i] < 0.0 ? -1.0 : 1.0) / sqrt(sums[i]) : 0.0;
  }
  for (int64_t j = warp_global(); j < N; j += nw) {
    double xi[kMaxImageSlots], row = 0.0;
#pragma unroll
    for (int s = 0; s < kMaxImageSlots; ++s) {
      const int i = lane + 32 * s;
      xi[s] = i < M ? ebuf[(size_t)j * M + i] * scale[s] : 0.0;
      row += xi[s];
    }
    row = warp_sum(row);
    const double flip = row < 0.0 ? -1.0 : 1.0;  // :212-215
#pragma unroll
    for (int s = 0; s < kMaxImageSlots; ++s) {
      const int i = lane + 32 * s;
      if (i < M) {
        const double* xv = x + ((size_t)j * M + i) * 3;
        z[(size_t)j * M + i] = flip * xi[s] / sqrt(xv[0] * xv[0] + xv[1] * xv[1] + xv[2] * xv[2]);  // :218
      }
    }
  }
}

// S[k][j] = sum_a U[a][k] W[j][a]  (= diag(Sigma) V^T of the rank-4 factorisation)
__global__ void __launch_bounds__(256)
factor_shape_kernel(int64_t N, int n, int ld, const double* __restrict__ Wk, const double* __restrict__ U4,
                    double* __restrict__ S) {
  extern __shared__ double su[];
  for (int k = threadIdx.x; k < 4 * n; k += blockDim.x) su[k] = U4[k];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t nw = warps_total();
  for (int64_t j = warp_global(); j < N; j += nw) {
    double c0 = 0, c1 = 0, c2 = 0, c3 = 0;
    for (int a = lane; a < n; a += 32) {
      const double w = Wk[(size_t)j * ld + a];
      c0 += w * su[4 * a]; c1 += w * su[4 * a + 1]; c2 += w * su[4 * a + 2]; c3 += w * su[4 * a + 3];
    }
    c0 = warp_sum(c0); c1 = warp_sum(c1); c2 = warp_sum(c2); c3 = warp_sum(c3);
    if (lane == 0) {
      S[j] = c0; S[(size_t)N + j] = c1; S[2 * (size_t)N + j] = c2; S[3 * (size_t)N + j] = c3;
    }
  }
}

// Device buffers of one call, freed together on every exit path.
struct DevBufs {
  cudaStream_t s;
  std::vector<void*> ptrs;
  explicit DevBufs(cudaStream_t s_) : s(s_) {}
  template <typename T>
  int alloc(T** p, size_t n) {
    *p = nullptr;
    if (cudaMallocAsync(reinterpret_cast<void**>(p), (n ? n : 1) * sizeof(T), s) != cudaSuccess) {
      set_error("out of device memory (%zu bytes)", n * sizeof(T));
      cudaGetLastError();
      return BA_ERR_CUDA;
    }
    ptrs.push_back(*p);
    return BA_OK;
  }
  ~DevBufs() {
    if (ptrs.empty()) return;  // the call was rejected before it touched the device
    for (void* p : ptrs) cudaFreeAsync(p, s);
    cudaStreamSynchronize(s);
  }
};

static int check_launches(const char* what) {
  if (cudaGetLastError() == cudaSuccess) return BA_OK;
  set_error("%s: a kernel launch failed", what);
  return BA_ERR_CUDA;
}

// What the two depth methods and the factorisation share: the device, the k-major operand Wk
// [k_pad][ld] (one row per point, n entries used), its Gram matrix and leading eigenspace, the input
// (x or W) staged on the device and the output (z or S).  Every buffer is in `bufs` and the Gram
// product is released by the destructor, so every exit path frees everything.
struct DepthCall {
  cudaStream_t s;
  DevBufs bufs;
  SyrkProduct gram;  // FP64 64-tiles
  int num_sms = 0, n = 0, ld = 0, grid = 0, mem = BA_MEM_HOST;
  int64_t N = 0, k_pad = 0;
  bool force_jacobi = false;
  const double* in = nullptr;
  double *out = nullptr, *out_user = nullptr;
  size_t out_count = 0;
  double *Wk = nullptr, *P = nullptr, *G = nullptr, *V = nullptr, *U4 = nullptr, *ev = nullptr;
  int* status = nullptr;

  explicit DepthCall(void* stream) : s((cudaStream_t)stream), bufs(s) {}
  ~DepthCall() { syrk_release(&gram, s); }

  // `args_ok` and `usage`: the entry point's own argument rule and its message.  Wk gets N_ rows (points,
  // or columns of W) of n_ entries; in / out hold in_count / out_count doubles, on the device with
  // BA_MEM_DEVICE.
  int open(bool args_ok, const char* what, const char* usage, int device, int64_t N_, int n_,
           const double* in_, size_t in_count, double* out_, size_t out_count_, int mem_) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
      set_error("no CUDA device: %s has no CPU path", what);
      return BA_ERR_NO_DEVICE;
    }
    if (!args_ok || device < 0 || device >= ndev) {
      set_error("%s", usage);
      return BA_ERR_INVALID;
    }
    BA_CUDA(cudaSetDevice(device));
    BA_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, device));
    N = N_;
    n = n_;
    ld = (n + 7) / 8 * 8;
    k_pad = (N + 31) / 32 * 32;
    grid = balanced_blocks((N + 7) / 8, (int64_t)num_sms * 8);
    force_jacobi = std::getenv("BA_DEPTH_JACOBI") != nullptr;  // tests: the fallback path
    mem = mem_;
    out_user = out_;
    out_count = out_count_;
    BA_TRY(bufs.alloc(&Wk, (size_t)k_pad * ld));
    BA_TRY(bufs.alloc(&P, (size_t)ld * ld));
    BA_TRY(bufs.alloc(&G, (size_t)n * n));
    BA_TRY(bufs.alloc(&V, (size_t)2 * n * n));
    BA_TRY(bufs.alloc(&U4, (size_t)4 * n));
    BA_TRY(bufs.alloc(&ev, 4));
    BA_TRY(bufs.alloc(&status, 1));
    if (mem == BA_MEM_DEVICE) {
      in = in_;
      out = out_;
    } else {
      double* din = nullptr;
      BA_TRY(bufs.alloc(&din, in_count));
      BA_TRY(bufs.alloc(&out, out_count));
      BA_CUDA(cudaMemcpyAsync(din, in_, in_count * sizeof(double), cudaMemcpyHostToDevice, s));
      in = din;
    }
    BA_CUDA(cudaMemsetAsync(Wk, 0, (size_t)k_pad * ld * sizeof(double), s));
    BA_CUDA(cudaMemsetAsync(P, 0, (size_t)ld * ld * sizeof(double), s));
    BA_CUDA(cudaMemsetAsync(status, 0, sizeof(int), s));
    return syrk_prepare(&gram, SYRK_TILE64, ld, k_pad, num_sms, s);
  }

  // U4 = a basis of the leading four-dimensional eigenspace of G = Wk^T Wk, which stays intact: the
  // subspace iteration (warm-started from U4), then the Jacobi solver if that did not converge.
  int leading_subspace(bool warm) {
    BA_TRY(syrk_launch(&gram, Wk, P, nullptr, s, nullptr));
    gram_symmetrize_kernel<<<(n * n + 255) / 256, 256, 0, s>>>(n, ld, P, G);
    if (!force_jacobi)
      subspace_eig_kernel<<<1, 256, (size_t)8 * n * sizeof(double), s>>>(n, G, U4, warm ? 1 : 0, 2000, status);
    const size_t jac_smem = (size_t)(2 * ((n + 1) / 2)) * sizeof(double) + (size_t)2 * (n + 1) * sizeof(int) + 16;
    // V [2][n][n]: the eigenvectors, then the Jacobi solver's copy of G
    jacobi_eig_kernel<<<1, 256, jac_smem, s>>>(n, G, V + (size_t)n * n, V, U4, ev, force_jacobi ? nullptr : status);
    g_launch_count += 3;
    return BA_OK;
  }

  // with BA_MEM_HOST: the result to the caller's buffer (with BA_MEM_DEVICE the kernels wrote it there)
  cudaError_t copy_out() const {
    if (mem == BA_MEM_DEVICE) return cudaSuccess;
    return cudaMemcpyAsync(out_user, out, out_count * sizeof(double), cudaMemcpyDeviceToHost, s);
  }
};

// The pass loop of both depth methods.  z starts at 1 (:80, :160); pass(it) enqueues one pass, which
// updates z and leaves its reprojection error in dE; the host reads E and stops when E < tolerance or
// after max_iter passes (:138-142, :228-229).
template <class Pass>
static int run_passes(DepthCall& c, const char* what, const double* dE, double tolerance, int max_iter,
                      double* errors, int* n_iter, Pass pass) {
  {
    std::vector<double> ones(c.out_count, 1.0);
    BA_CUDA(cudaMemcpyAsync(c.out, ones.data(), ones.size() * sizeof(double), cudaMemcpyHostToDevice, c.s));
    BA_CUDA(cudaStreamSynchronize(c.s));
  }
  int st = BA_OK, it = 0;
  for (;;) {
    st = pass(it);
    if (st == BA_OK) st = check_launches(what);
    if (st != BA_OK) break;
    double E = 0.0;
    if (cudaMemcpyAsync(&E, dE, sizeof(double), cudaMemcpyDeviceToHost, c.s) != cudaSuccess ||
        cudaStreamSynchronize(c.s) != cudaSuccess) {
      set_error("%s: %s", what, cudaGetErrorString(cudaGetLastError()));
      st = BA_ERR_CUDA;
      break;
    }
    if (errors) errors[it] = E;
    ++it;
    if (E < tolerance || it >= max_iter) break;
  }
  *n_iter = it;
  if (st == BA_OK && c.copy_out() != cudaSuccess) st = BA_ERR_CUDA;
  return st;
}

}  // namespace ba

using namespace ba;

extern "C" int ba_projective_depth_primary(int device, int64_t n_points, int32_t n_images, const double* x,
                                           double f0, double tolerance, int max_iter, double* z,
                                           double* errors, int* n_iter, int mem, void* stream) {
  DepthCall c(stream);
  BA_TRY(c.open(x && z && n_iter && n_points >= 4 && n_images >= 2 && n_images <= 64 && max_iter >= 1,
                "the projective-depth iteration",
                "projective depth: need >= 4 points, 2..64 images, max_iter >= 1 and valid pointers", device,
                n_points, 3 * n_images, x, (size_t)n_points * n_images * 3, z, (size_t)n_points * n_images, mem));
  const int64_t N = n_points;
  const int M = n_images, grid = c.grid;
  cudaStream_t s = c.s;
  const double* dx = c.in;
  double* dz = c.out;
  double *part = nullptr, *dE = nullptr;
  BA_TRY(c.bufs.alloc(&part, (size_t)grid));
  BA_TRY(c.bufs.alloc(&dE, 1));
  auto pass = [&](int it) -> int {
    depth_scale_kernel<<<grid, 256, 0, s>>>(N, M, c.ld, dx, dz, c.Wk);
    BA_TRY(c.leading_subspace(it > 0));
    depth_update_kernel<<<grid, 256, (size_t)12 * M * sizeof(double), s>>>(N, M, c.ld, dx, c.Wk, c.U4, dz, part);
    depth_error_kernel<<<1, 256, 0, s>>>(part, grid, (double)N * (double)M, f0, dE);
    g_launch_count += 3;
    return BA_OK;
  };
  return run_passes(c, "projective depth", dE, tolerance, max_iter, errors, n_iter, pass);
}

extern "C" int ba_projective_depth_dual(int device, int64_t n_points, int32_t n_images, const double* x, double f0,
                                        double tolerance, int max_iter, double* z, double* errors, int* n_iter,
                                        int mem, void* stream) {
  DepthCall c(stream);
  BA_TRY(c.open(x && z && n_iter && n_points >= 4 && n_images >= 2 && n_images <= 32 * kMaxImageSlots,
                "the projective-depth iteration",
                "projective depth (dual): need >= 4 points, 2..64 images and valid pointers", device, n_points,
                3 * n_images, x, (size_t)n_points * n_images * 3, z, (size_t)n_points * n_images, mem));
  if (max_iter < 1) max_iter = 1;  // the reference runs at least one pass (:162-231)
  const int64_t N = n_points;
  const int M = n_images, n = c.n, grid = c.grid;
  const int64_t nwarps = (int64_t)grid * 8;
  const size_t d = sizeof(double);
  cudaStream_t s = c.s;
  double *part = nullptr, *sums = nullptr, *small = nullptr, *V4 = nullptr, *R60 = nullptr, *W12 = nullptr,
         *ebuf = nullptr, *errp = nullptr, *dE = nullptr;
  BA_TRY(c.bufs.alloc(&part, (size_t)nwarps * M * 60));
  BA_TRY(c.bufs.alloc(&sums, (size_t)2 * M));
  BA_TRY(c.bufs.alloc(&small, 32));
  BA_TRY(c.bufs.alloc(&V4, (size_t)4 * N));
  BA_TRY(c.bufs.alloc(&R60, (size_t)60 * M));
  BA_TRY(c.bufs.alloc(&W12, (size_t)12 * M));
  BA_TRY(c.bufs.alloc(&ebuf, (size_t)N * M));
  BA_TRY(c.bufs.alloc(&errp, (size_t)grid));
  BA_TRY(c.bufs.alloc(&dE, 1));
  const double* dx = c.in;
  double* dz = c.out;
  auto pass = [&](int it) -> int {
    dual_norm_kernel<<<grid, 256, 0, s>>>(N, M, dx, dz, part);
    colsum_finish_kernel<<<(M + 63) / 64, 64, 0, s>>>(part, nwarps, M, sums);
    dual_scale_kernel<<<grid, 256, 0, s>>>(N, M, c.ld, dx, dz, sums, c.Wk);
    BA_TRY(c.leading_subspace(it > 0));
    dual_small_kernel<<<1, 256, (size_t)4 * n * d, s>>>(n, c.G, c.U4, small, 0);
    dual_v_kernel<<<grid, 256, (size_t)12 * M * d, s>>>(N, M, c.ld, dx, c.Wk, c.U4, small, V4, errp);
    depth_error_kernel<<<1, 256, 0, s>>>(errp, grid, (double)N * (double)M, f0, dE);
    dual_outer_kernel<<<grid, 256, 0, s>>>(N, M, dx, V4, part);
    colsum_finish_kernel<<<(60 * M + 127) / 128, 128, 0, s>>>(part, nwarps, 60 * M, R60);
    dual_eig12_kernel<<<M, 32, 0, s>>>(M, R60, W12);
    dual_e_kernel<<<grid, 256, 0, s>>>(N, M, dx, V4, W12, ebuf, part);
    colsum_finish_kernel<<<(2 * M + 63) / 64, 64, 0, s>>>(part, nwarps, 2 * M, sums);
    dual_z_kernel<<<grid, 256, 0, s>>>(N, M, dx, ebuf, sums, dz);
    g_launch_count += 12;
    return BA_OK;
  };
  return run_passes(c, "projective depth (dual)", dE, tolerance, max_iter, errors, n_iter, pass);
}

static int factorize_rank4_impl(int device, int64_t n_cols, int32_t n_rows, const double* Wt, bool centre,
                                double* mean_out, double* M_out, double* S_out, double* sigma_out, int mem,
                                void* stream) {
  DepthCall c(stream);
  BA_TRY(c.open(Wt && M_out && S_out && n_cols >= 4 && n_rows >= 4 && n_rows <= 192, "the factorisation",
                "factorisation: need >= 4 columns, 4..192 rows and valid pointers", device, n_cols, n_rows, Wt,
                (size_t)n_cols * n_rows, S_out, (size_t)4 * n_cols, mem));
  const int64_t N = n_cols;
  const int n = n_rows, grid = c.grid;
  const size_t d = sizeof(double);
  cudaStream_t s = c.s;
  const cudaMemcpyKind kind = mem == BA_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  double* small = nullptr;
  BA_TRY(c.bufs.alloc(&small, 32));
  if (centre) {
    double *part = nullptr, *colsum = nullptr, *mean = nullptr;
    const int64_t warps = (int64_t)grid * 8;
    BA_TRY(c.bufs.alloc(&part, (size_t)warps * n));
    BA_TRY(c.bufs.alloc(&colsum, (size_t)n));
    BA_TRY(c.bufs.alloc(&mean, (size_t)n));
    col_partial_kernel<<<grid, 256, 0, s>>>(N, n, c.in, part);
    colsum_finish_kernel<<<(n + 63) / 64, 64, 0, s>>>(part, warps, n, colsum);
    pad_rows_centred_kernel<<<grid, 256, 0, s>>>(N, n, c.ld, c.in, colsum, mean, c.Wk);
    g_launch_count += 2;
    if (mean_out) BA_CUDA(cudaMemcpyAsync(mean_out, mean, (size_t)n * d, kind, s));
  } else {
    pad_rows_kernel<<<grid, 256, 0, s>>>(N, n, c.ld, c.in, c.Wk);
  }
  BA_TRY(c.leading_subspace(false));
  dual_small_kernel<<<1, 256, (size_t)4 * n * d, s>>>(n, c.G, c.U4, small, 1);
  factor_shape_kernel<<<grid, 256, (size_t)4 * n * d, s>>>(N, n, c.ld, c.Wk, c.U4, c.out);
  g_launch_count += 3;
  BA_TRY(check_launches("factorisation"));
  if (cudaMemcpyAsync(M_out, c.U4, (size_t)4 * n * d, kind, s) != cudaSuccess ||
      (sigma_out && cudaMemcpyAsync(sigma_out, small + 16, 4 * d, kind, s) != cudaSuccess) ||
      c.copy_out() != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) {
    set_error("factorisation: %s", cudaGetErrorString(cudaGetLastError()));
    return BA_ERR_CUDA;
  }
  return BA_OK;
}

extern "C" int ba_factorize_rank4(int device, int64_t n_cols, int32_t n_rows, const double* Wt, double* M_out,
                                  double* S_out, double* sigma_out, int mem, void* stream) {
  return factorize_rank4_impl(device, n_cols, n_rows, Wt, false, nullptr, M_out, S_out, sigma_out, mem, stream);
}

extern "C" int ba_factorize_centred_rank4(int device, int64_t n_cols, int32_t n_rows, const double* Wt,
                                          double* mean_out, double* M_out, double* S_out, double* sigma_out,
                                          int mem, void* stream) {
  return factorize_rank4_impl(device, n_cols, n_rows, Wt, true, mean_out, M_out, S_out, sigma_out, mem, stream);
}
