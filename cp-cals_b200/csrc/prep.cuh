// Streaming (HBM-bound) kernels that run once per tensor: device layouts and norms.
//
//   pad_copy_kernel        X (dense, mode 0 fastest)  ->  Xp with the fastest dimension padded to an even pitch
//   swap01_copy_kernel     X -> Xt with modes 0 and 1 swapped (mode 1 fastest), pitch padded to even
//   rot201_copy_kernel     3-mode X -> Xr with mode order (2, 0, 1) (mode 2 fastest), pitch padded to even
//   halves_swap_kernel     4-mode X -> Xq with the mode pairs (0,1) and (2,3) exchanged (mode 2 fastest), pitch padded
//   rowsumsq_*             per mode-0 index sums of squares in ONE pass over X, from which both
//                            ||X||          Tensor::norm                       reference include/tensor.h:196
//                            ||X||_jk[i]    utils::calculate_jackknifing_norms reference src/utils/utils.cpp:103-152
//                          follow.
//   khatri_rao_kernel      K = A (.) B, the explicit two-matrix Khatri-Rao product of the reference's API
//                            (mttkrp::khatri_rao, reference src/utils/mttkrp.cpp:78-103; its CUDA twin
//                            src/utils/khatri_rao.cu:10-55).  The iteration path never materialises K (mttkrp.cuh); this
//                            kernel only serves callers of that API function.
#pragma once
#include <cuda_runtime.h>

namespace calsb200 {

// K[ib + IB * ia, c] = A[ia, c] * B[ib, c]   (B's row index fastest, reference src/utils/mttkrp.cpp:88-96).
// grid = (ceil(IA*IB / 1024), cols): one column per blockIdx.y, 4 consecutive rows of K per thread -> coalesced stores;
// the column of A is read through L1/L2 (IA values per column), B's column likewise.
__global__ void __launch_bounds__(256)
khatri_rao_kernel(const double *__restrict__ A, const double *__restrict__ B, int IA, int IB, double *__restrict__ K) {
  const long long c = blockIdx.y;
  const long long rows = (long long)IA * IB;
  const double *a = A + c * IA, *b = B + c * IB;
  double *k = K + c * rows;
  const long long r0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
#pragma unroll
  for (int u = 0; u < 4; u++) {
    const long long r = r0 + u;
    if (r < rows) {
      const int ia = (int)(r / IB), ib = (int)(r - (long long)ia * IB);
      k[r] = a[ia] * b[ib];
    }
  }
}

__global__ void pad_copy_kernel(const double *__restrict__ X, double *__restrict__ Xp, int I0, int ld0,
                                long long rest) {
  const long long total = (long long)ld0 * rest;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
       e += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(e % ld0);
    const long long r = e / ld0;
    Xp[e] = i < I0 ? X[r * I0 + i] : 0.0;
  }
}

// Xt[i1 + ld1 * (i0 + I0 * r)] = X[i0 + I0 * (i1 + I1 * r)],  grid = (ceil(I0/32), ceil(I1/32), rest2 chunks)
__global__ void swap01_copy_kernel(const double *__restrict__ X, double *__restrict__ Xt, int I0, int I1, int ld1,
                                   long long rest2) {
  __shared__ double t[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5; // 256 threads
  const int a0 = blockIdx.x * 32, b0 = blockIdx.y * 32;
  for (long long r = blockIdx.z; r < rest2; r += gridDim.z) {
    const double *Xs = X + r * (long long)I0 * I1;
    double *Xd = Xt + r * (long long)ld1 * I0;
    __syncthreads();
    for (int bb = ty; bb < 32; bb += 8) {
      const int i0 = a0 + tx, i1 = b0 + bb;
      t[bb][tx] = (i0 < I0 && i1 < I1) ? Xs[(long long)i1 * I0 + i0] : 0.0;
    }
    __syncthreads();
    for (int aa = ty; aa < 32; aa += 8) {
      const int i0 = a0 + aa, i1 = b0 + tx;
      if (i0 < I0 && i1 < ld1)
        Xd[(long long)i0 * ld1 + i1] = (i1 < I1) ? t[tx][aa] : 0.0;
    }
  }
}

// 3 modes: Xr[i2 + ldr * (i0 + I0 * i1)] = Xp[i0 + ld0 * (i1 + I1 * i2)], mode order (2, 0, 1): the contraction over mode
// 2 of the multi-sweep dimension tree reads it with mode 2 contiguous (engine.cu).  The transpose of X viewed as the
// (I0*I1) x I2 matrix; grid = (ceil(I0*I1 / 32), ceil(I2 / 32))
__global__ void rot201_copy_kernel(const double *__restrict__ Xp, double *__restrict__ Xr, int I0, int I1, int I2,
                                   int ld0, int ldr) {
  __shared__ double t[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5; // 256 threads
  const long long R = (long long)I0 * I1, r0 = (long long)blockIdx.x * 32;
  const int k0 = blockIdx.y * 32;
  for (int kk = ty; kk < 32; kk += 8) {
    const long long r = r0 + tx;
    const int i2 = k0 + kk;
    double v = 0.0;
    if (r < R && i2 < I2) {
      const long long i1 = r / I0, i0 = r - i1 * I0;
      v = Xp[i0 + (long long)ld0 * (i1 + (long long)I1 * i2)];
    }
    t[kk][tx] = v;
  }
  __syncthreads();
  for (int rr = ty; rr < 32; rr += 8) {
    const long long r = r0 + rr;
    const int i2 = k0 + tx;
    if (r < R && i2 < ldr)
      Xr[i2 + (long long)ldr * r] = i2 < I2 ? t[tx][rr] : 0.0;
  }
}

// 4 modes: Xq[i2 + ldq * (i3 + I3 * (i0 + I0 * i1))] = Xp[i0 + ld0 * (i1 + I1 * (i2 + I2 * i3))], i.e. the transpose of X
// viewed as the (I0*I1) x (I2*I3) matrix; the pair node of modes (0,1) contracts modes 2 and 3 along Xq's contiguous
// dimension (pairnode.cuh).  grid = (ceil(I0/32), ceil(I2/32), chunks of I1*I3)
__global__ void halves_swap_kernel(const double *__restrict__ Xp, double *__restrict__ Xq, int I0, int I1, int I2,
                                   int I3, int ld0, int ldq) {
  __shared__ double t[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5; // 256 threads
  const int a0 = blockIdx.x * 32, b0 = blockIdx.y * 32;
  const long long rest = (long long)I1 * I3;
  for (long long r = blockIdx.z; r < rest; r += gridDim.z) {
    const int i1 = (int)(r % I1), i3 = (int)(r / I1);
    __syncthreads();
    for (int bb = ty; bb < 32; bb += 8) {
      const int i0 = a0 + tx, i2 = b0 + bb;
      t[bb][tx] = (i0 < I0 && i2 < I2) ? Xp[i0 + (long long)ld0 * (i1 + (long long)I1 * (i2 + (long long)I2 * i3))] : 0.0;
    }
    __syncthreads();
    for (int aa = ty; aa < 32; aa += 8) {
      const int i0 = a0 + aa, i2 = b0 + tx;
      if (i0 < I0 && i2 < ldq)
        Xq[i2 + (long long)ldq * (i3 + (long long)I3 * (i0 + (long long)I0 * i1))] = (i2 < I2) ? t[tx][aa] : 0.0;
    }
  }
}

// partial[cta][i] = sum over this CTA's column range of X(i, j)^2.   X viewed I0 x cols with pitch ld0.
__global__ void __launch_bounds__(256)
rowsumsq_partial_kernel(const double *__restrict__ Xp, int I0, int ld0, long long cols, double *__restrict__ partial) {
  extern __shared__ double sh[]; // 256 doubles
  const int rpp = min(256, (I0 + 31) / 32 * 32); // rows per pass
  const int lanes = 256 / rpp;                   // column lanes
  const int r = threadIdx.x % rpp, cl = threadIdx.x / rpp;
  const long long per = (cols + gridDim.x - 1) / gridDim.x;
  const long long j0 = per * blockIdx.x, j1 = min(cols, j0 + per);
  for (int rb = 0; rb < I0; rb += rpp) {
    const int i = rb + r;
    double acc = 0.0;
    if (i < I0 && cl < lanes)
      for (long long j = j0 + cl; j < j1; j += lanes) {
        const double v = Xp[j * ld0 + i];
        acc += v * v;
      }
    __syncthreads();
    sh[threadIdx.x] = acc;
    __syncthreads();
    if (cl == 0 && i < I0) {
      double s = 0.0;
      for (int l = 0; l < lanes; l++)
        s += sh[l * rpp + r];
      partial[(long long)blockIdx.x * I0 + i] = s;
    }
  }
}

// rowsum[i] = sum_cta partial[cta][i] (fixed order); out[0] = ||X||, jk[i] = sqrt(total - rowsum[i]).  One CTA.
__global__ void __launch_bounds__(256)
rowsumsq_final_kernel(const double *__restrict__ partial, int n_ctas, int I0, double *__restrict__ jk,
                      double *__restrict__ out_norm) {
  __shared__ double sh[256];
  double local = 0.0;
  for (int i = threadIdx.x; i < I0; i += 256) {
    double s = 0.0;
    for (int c = 0; c < n_ctas; c++)
      s += partial[(long long)c * I0 + i];
    jk[i] = s;
    local += s;
  }
  sh[threadIdx.x] = local;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o)
      sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  const double total = sh[0];
  for (int i = threadIdx.x; i < I0; i += 256)
    jk[i] = sqrt(total - jk[i]);
  if (threadIdx.x == 0)
    out_norm[0] = sqrt(total);
}

} // namespace calsb200
