// Shared device helpers for libswb200 (sm_100a).  No tensor cores anywhere: every kernel here is an
// elementwise / row-column reduction path (SURVEY.md §2.2), so the tools are warp shuffles,
// shared-memory staging and vectorised global accesses.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/swb200.h"

#define SWB_WARP 32
#define SWB_FULL 0xffffffffu

namespace swb {

// the first 16-byte boundary at or after p (shared-memory and scratch carve-ups)
__host__ __device__ __forceinline__ unsigned char *align16(unsigned char *p) {
  return reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(p) + 15) & ~uintptr_t(15));
}

// Piecewise-linear log through (base_b, logv_b): the reference's SOS2 model (shockwave.py:384-419)
// evaluated directly — for a concave maximise the LP picks adjacent breakpoints, so
// plog(u) == min_b(slope_b * (u - base_b) + logv_b) on [0,1].
struct Pwl {
  int B;
  double base[SWB_MAX_BASES];
  double logv[SWB_MAX_BASES];
  double slope[SWB_MAX_BASES];  // slope[b] of segment [base[b], base[b+1]], b < B-1
};

__device__ __forceinline__ double plog(const Pwl &P, double u) {
  u = fmax(u, 0.0);
  // exact at the last breakpoint (lambda_B = 1 in the reference's model): the fallback priorities
  // reach 1e21 and would turn the ~1e-17 residual of slope*(1-base)+logv into O(10) of objective
  if (u >= P.base[P.B - 1]) return P.logv[P.B - 1];
  int b = 0;
  for (int i = 1; i < P.B - 1; ++i) b = (u >= P.base[i]) ? i : b;
  return fma(P.slope[b], u - P.base[b], P.logv[b]);
}

// the breakpoints of a scenario and the slopes between them
__device__ __forceinline__ void make_pwl(Pwl &P, const swb_params &prm) {
  const int B = prm.nbases;
  P.B = B;
  for (int b = 0; b < B; ++b) { P.base[b] = prm.bases[b]; P.logv[b] = prm.logv[b]; }
  for (int b = 0; b + 1 < B; ++b)
    P.slope[b] = (prm.logv[b + 1] - prm.logv[b]) / (prm.bases[b + 1] - prm.bases[b]);
}

// utility u of a job after n rounds: u0 + a n, or exactly 1 once the job completes inside the window (the fallback
// priorities reach 1e20 and would amplify a 1-ulp error in u to O(1))
__device__ __forceinline__ double util_u(double a, double u0, double cap, double D, int n) {
  return (D * (double)n >= cap) ? 1.0 : fma(a, (double)n, u0);
}

// unsigned key that sorts like the double it is made from (ascending)
__device__ __forceinline__ unsigned long long order_key(double v) {
  unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}

__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(SWB_FULL, v, o);
  return v;
}
__device__ __forceinline__ long long warp_sum(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(SWB_FULL, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(SWB_FULL, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(SWB_FULL, v, o));
  return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(SWB_FULL, v, o));
  return v;
}

// exclusive block scan of one int per thread; returns the exclusive prefix, total in *tot.
// wsum needs 33 ints.  Two barriers; the 32 warp totals are scanned by warp 0 with shuffles.
__device__ __forceinline__ int block_excl_scan(int v, int *wsum, int *tot) {
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(SWB_FULL, incl, o);
    if ((threadIdx.x & 31) >= o) incl += t;
  }
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();  // protect wsum from the previous use
  if (lane == 31) wsum[w] = incl;
  __syncthreads();
  // every warp scans the (<= 32) warp totals redundantly: no third barrier
  int ws = lane < nw ? wsum[lane] : 0;
  int wincl = ws;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(SWB_FULL, wincl, o);
    if (lane >= o) wincl += t;
  }
  *tot = __shfl_sync(SWB_FULL, wincl, 31);
  const int off = __shfl_sync(SWB_FULL, wincl - ws, w);
  return off + incl - v;
}

// Block reductions with ONE __syncthreads each: two scratch rows used alternately (ping-pong), so
// a warp that races ahead into reduction k+1 writes the other row and cannot reach reduction k+2
// before every warp has left reduction k.  `scratch` is 2 x 32 x 16 bytes.
struct BlockRed {
  double *s;       // [2][32][2]
  int phase;
  __device__ __forceinline__ BlockRed(double *scratch) : s(scratch), phase(0) {}

  // (sum of a, sum of b) over the block, both double
  __device__ __forceinline__ void sum2(double &a, double &b) {
    a = warp_sum(a);
    b = warp_sum(b);
    double *row = s + phase * 64;
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    if (l == 0) { row[2 * w] = a; row[2 * w + 1] = b; }
    __syncthreads();
    double ra = (l < nw) ? row[2 * l] : 0.0, rb = (l < nw) ? row[2 * l + 1] : 0.0;
    a = warp_sum(ra);
    b = warp_sum(rb);
    phase ^= 1;
  }
  __device__ __forceinline__ double sum(double a) { double b = 0.0; sum2(a, b); return a; }
  __device__ __forceinline__ long long sumll(long long a) {
    a = warp_sum(a);
    long long *row = reinterpret_cast<long long *>(s + phase * 64);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    if (l == 0) row[w] = a;
    __syncthreads();
    long long r = (l < nw) ? row[l] : 0;
    a = warp_sum(r);
    phase ^= 1;
    return a;
  }
  // int32 sum on the hardware warp reduction (REDUX.SUM): two instructions and one barrier instead of twenty
  // 32-bit shuffles — the demand sums of the price search are evaluated hundreds of times per solve
  __device__ __forceinline__ int sumi(int a) {
    a = __reduce_add_sync(SWB_FULL, a);
    int *row = reinterpret_cast<int *>(s + phase * 64);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    if (l == 0) row[w] = a;
    __syncthreads();
    a = __reduce_add_sync(SWB_FULL, (l < nw) ? row[l] : 0);
    phase ^= 1;
    return a;
  }
  // three int32 sums with ONE barrier (the price search evaluates three candidate prices per pass)
  __device__ __forceinline__ void sumi3(int &a, int &b, int &c) {
    a = __reduce_add_sync(SWB_FULL, a); b = __reduce_add_sync(SWB_FULL, b); c = __reduce_add_sync(SWB_FULL, c);
    int *row = reinterpret_cast<int *>(s + phase * 64);       // 128 ints per row: [32 warps][3]
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    if (l == 0) { row[3 * w] = a; row[3 * w + 1] = b; row[3 * w + 2] = c; }
    __syncthreads();
    a = __reduce_add_sync(SWB_FULL, (l < nw) ? row[3 * l] : 0);
    b = __reduce_add_sync(SWB_FULL, (l < nw) ? row[3 * l + 1] : 0);
    c = __reduce_add_sync(SWB_FULL, (l < nw) ? row[3 * l + 2] : 0);
    phase ^= 1;
  }
  __device__ __forceinline__ double max(double a) {
    a = warp_max(a);
    double *row = s + phase * 64;
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    if (l == 0) row[w] = a;
    __syncthreads();
    double r = (l < nw) ? row[l] : -1.0e300;
    a = warp_max(r);
    phase ^= 1;
    return a;
  }
  __device__ __forceinline__ double min(double a) { return -max(-a); }
};

}  // namespace swb
