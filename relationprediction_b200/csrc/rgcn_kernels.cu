// rgcn_kernels.cu -- sm_100a kernels of the R-GCN relational message-passing hot path.
//
// Design (see DESIGN.md): every kernel is WARP-CENTRIC.  A warp owns one work item = a run of at
// most `item_max` messages of ONE row of a sorted message list (graph.cu).  A lane owns NV float4
// "quads" of the feature row (columns c0 + 4*(lane + 32k)), so one message = NV coalesced 128-bit
// loads per lane (a 2000/2048-byte row is 4 LDG.128 per lane), U messages are kept in flight per
// lane, and all reductions over messages happen in registers: no atomics per message, none at all
// for rows that fit one item.  Rows cut into several items combine their partial sums with vector
// reductions (red.global.add.v4.f32) into an L2-resident scratch row; the last arriver applies the
// epilogue.
//
// Block-diagonal trick: messages of a row are sorted by weight id, and blockdiag(W_r) is linear, so
// for a run of messages with the same (row, weight id) we first sum norm_m * x_m and apply W_r
// ONCE per run (FB15k-237: 544k messages -> 150k runs).  The weight tables are re-laid out per
// call into [w][j][d] ("j-major") so the per-run weight read is s*NV coalesced 128-bit loads that
// hit L2/L1, and the per-edge [E,B,s,s] weight gather of the reference
// (gcn_basis_concat.py:38-39) is never materialised.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>

#include "kernels.cuh"

int64_t g_rgcn_launches = 0;

#define FULL 0xffffffffu

namespace {

constexpr int U_MSG = 4;  // messages in flight per lane

__device__ __forceinline__ float4 ldg4(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}
__device__ __forceinline__ float4 ldcg4(const float* p) {
  return __ldcg(reinterpret_cast<const float4*>(p));
}
__device__ __forceinline__ void red4(float* p, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w)
               : "memory");
}
__device__ __forceinline__ void red1(float* p, float v) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
__device__ __forceinline__ void fma4(float4& a, float s, const float4& x) {
  a.x = fmaf(s, x.x, a.x);
  a.y = fmaf(s, x.y, a.y);
  a.z = fmaf(s, x.z, a.z);
  a.w = fmaf(s, x.w, a.w);
}
__device__ __forceinline__ float4 zero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}
template <int S>
__device__ __forceinline__ int blk_base(int col, int s_rt) {
  if constexpr (S > 0) return (col / S) * S;
  return (col / s_rt) * s_rt;
}

// ------------------------------------------------------------------------------------------------
// Block-diagonal aggregation.
// ------------------------------------------------------------------------------------------------
template <int S, int NV>
__device__ __forceinline__ void block_apply(float4 (&acc)[NV], const float4 (&xs)[NV], float* xbuf,
                                            const float* __restrict__ wr, int d, int s, int c0,
                                            int lane, const int (&xo)[NV][4]) {
  __syncwarp();
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int lc = 4 * (lane + 32 * k);
    if (c0 + lc < d) *reinterpret_cast<float4*>(xbuf + lc) = xs[k];
  }
  __syncwarp();
  auto body = [&](int j) {
    const float* wj = wr + (size_t)j * d;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int col = c0 + 4 * (lane + 32 * k);
      if (col < d) {
        const float4 w = ldg4(wj + col);
        if (S > 0 && S % 4 == 0) {
          const float x = xbuf[xo[k][0] + j];
          acc[k].x = fmaf(w.x, x, acc[k].x);
          acc[k].y = fmaf(w.y, x, acc[k].y);
          acc[k].z = fmaf(w.z, x, acc[k].z);
          acc[k].w = fmaf(w.w, x, acc[k].w);
        } else {
          acc[k].x = fmaf(w.x, xbuf[xo[k][0] + j], acc[k].x);
          acc[k].y = fmaf(w.y, xbuf[xo[k][1] + j], acc[k].y);
          acc[k].z = fmaf(w.z, xbuf[xo[k][2] + j], acc[k].z);
          acc[k].w = fmaf(w.w, xbuf[xo[k][3] + j], acc[k].w);
        }
      }
    }
  };
  if (S > 0) {
#pragma unroll
    for (int j = 0; j < (S > 0 ? S : 1); ++j) body(j);
  } else {
    for (int j = 0; j < s; ++j) body(j);
  }
}

template <int S, int NV>
__global__ void __launch_bounds__(RGCN_THREADS, 2)
    k_block_agg(AggLaunch a, int s_rt, const float* __restrict__ Wt, float* __restrict__ out,
                const uint8_t* __restrict__ mask, float inv_keep, int relu) {
  __shared__ __align__(16) float xbuf_all[RGCN_WARPS_PER_BLOCK][NV * 128];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * RGCN_WARPS_PER_BLOCK + warp;
  if (item >= a.n_items) return;
  const int s = S > 0 ? S : s_rt;
  const int d = a.d;
  const int c0 = blockIdx.y * (NV * 128);
  float* xbuf = xbuf_all[warp];
  const int4 itv = __ldg(reinterpret_cast<const int4*>(a.items) + item);
  const int beg = itv.x, end = itv.y, row = itv.z, split = itv.w;

  float4 acc[NV], xs[NV];
  int xo[NV][4];  // xbuf offset of the block each owned output column belongs to
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    acc[k] = xs[k] = zero4();
#pragma unroll
    for (int c = 0; c < 4; ++c) xo[k][c] = blk_base<S>(c0 + 4 * (lane + 32 * k) + c, s) - c0;
  }
  int cur = -1;

  for (int base = beg; base < end; base += 32) {
    const int n = min(32, end - base);
    int my_nbr = 0, my_rw = 0;
    float my_nm = 0.f;
    if (lane < n) {
      my_nbr = __ldg(a.nbr + base + lane);
      my_rw = __ldg(a.relw + base + lane);
      my_nm = __ldg(a.norm + base + lane);
    }
    for (int t = 0; t < n; t += U_MSG) {
      float4 x[U_MSG][NV];
      int rw[U_MSG];
      float nm[U_MSG];
#pragma unroll
      for (int u = 0; u < U_MSG; ++u) {
        const int tt = min(t + u, n - 1);  // tail: re-read the last row, weight forced to 0 below
        const int src = __shfl_sync(FULL, my_nbr, tt);
        rw[u] = __shfl_sync(FULL, my_rw, tt);
        nm[u] = __shfl_sync(FULL, my_nm, tt);
        const float* xr = a.X + (size_t)src * a.ldx + c0;
#pragma unroll
        for (int k = 0; k < NV; ++k) {
          const int lc = 4 * (lane + 32 * k);
          x[u][k] = (c0 + lc < d) ? ldg4(xr + lc) : zero4();
        }
      }
#pragma unroll
      for (int u = 0; u < U_MSG; ++u) {
        if (t + u < n) {
          if (rw[u] != cur) {
            if (cur >= 0)
              block_apply<S, NV>(acc, xs, xbuf, Wt + (size_t)cur * s * d, d, s, c0, lane, xo);
            cur = rw[u];
#pragma unroll
            for (int k = 0; k < NV; ++k) xs[k] = zero4();
          }
#pragma unroll
          for (int k = 0; k < NV; ++k) fma4(xs[k], nm[u], x[u][k]);
        }
      }
    }
  }
  if (cur >= 0) block_apply<S, NV>(acc, xs, xbuf, Wt + (size_t)cur * s * d, d, s, c0, lane, xo);

  // ---- epilogue ----
  bool do_epilogue = true;
  if (split >= 0) {
    float* sc = a.scratch + (size_t)split * d + c0;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int lc = 4 * (lane + 32 * k);
      if (c0 + lc < d) red4(sc + lc, acc[k]);
    }
    __threadfence();
    __syncwarp();
    int last = 0;
    if (lane == 0) {
      const int old = atomicAdd(a.counters + (size_t)split * gridDim.y + blockIdx.y, 1);
      last = (old == __ldg(a.split_nitems + split) - 1);
    }
    last = __shfl_sync(FULL, last, 0);
    do_epilogue = last != 0;
    if (do_epilogue) {
      __threadfence();
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        const int lc = 4 * (lane + 32 * k);
        if (c0 + lc < d) acc[k] = ldcg4(sc + lc);
      }
    }
  }
  if (do_epilogue) {
    float* po = out + (size_t)row * d + c0;
    const uint8_t* pm = mask ? mask + (size_t)row * d + c0 : nullptr;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int lc = 4 * (lane + 32 * k);
      if (c0 + lc < d) {
        float4 sl = *reinterpret_cast<const float4*>(po + lc);
        if (pm) {
          const uchar4 mk = *reinterpret_cast<const uchar4*>(pm + lc);
          sl.x = mk.x ? sl.x * inv_keep : 0.f;
          sl.y = mk.y ? sl.y * inv_keep : 0.f;
          sl.z = mk.z ? sl.z * inv_keep : 0.f;
          sl.w = mk.w ? sl.w * inv_keep : 0.f;
        }
        float4 r = make_float4(acc[k].x + sl.x, acc[k].y + sl.y, acc[k].z + sl.z, acc[k].w + sl.w);
        if (relu) {
          r.x = fmaxf(r.x, 0.f);
          r.y = fmaxf(r.y, 0.f);
          r.z = fmaxf(r.z, 0.f);
          r.w = fmaxf(r.w, 0.f);
        }
        *reinterpret_cast<float4*>(po + lc) = r;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Block-diagonal weight gradient (weight-id major list sorted by (weight id, dst)).
// Runs of messages with the same destination share G[dst]: sum norm*H[src] first, then ONE outer
// product per run.  Accumulators acc[JC][NV] live in registers; partial results of the items of one
// weight id are combined with vector reductions into dWt (zeroed by the caller).
// ------------------------------------------------------------------------------------------------
template <int S, int JC, int NV>
__global__ void __launch_bounds__(RGCN_THREADS, 1)
    k_block_dw(const WorkItem* __restrict__ items, int n_items, const int32_t* __restrict__ r_dst,
               const int32_t* __restrict__ r_src, const float* __restrict__ r_norm,
               const float* __restrict__ H, int ldh, const float* __restrict__ G, int ldg, int d,
               int s_rt, float* __restrict__ dWt) {
  __shared__ __align__(16) float xbuf_all[RGCN_WARPS_PER_BLOCK][NV * 128];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * RGCN_WARPS_PER_BLOCK + warp;
  if (item >= n_items) return;
  const int s = S > 0 ? S : s_rt;
  const int c0 = blockIdx.y * (NV * 128);
  float* xbuf = xbuf_all[warp];
  const int4 itv = __ldg(reinterpret_cast<const int4*>(items) + item);
  const int beg = itv.x, end = itv.y, w = itv.z;
  constexpr int U = 2;  // messages in flight per lane (each may also carry the G row of a new run)

  int xo[NV][4];
#pragma unroll
  for (int k = 0; k < NV; ++k)
#pragma unroll
    for (int c = 0; c < 4; ++c) xo[k][c] = blk_base<S>(c0 + 4 * (lane + 32 * k) + c, s) - c0;

  for (int j0 = 0; j0 < s; j0 += JC) {
    float4 acc[JC][NV], hs[NV], gcur[NV];
#pragma unroll
    for (int jj = 0; jj < JC; ++jj)
#pragma unroll
      for (int k = 0; k < NV; ++k) acc[jj][k] = zero4();
#pragma unroll
    for (int k = 0; k < NV; ++k) hs[k] = gcur[k] = zero4();
    int cur = -1;

    // one outer product per run: acc[j][cols] += G[run dst][cols] * (sum norm*H[src])[block(col) + j]
    auto flush = [&]() {
      __syncwarp();
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        const int lc = 4 * (lane + 32 * k);
        if (c0 + lc < d) *reinterpret_cast<float4*>(xbuf + lc) = hs[k];
      }
      __syncwarp();
#pragma unroll
      for (int jj = 0; jj < JC; ++jj) {
        const int j = j0 + jj;
        if (j < s) {
#pragma unroll
          for (int k = 0; k < NV; ++k) {
            if (c0 + 4 * (lane + 32 * k) < d) {
              if (S > 0 && S % 4 == 0) {
                fma4(acc[jj][k], xbuf[xo[k][0] + j], gcur[k]);
              } else {
                acc[jj][k].x = fmaf(gcur[k].x, xbuf[xo[k][0] + j], acc[jj][k].x);
                acc[jj][k].y = fmaf(gcur[k].y, xbuf[xo[k][1] + j], acc[jj][k].y);
                acc[jj][k].z = fmaf(gcur[k].z, xbuf[xo[k][2] + j], acc[jj][k].z);
                acc[jj][k].w = fmaf(gcur[k].w, xbuf[xo[k][3] + j], acc[jj][k].w);
              }
            }
          }
        }
      }
    };

    for (int base = beg; base < end; base += 32) {
      const int n = min(32, end - base);
      int my_dst = 0, my_src = 0;
      float my_nm = 0.f;
      if (lane < n) {
        my_dst = __ldg(r_dst + base + lane);
        my_src = __ldg(r_src + base + lane);
        my_nm = __ldg(r_norm + base + lane);
      }
      for (int t = 0; t < n; t += U) {
        float4 x[U][NV], gx[U][NV];
        int dv[U];
        float nm[U];
        bool starts[U];
        int prev = cur;
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int tt = min(t + u, n - 1);
          const int src = __shfl_sync(FULL, my_src, tt);
          dv[u] = __shfl_sync(FULL, my_dst, tt);
          nm[u] = __shfl_sync(FULL, my_nm, tt);
          starts[u] = (t + u < n) && (dv[u] != prev);  // warp-uniform
          prev = dv[u];
          const float* xr = H + (size_t)src * ldh + c0;
          const float* gr = G + (size_t)dv[u] * ldg + c0;
#pragma unroll
          for (int k = 0; k < NV; ++k) {
            const int lc = 4 * (lane + 32 * k);
            const bool ok = c0 + lc < d;
            x[u][k] = ok ? ldg4(xr + lc) : zero4();
            // the G row of a run is fetched together with the run's first H row (no dependent load)
            gx[u][k] = (ok && starts[u]) ? ldg4(gr + lc) : zero4();
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (t + u < n) {
            if (starts[u]) {
              if (cur >= 0) flush();
              cur = dv[u];
#pragma unroll
              for (int k = 0; k < NV; ++k) {
                hs[k] = zero4();
                gcur[k] = gx[u][k];
              }
            }
#pragma unroll
            for (int k = 0; k < NV; ++k) fma4(hs[k], nm[u], x[u][k]);
          }
        }
      }
    }
    if (cur >= 0) flush();

#pragma unroll
    for (int jj = 0; jj < JC; ++jj) {
      const int j = j0 + jj;
      if (j < s) {
        float* pw = dWt + ((size_t)w * s + j) * d + c0;
#pragma unroll
        for (int k = 0; k < NV; ++k) {
          const int lc = 4 * (lane + 32 * k);
          if (c0 + lc < d) red4(pw + lc, acc[jj][k]);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Block-diagonal aggregation, WEIGHT-ID MAJOR ("rel-major").  A warp owns <= item_max messages of
// ONE weight id (and one column slab): the block weights W_r live in REGISTERS for the whole item
// (loaded once, coalesced, from the j-major table), messages are walked in row order so runs with
// the same accumulation row are summed first (one transform per run), and each run's result is
// added to out[row] with a 128-bit vector reduction that resolves in L2 (the message list is sorted
// by L2-sized supertiles of rows, graph.cu).  Weight traffic drops from d*s*4 bytes per run to
// d*s*4 bytes per item; the price is a non-deterministic fp32 summation order across items.
// ------------------------------------------------------------------------------------------------
template <int S, int NV, bool FUSE_DW>
__global__ void __launch_bounds__(RGCN_THREADS, (FUSE_DW || S * NV > 16) ? 1 : (S * NV > 8 ? 2 : 3))
    k_block_rel(const WorkItem* __restrict__ items, int n_items, const int32_t* __restrict__ r_row,
                const int32_t* __restrict__ r_nbr, const float* __restrict__ r_norm,
                const float* __restrict__ X, int ldx, int d, const float* __restrict__ Wt,
                float* __restrict__ out, const float* __restrict__ Hrow, int ldh,
                float* __restrict__ dWt) {
  // FUSE_DW (backward pass only: X = G, rows = sources, Wt = the TRANSPOSED table): the same walk also
  // produces the block weight gradient.  With g = sum_run norm*G[dst] and h = H[row]:
  //   dH[row][b*s+j] += sum_i W[b][i][j] g[b*s+i]     (the transform: lane owns column b*s+j, reads g from smem)
  //   dW[b][i][j]    += g[b*s+i] * h[b*s+j]           (same g values from smem, h quad in registers)
  // so the gradient accumulates in the transposed-table layout dWt[w][i][b*s+j] with NO extra shared
  // memory traffic, and the separate dW pass (a second round of gathers) disappears.
  static_assert(S > 0, "rel-major kernel needs a compile-time block size");
  __shared__ __align__(16) float xbuf_all[RGCN_WARPS_PER_BLOCK][NV * 128];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * RGCN_WARPS_PER_BLOCK + warp;
  if (item >= n_items) return;
  const int c0 = blockIdx.y * (NV * 128);
  float* xbuf = xbuf_all[warp];
  const int4 itv = __ldg(reinterpret_cast<const int4*>(items) + item);
  const int beg = itv.x, end = itv.y, w = itv.z;

  // weights of this (weight id, slab) -> registers; x offsets of the lane's outputs -> registers
  float4 wreg[S][NV];
  float4 acc[FUSE_DW ? S : 1][NV];
  int xo[NV][4];
  const float* wr = Wt + (size_t)w * S * d;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int col = c0 + 4 * (lane + 32 * k);
#pragma unroll
    for (int j = 0; j < S; ++j) wreg[j][k] = (col < d) ? ldg4(wr + (size_t)j * d + col) : zero4();
#pragma unroll
    for (int j = 0; j < (FUSE_DW ? S : 1); ++j) acc[j][k] = zero4();
#pragma unroll
    for (int c = 0; c < 4; ++c) xo[k][c] = ((col + c) / S) * S - c0;
  }

  float4 xs[NV], hcur[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) xs[k] = hcur[k] = zero4();
  int cur = -1;

  auto flush = [&](int row) {
    __syncwarp();
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int lc = 4 * (lane + 32 * k);
      if (c0 + lc < d) *reinterpret_cast<float4*>(xbuf + lc) = xs[k];
    }
    __syncwarp();
    float* po = out + (size_t)row * d + c0;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int lc = 4 * (lane + 32 * k);
      if (c0 + lc < d) {
        float4 y = zero4();
#pragma unroll
        for (int j = 0; j < S; ++j) {
          if (S % 4 == 0) {
            const float xv = xbuf[xo[k][0] + j];
            fma4(y, xv, wreg[j][k]);
            if (FUSE_DW) fma4(acc[FUSE_DW ? j : 0][k], xv, hcur[k]);
          } else {
            const float x0 = xbuf[xo[k][0] + j], x1 = xbuf[xo[k][1] + j];
            const float x2 = xbuf[xo[k][2] + j], x3 = xbuf[xo[k][3] + j];
            y.x = fmaf(wreg[j][k].x, x0, y.x);
            y.y = fmaf(wreg[j][k].y, x1, y.y);
            y.z = fmaf(wreg[j][k].z, x2, y.z);
            y.w = fmaf(wreg[j][k].w, x3, y.w);
            if (FUSE_DW) {
              float4& a = acc[FUSE_DW ? j : 0][k];
              a.x = fmaf(x0, hcur[k].x, a.x);
              a.y = fmaf(x1, hcur[k].y, a.y);
              a.z = fmaf(x2, hcur[k].z, a.z);
              a.w = fmaf(x3, hcur[k].w, a.w);
            }
          }
        }
        red4(po + lc, y);
      }
    }
  };

  constexpr int U = 2;
  for (int base = beg; base < end; base += 32) {
    const int n = min(32, end - base);
    int my_row = 0, my_nbr = 0;
    float my_nm = 0.f;
    if (lane < n) {
      my_row = __ldg(r_row + base + lane);
      my_nbr = __ldg(r_nbr + base + lane);
      my_nm = __ldg(r_norm + base + lane);
    }
    for (int t = 0; t < n; t += U) {
      float4 x[U][NV], hx[FUSE_DW ? U : 1][NV];
      int rv[U];
      float nm[U];
      bool starts[U];
      int prev = cur;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int tt = min(t + u, n - 1);
        const int src = __shfl_sync(FULL, my_nbr, tt);
        rv[u] = __shfl_sync(FULL, my_row, tt);
        nm[u] = __shfl_sync(FULL, my_nm, tt);
        starts[u] = (t + u < n) && (rv[u] != prev);  // warp-uniform
        prev = rv[u];
        const float* xr = X + (size_t)src * ldx + c0;
#pragma unroll
        for (int k = 0; k < NV; ++k) {
          const int lc0 = 4 * (lane + 32 * k);
          const bool ok = c0 + lc0 < d;
          const int lc = lc0;
          x[u][k] = ok ? ldg4(xr + lc) : zero4();
          if (FUSE_DW)  // the run's own H row travels with the run's first gathered row
            hx[FUSE_DW ? u : 0][k] = (ok && starts[u]) ? ldg4(Hrow + (size_t)rv[u] * ldh + c0 + lc) : zero4();
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (t + u < n) {
          if (starts[u]) {
            if (cur >= 0) flush(cur);
            cur = rv[u];
#pragma unroll
            for (int k = 0; k < NV; ++k) {
              xs[k] = zero4();
              if (FUSE_DW) hcur[k] = hx[FUSE_DW ? u : 0][k];
            }
          }
#pragma unroll
          for (int k = 0; k < NV; ++k) fma4(xs[k], nm[u], x[u][k]);
        }
      }
    }
  }
  if (cur >= 0) flush(cur);
  if (FUSE_DW) {
#pragma unroll
    for (int j = 0; j < S; ++j) {
      float* pw = dWt + ((size_t)w * S + j) * d + c0;
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        const int lc = 4 * (lane + 32 * k);
        if (c0 + lc < d) red4(pw + lc, acc[FUSE_DW ? j : 0][k]);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Weight-id-major aggregation with G WARPS PER ITEM (block sizes that do not divide 128, i.e. s = 5).
// The G warps of a group walk the same messages; warp g owns the contiguous column range
// [g*512/G, (g+1)*512/G) of every row (so a 2000-byte row is 4 coalesced 500-byte pieces), which
// cuts the per-lane register state by G (weights, pre-sums, rows in flight) and lets 3 blocks =
// 24 warps live on an SM instead of 8.  Blocks of 5 straddle the column ranges, so the pre-summed
// row is exchanged through a double-buffered shared-memory row per group and ONE named barrier
// (bar.sync id, 32*G) per run.
// ------------------------------------------------------------------------------------------------
template <int S, int G, bool FUSE_DW>
__global__ void __launch_bounds__(RGCN_THREADS, FUSE_DW ? 2 : 3)
    k_block_relg(const WorkItem* __restrict__ items, int n_items, const int32_t* __restrict__ r_row,
                 const int32_t* __restrict__ r_nbr, const float* __restrict__ r_norm,
                 const float* __restrict__ X, int ldx, int d, const float* __restrict__ Wt,
                 float* __restrict__ out, const float* __restrict__ Hrow, int ldh,
                 float* __restrict__ dWt) {
  constexpr int NV = 4 / G;                       // quads per lane
  constexpr int GROUPS = RGCN_WARPS_PER_BLOCK / G;
  constexpr int U = FUSE_DW ? 2 : 4;              // rows in flight per lane
  __shared__ __align__(16) float xbuf_all[GROUPS][2][512];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gi = warp / G, g = warp % G;
  const int item = blockIdx.x * GROUPS + gi;
  if (item >= n_items) return;  // the whole group leaves together
  const int4 itv = __ldg(reinterpret_cast<const int4*>(items) + item);
  const int beg = itv.x, end = itv.y, w = itv.z;
  const int bar_id = 1 + gi;

  int colq[NV];  // first column of each owned quad
  float4 wreg[S][NV];
  float4 acc[FUSE_DW ? S : 1][NV];
  int xo[NV][4];
  const float* wr = Wt + (size_t)w * S * d;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    colq[k] = 4 * (g * 32 * NV + lane + 32 * k);
#pragma unroll
    for (int j = 0; j < S; ++j) wreg[j][k] = (colq[k] < d) ? ldg4(wr + (size_t)j * d + colq[k]) : zero4();
#pragma unroll
    for (int j = 0; j < (FUSE_DW ? S : 1); ++j) acc[j][k] = zero4();
#pragma unroll
    for (int c = 0; c < 4; ++c) xo[k][c] = ((colq[k] + c) / S) * S;
  }
  float4 xs[NV], hcur[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) xs[k] = hcur[k] = zero4();
  int cur = -1, par = 0;

  auto flush = [&](int row) {
    float* xb = xbuf_all[gi][par];
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      if (colq[k] < d) *reinterpret_cast<float4*>(xb + colq[k]) = xs[k];
    }
    asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(32 * G) : "memory");
    float* po = out + (size_t)row * d;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      if (colq[k] < d) {
        float4 y = zero4();
#pragma unroll
        for (int j = 0; j < S; ++j) {
          const float x0 = xb[xo[k][0] + j], x1 = xb[xo[k][1] + j];
          const float x2 = xb[xo[k][2] + j], x3 = xb[xo[k][3] + j];
          y.x = fmaf(wreg[j][k].x, x0, y.x);
          y.y = fmaf(wreg[j][k].y, x1, y.y);
          y.z = fmaf(wreg[j][k].z, x2, y.z);
          y.w = fmaf(wreg[j][k].w, x3, y.w);
          if (FUSE_DW) {  // dW[b][i=j][.] += g[b*s+i] * h[col]: same smem values, h quad in registers
            float4& a = acc[FUSE_DW ? j : 0][k];
            a.x = fmaf(x0, hcur[k].x, a.x);
            a.y = fmaf(x1, hcur[k].y, a.y);
            a.z = fmaf(x2, hcur[k].z, a.z);
            a.w = fmaf(x3, hcur[k].w, a.w);
          }
        }
        red4(po + colq[k], y);
      }
    }
    par ^= 1;
  };

  for (int base = beg; base < end; base += 32) {
    const int n = min(32, end - base);
    int my_row = 0, my_nbr = 0;
    float my_nm = 0.f;
    if (lane < n) {
      my_row = __ldg(r_row + base + lane);
      my_nbr = __ldg(r_nbr + base + lane);
      my_nm = __ldg(r_norm + base + lane);
    }
    for (int t = 0; t < n; t += U) {
      float4 x[U][NV], hx[FUSE_DW ? U : 1][NV];
      int rv[U];
      float nm[U];
      bool starts[U];
      int prev = cur;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int tt = min(t + u, n - 1);
        const int src = __shfl_sync(FULL, my_nbr, tt);
        rv[u] = __shfl_sync(FULL, my_row, tt);
        nm[u] = __shfl_sync(FULL, my_nm, tt);
        starts[u] = (t + u < n) && (rv[u] != prev);
        prev = rv[u];
        const float* xr = X + (size_t)src * ldx;
#pragma unroll
        for (int k = 0; k < NV; ++k) {
          const bool ok = colq[k] < d;
          const int cq = colq[k];
          x[u][k] = ok ? ldg4(xr + cq) : zero4();
          if (FUSE_DW)
            hx[FUSE_DW ? u : 0][k] = (ok && starts[u]) ? ldg4(Hrow + (size_t)rv[u] * ldh + cq) : zero4();
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (t + u < n) {
          if (starts[u]) {
            if (cur >= 0) flush(cur);
            cur = rv[u];
#pragma unroll
            for (int k = 0; k < NV; ++k) {
              xs[k] = zero4();
              if (FUSE_DW) hcur[k] = hx[FUSE_DW ? u : 0][k];
            }
          }
#pragma unroll
          for (int k = 0; k < NV; ++k) fma4(xs[k], nm[u], x[u][k]);
        }
      }
    }
  }
  if (cur >= 0) flush(cur);
  if (FUSE_DW) {
#pragma unroll
    for (int j = 0; j < S; ++j) {
      float* pw = dWt + ((size_t)w * S + j) * d;
#pragma unroll
      for (int k = 0; k < NV; ++k)
        if (colq[k] < d) red4(pw + colq[k], acc[FUSE_DW ? j : 0][k]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Weight-table re-layouts (tiny, L2-resident).
// ------------------------------------------------------------------------------------------------
__global__ void k_block_relayout(const float* __restrict__ Wf, const float* __restrict__ Wb, int R,
                                 int B, int s, int transpose, float* __restrict__ Wt) {
  const int d = B * s;
  const int64_t per = (int64_t)d * s;
  const int64_t total = 2 * (int64_t)R * per;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    // destination index: [w][q][col]   with col = b*s + p
    const int w = (int)(idx / per);
    const int rem = (int)(idx % per);
    const int q = rem / d;
    const int col = rem % d;
    const int b = col / s, p = col % s;
    // forward  (transpose=0): Wt[w][j=q][b*s+i=p] = W[b][i=p][j=q]
    // backward (transpose=1): Wt[w][i=q][b*s+j=p] = W[b][i=q][j=p]
    const int i = transpose ? q : p;
    const int j = transpose ? p : q;
    const float* W = (w < R) ? Wf + (size_t)w * per : Wb + (size_t)(w - R) * per;
    Wt[idx] = __ldg(W + ((size_t)b * s + i) * s + j);
  }
}

// table_t = 0: dWt is j-major (dWt[w][j][b*s+i]); table_t = 1: i-major (dWt[w][i][b*s+j], fused kernels)
__global__ void k_block_unlayout(const float* __restrict__ dWt, int R, int B, int s,
                                 float* __restrict__ dWf, float* __restrict__ dWb, int accumulate,
                                 int table_t) {
  const int d = B * s;
  const int64_t per = (int64_t)d * s;
  const int64_t total = 2 * (int64_t)R * per;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    // destination index: [w][b][i][j]
    const int w = (int)(idx / per);
    const int rem = (int)(idx % per);
    const int b = rem / (s * s);
    const int i = (rem / s) % s;
    const int j = rem % s;
    const float v = table_t ? __ldg(dWt + ((size_t)w * s + i) * d + b * s + j)
                            : __ldg(dWt + ((size_t)w * s + j) * d + b * s + i);
    float* p = (w < R) ? dWf + (size_t)w * per + rem : dWb + (size_t)(w - R) * per + rem;
    *p = accumulate ? *p + v : v;
  }
}

// ------------------------------------------------------------------------------------------------
// Basis aggregation:  Agg[row][dir][k,b] = sum_m norm_m * C[relw_m, b] * X[nbr_m, k]
// ------------------------------------------------------------------------------------------------
template <int BC, int NV, int LAYOUT>
__global__ void __launch_bounds__(RGCN_THREADS, 1)
    k_basis_agg(AggLaunch a, const float* __restrict__ C, int B, int half, float* __restrict__ Agg) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * RGCN_WARPS_PER_BLOCK + warp;
  if (item >= a.n_items) return;
  const int d = a.d;
  const int c0 = blockIdx.y * (NV * 128);
  const int4 itv = __ldg(reinterpret_cast<const int4*>(a.items) + item);
  const int beg = itv.x, end = itv.y, row = itv.z, split = itv.w;
  const size_t dB = (size_t)d * B;
  float* arow = Agg + (size_t)row * 2 * dB;

  for (int b0 = 0; b0 < B; b0 += BC) {
    float4 acc[BC][NV], xs[NV];
#pragma unroll
    for (int b = 0; b < BC; ++b)
#pragma unroll
      for (int k = 0; k < NV; ++k) acc[b][k] = zero4();
#pragma unroll
    for (int k = 0; k < NV; ++k) xs[k] = zero4();
    int cur = -1, curdir = -1, written = 0;

    auto write_out = [&](int dir) {
      float* ad = arow + (size_t)dir * dB;
#pragma unroll
      for (int b = 0; b < BC; ++b) {
        if (b0 + b < B) {
#pragma unroll
          for (int k = 0; k < NV; ++k) {
            const int col = c0 + 4 * (lane + 32 * k);
            if (col < d) {
              if (LAYOUT == 1) {
                float* p = ad + (size_t)(b0 + b) * d + col;
                if (split >= 0)
                  red4(p, acc[b][k]);
                else
                  *reinterpret_cast<float4*>(p) = acc[b][k];
              } else {
                float* p = ad + (size_t)col * B + (b0 + b);
                if (split >= 0) {
                  red1(p, acc[b][k].x);
                  red1(p + B, acc[b][k].y);
                  red1(p + 2 * B, acc[b][k].z);
                  red1(p + 3 * B, acc[b][k].w);
                } else {
                  p[0] = acc[b][k].x;
                  p[B] = acc[b][k].y;
                  p[2 * B] = acc[b][k].z;
                  p[3 * B] = acc[b][k].w;
                }
              }
            }
          }
        }
      }
      written |= (1 << dir);
    };
    auto flush = [&](int w) {
      const int dir = (w >= half) ? 1 : 0;
      if (dir != curdir) {
        if (curdir >= 0) write_out(curdir);
#pragma unroll
        for (int b = 0; b < BC; ++b)
#pragma unroll
          for (int k = 0; k < NV; ++k) acc[b][k] = zero4();
        curdir = dir;
      }
#pragma unroll
      for (int b = 0; b < BC; ++b) {
        const float cb = (b0 + b < B) ? __ldg(C + (size_t)w * B + b0 + b) : 0.f;
#pragma unroll
        for (int k = 0; k < NV; ++k) fma4(acc[b][k], cb, xs[k]);
      }
    };

    for (int base = beg; base < end; base += 32) {
      const int n = min(32, end - base);
      int my_nbr = 0, my_rw = 0;
      float my_nm = 0.f;
      if (lane < n) {
        my_nbr = __ldg(a.nbr + base + lane);
        my_rw = __ldg(a.relw + base + lane);
        my_nm = __ldg(a.norm + base + lane);
      }
      for (int t = 0; t < n; t += U_MSG) {
        float4 x[U_MSG][NV];
        int rw[U_MSG];
        float nm[U_MSG];
#pragma unroll
        for (int u = 0; u < U_MSG; ++u) {
          const int tt = min(t + u, n - 1);
          const int src = __shfl_sync(FULL, my_nbr, tt);
          rw[u] = __shfl_sync(FULL, my_rw, tt);
          nm[u] = __shfl_sync(FULL, my_nm, tt);
          const float* xr = a.X + (size_t)src * a.ldx + c0;
#pragma unroll
          for (int k = 0; k < NV; ++k) {
            const int lc = 4 * (lane + 32 * k);
            x[u][k] = (c0 + lc < d) ? ldg4(xr + lc) : zero4();
          }
        }
#pragma unroll
        for (int u = 0; u < U_MSG; ++u) {
          if (t + u < n) {
            if (rw[u] != cur) {
              if (cur >= 0) flush(cur);
              cur = rw[u];
#pragma unroll
              for (int k = 0; k < NV; ++k) xs[k] = zero4();
            }
#pragma unroll
            for (int k = 0; k < NV; ++k) fma4(xs[k], nm[u], x[u][k]);
          }
        }
      }
    }
    if (cur >= 0) flush(cur);
    if (curdir >= 0) write_out(curdir);
    if (split < 0) {
      // directions that received no message: explicit zeros (Agg is not pre-zeroed for these rows)
#pragma unroll
      for (int b = 0; b < BC; ++b)
#pragma unroll
        for (int k = 0; k < NV; ++k) acc[b][k] = zero4();
      if (!(written & 1)) write_out(0);
      if (!(written & 2)) write_out(1);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Basis coefficient gradient.
// ------------------------------------------------------------------------------------------------
template <int BC, int NV>
__global__ void __launch_bounds__(RGCN_THREADS, 1)
    k_basis_dc(AggLaunch a, const float* __restrict__ dAgg, int B, int half, float* __restrict__ dC) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * RGCN_WARPS_PER_BLOCK + warp;
  if (item >= a.n_items) return;
  const int d = a.d;
  const int c0 = blockIdx.y * (NV * 128);
  const int4 itv = __ldg(reinterpret_cast<const int4*>(a.items) + item);
  const int beg = itv.x, end = itv.y, row = itv.z;
  if (beg == end) return;
  const size_t dB = (size_t)d * B;
  const float* drow = dAgg + (size_t)row * 2 * dB;

  for (int b0 = 0; b0 < B; b0 += BC) {
    float4 da[BC][NV], xs[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) xs[k] = zero4();
    int cur = -1, loaded = -1;

    auto flush = [&](int w) {
      const int dir = (w >= half) ? 1 : 0;
      if (dir != loaded) {
        const float* dd = drow + (size_t)dir * dB;
#pragma unroll
        for (int b = 0; b < BC; ++b)
#pragma unroll
          for (int k = 0; k < NV; ++k) {
            const int col = c0 + 4 * (lane + 32 * k);
            if (col < d && b0 + b < B) {
              const float* p = dd + (size_t)col * B + (b0 + b);
              da[b][k] = make_float4(__ldg(p), __ldg(p + B), __ldg(p + 2 * B), __ldg(p + 3 * B));
            } else {
              da[b][k] = zero4();
            }
          }
        loaded = dir;
      }
#pragma unroll
      for (int b = 0; b < BC; ++b) {
        float p = 0.f;
#pragma unroll
        for (int k = 0; k < NV; ++k) {
          p = fmaf(xs[k].x, da[b][k].x, p);
          p = fmaf(xs[k].y, da[b][k].y, p);
          p = fmaf(xs[k].z, da[b][k].z, p);
          p = fmaf(xs[k].w, da[b][k].w, p);
        }
        p = warp_sum(p);
        if (lane == 0 && b0 + b < B) atomicAdd(dC + (size_t)w * B + b0 + b, p);
      }
    };

    for (int base = beg; base < end; base += 32) {
      const int n = min(32, end - base);
      int my_nbr = 0, my_rw = 0;
      float my_nm = 0.f;
      if (lane < n) {
        my_nbr = __ldg(a.nbr + base + lane);
        my_rw = __ldg(a.relw + base + lane);
        my_nm = __ldg(a.norm + base + lane);
      }
      for (int t = 0; t < n; t += U_MSG) {
        float4 x[U_MSG][NV];
        int rw[U_MSG];
        float nm[U_MSG];
#pragma unroll
        for (int u = 0; u < U_MSG; ++u) {
          const int tt = min(t + u, n - 1);
          const int src = __shfl_sync(FULL, my_nbr, tt);
          rw[u] = __shfl_sync(FULL, my_rw, tt);
          nm[u] = __shfl_sync(FULL, my_nm, tt);
          const float* xr = a.X + (size_t)src * a.ldx + c0;
#pragma unroll
          for (int k = 0; k < NV; ++k) {
            const int lc = 4 * (lane + 32 * k);
            x[u][k] = (c0 + lc < d) ? ldg4(xr + lc) : zero4();
          }
        }
#pragma unroll
        for (int u = 0; u < U_MSG; ++u) {
          if (t + u < n) {
            if (rw[u] != cur) {
              if (cur >= 0) flush(cur);
              cur = rw[u];
#pragma unroll
              for (int k = 0; k < NV; ++k) xs[k] = zero4();
            }
#pragma unroll
            for (int k = 0; k < NV; ++k) fma4(xs[k], nm[u], x[u][k]);
          }
        }
      }
    }
    if (cur >= 0) flush(cur);
  }
}

// ------------------------------------------------------------------------------------------------
// Elementwise helpers.
// ------------------------------------------------------------------------------------------------
__global__ void k_grad_prologue(const float* __restrict__ dOut, const float* __restrict__ out,
                                const uint8_t* __restrict__ mask, float inv_keep, int relu,
                                int64_t n4, float* __restrict__ G, float* __restrict__ dS) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4;
       i += (int64_t)gridDim.x * blockDim.x) {
    float4 g = reinterpret_cast<const float4*>(dOut)[i];
    if (relu) {
      const float4 o = reinterpret_cast<const float4*>(out)[i];
      g.x = o.x > 0.f ? g.x : 0.f;
      g.y = o.y > 0.f ? g.y : 0.f;
      g.z = o.z > 0.f ? g.z : 0.f;
      g.w = o.w > 0.f ? g.w : 0.f;
    }
    reinterpret_cast<float4*>(G)[i] = g;
    if (mask) {
      const uchar4 mk = reinterpret_cast<const uchar4*>(mask)[i];
      float4 s;
      s.x = mk.x ? g.x * inv_keep : 0.f;
      s.y = mk.y ? g.y * inv_keep : 0.f;
      s.z = mk.z ? g.z * inv_keep : 0.f;
      s.w = mk.w ? g.w * inv_keep : 0.f;
      reinterpret_cast<float4*>(dS)[i] = s;
    }
  }
}

__global__ void k_mask_relu(float* __restrict__ x, const uint8_t* __restrict__ mask, float inv_keep,
                            int relu, int64_t n4) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4;
       i += (int64_t)gridDim.x * blockDim.x) {
    float4 v = reinterpret_cast<float4*>(x)[i];
    if (mask) {
      const uchar4 mk = reinterpret_cast<const uchar4*>(mask)[i];
      v.x = mk.x ? v.x * inv_keep : 0.f;
      v.y = mk.y ? v.y * inv_keep : 0.f;
      v.z = mk.z ? v.z * inv_keep : 0.f;
      v.w = mk.w ? v.w * inv_keep : 0.f;
    }
    if (relu) {
      v.x = fmaxf(v.x, 0.f);
      v.y = fmaxf(v.y, 0.f);
      v.z = fmaxf(v.z, 0.f);
      v.w = fmaxf(v.w, 0.f);
    }
    reinterpret_cast<float4*>(x)[i] = v;
  }
}

// dst[rows[i], :] += src[i, :]  for UNIQUE rows (no atomics): the halo-gradient return of the node-sharded path, one
// peer segment per call (a row receives at most one contribution per peer)
__global__ void __launch_bounds__(256)
    k_rows_add(float* __restrict__ dst, const int64_t* __restrict__ rows, const float* __restrict__ src, int64_t n,
               int d4) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t i = (int64_t)blockIdx.x * 8 + warp; i < n; i += (int64_t)gridDim.x * 8) {
    float4* pd = reinterpret_cast<float4*>(dst) + (size_t)__ldg(rows + i) * d4;
    const float4* ps = reinterpret_cast<const float4*>(src) + (size_t)i * d4;
    for (int k = lane; k < d4; k += 32) {
      const float4 a = __ldcs(ps + k);
      float4 b = pd[k];
      b.x += a.x;
      b.y += a.y;
      b.z += a.z;
      b.w += a.w;
      pd[k] = b;
    }
  }
}

// dst[i, :] = src[rows[i], :]: the halo PUSH of the node-sharded path.  `dst` is normally a peer GPU's halo buffer mapped
// into this address space (NVLink stores are posted: the kernel is bound by the local row gather and the link, not by
// store latency), so the rows go straight from H to their consumer without a packed send buffer and an all-to-all.
// Two rows per warp iteration keep 8 x 16 B loads in flight per lane; the grid is kept small on purpose (the caller
// passes max_ctas) so that the push overlaps the layer's local work instead of occupying every SM.
__global__ void __launch_bounds__(256)
    k_rows_gather(float4* __restrict__ dst, const float4* __restrict__ src, const int64_t* __restrict__ rows, int64_t n,
                  int d4) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t i = ((int64_t)blockIdx.x * 8 + warp) * 2; i < n; i += (int64_t)gridDim.x * 16) {
    const bool two = i + 1 < n;
    const float4* p0 = src + (size_t)__ldg(rows + i) * d4;
    const float4* p1 = src + (size_t)__ldg(rows + (two ? i + 1 : i)) * d4;
    float4* q0 = dst + (size_t)i * d4;
    float4* q1 = q0 + d4;
    int k = lane;
    for (; k + 96 < d4; k += 128) {
      const float4 a0 = __ldg(p0 + k), a1 = __ldg(p0 + k + 32), a2 = __ldg(p0 + k + 64), a3 = __ldg(p0 + k + 96);
      const float4 b0 = __ldg(p1 + k), b1 = __ldg(p1 + k + 32), b2 = __ldg(p1 + k + 64), b3 = __ldg(p1 + k + 96);
      q0[k] = a0, q0[k + 32] = a1, q0[k + 64] = a2, q0[k + 96] = a3;
      if (two) q1[k] = b0, q1[k + 32] = b1, q1[k + 64] = b2, q1[k + 96] = b3;
    }
    for (; k < d4; k += 32) {
      const float4 a = __ldg(p0 + k), b = __ldg(p1 + k);
      q0[k] = a;
      if (two) q1[k] = b;
    }
  }
}

__global__ void k_zero_rows(float* __restrict__ A, int64_t width4, const int32_t* __restrict__ rows,
                            int n_rows) {
  const int r = blockIdx.x;
  if (r >= n_rows) return;
  float4* p = reinterpret_cast<float4*>(A + (size_t)__ldg(rows + r) * width4 * 4);
  for (int64_t i = threadIdx.x; i < width4; i += blockDim.x) p[i] = zero4();
}

int grid_for(int64_t n, int threads) {
  int64_t b = (n + threads - 1) / threads;
  const int64_t cap = 148 * 16;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

int check_launch(const char* what) {
  ++g_rgcn_launches;
  return rgcn_check_cuda(cudaGetLastError(), what);
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// Launchers
// ------------------------------------------------------------------------------------------------
static int pick_nv(int d) {
  int nv = (d + 127) / 128;
  return nv > 4 ? 4 : nv;
}

template <int S>
static int launch_block_agg_s(const AggLaunch& a, int s, const float* Wt, float* out,
                              const uint8_t* mask, float inv_keep, int relu, cudaStream_t st) {
  const int nv = pick_nv(a.d);
  const int slabs = (a.d + nv * 128 - 1) / (nv * 128);
  dim3 grid((a.n_items + RGCN_WARPS_PER_BLOCK - 1) / RGCN_WARPS_PER_BLOCK, slabs);
  if (a.n_items == 0) return RGCN_OK;
  switch (nv) {
    case 1: k_block_agg<S, 1><<<grid, RGCN_THREADS, 0, st>>>(a, s, Wt, out, mask, inv_keep, relu); break;
    case 2: k_block_agg<S, 2><<<grid, RGCN_THREADS, 0, st>>>(a, s, Wt, out, mask, inv_keep, relu); break;
    case 3: k_block_agg<S, 3><<<grid, RGCN_THREADS, 0, st>>>(a, s, Wt, out, mask, inv_keep, relu); break;
    default: k_block_agg<S, 4><<<grid, RGCN_THREADS, 0, st>>>(a, s, Wt, out, mask, inv_keep, relu); break;
  }
  return check_launch("k_block_agg");
}

int launch_block_agg(const AggLaunch& a, int s, const float* Wt, float* out, const uint8_t* mask,
                     float inv_keep, int relu, cudaStream_t st) {
  const int nv = pick_nv(a.d);
  if (a.d > nv * 128 && (nv * 128) % s != 0) {
    rgcn_set_error("block layer: d > 512 needs a block size s that divides 512");
    return RGCN_ERR_INVALID;
  }
  switch (s) {
    case 4: return launch_block_agg_s<4>(a, s, Wt, out, mask, inv_keep, relu, st);
    case 5: return launch_block_agg_s<5>(a, s, Wt, out, mask, inv_keep, relu, st);
    case 8: return launch_block_agg_s<8>(a, s, Wt, out, mask, inv_keep, relu, st);
    case 16: return launch_block_agg_s<16>(a, s, Wt, out, mask, inv_keep, relu, st);
    default: return launch_block_agg_s<0>(a, s, Wt, out, mask, inv_keep, relu, st);
  }
}

template <int S, int JC, int NV>
static int launch_block_dw_t(const WorkItem* items, int n_items, const int32_t* r_dst,
                             const int32_t* r_src, const float* r_norm, const float* H, int ldh,
                             const float* G, int ldg, int d, int s, float* dWt, cudaStream_t st) {
  const int slabs = (d + NV * 128 - 1) / (NV * 128);
  if (slabs > 1 && (NV * 128) % s != 0) {
    rgcn_set_error("block layer backward: column slab not aligned to the block size");
    return RGCN_ERR_INVALID;
  }
  dim3 grid((n_items + RGCN_WARPS_PER_BLOCK - 1) / RGCN_WARPS_PER_BLOCK, slabs);
  k_block_dw<S, JC, NV><<<grid, RGCN_THREADS, 0, st>>>(items, n_items, r_dst, r_src, r_norm, H, ldh,
                                                        G, ldg, d, s, dWt);
  return check_launch("k_block_dw");
}

int launch_block_dw(const WorkItem* items, int n_items, const int32_t* r_dst, const int32_t* r_src,
                    const float* r_norm, const float* H, int ldh, const float* G, int ldg, int d,
                    int s, float* dWt, cudaStream_t st) {
  if (n_items == 0) return RGCN_OK;
#define DW(S_, JC_, NV_) \
  return launch_block_dw_t<S_, JC_, NV_>(items, n_items, r_dst, r_src, r_norm, H, ldh, G, ldg, d, s, dWt, st)
  const int nv = pick_nv(d);
  if (s == 5) {
    switch (nv) { case 1: DW(5, 5, 1); case 2: DW(5, 5, 2); case 3: DW(5, 5, 3); default: DW(5, 5, 4); }
  } else if (s == 4) {
    switch (nv) { case 1: DW(4, 4, 1); case 2: DW(4, 4, 2); case 3: DW(4, 4, 3); default: DW(4, 4, 4); }
  } else if (s == 8) {
    if (nv == 1) DW(8, 8, 1);
    DW(8, 8, 2);
  } else if (s == 16) {
    DW(16, 16, 1);
  } else {
    switch (nv) { case 1: DW(0, 4, 1); case 2: DW(0, 4, 2); case 3: DW(0, 4, 3); default: DW(0, 4, 4); }
  }
#undef DW
}


template <int S, int NV, bool FUSE>
static int launch_block_rel_t(const WorkItem* items, int n_items, const int32_t* r_row,
                              const int32_t* r_nbr, const float* r_norm, const float* X, int ldx,
                              int d, const float* Wt, float* out, const float* Hrow, int ldh,
                              float* dWt, cudaStream_t st) {
  const int slabs = (d + NV * 128 - 1) / (NV * 128);
  dim3 grid((n_items + RGCN_WARPS_PER_BLOCK - 1) / RGCN_WARPS_PER_BLOCK, slabs);
  k_block_rel<S, NV, FUSE><<<grid, RGCN_THREADS, 0, st>>>(items, n_items, r_row, r_nbr, r_norm, X, ldx,
                                                                 d, Wt, out, Hrow, ldh, dWt);
  return check_launch("k_block_rel");
}

bool block_rel_supported(int d, int s) {
  if (s == 5) return d <= 512;
  if (s == 4 || s == 8 || s == 16) return true;
  return false;
}

// s = 5: warps per group of the group kernel k_block_relg (4 by default; $RGCN_REL_GROUP = 2 | 4, any other value
// selects the one-warp kernel k_block_rel<5, NV, false>)
static int rel_group_s5() {
  int G = 4;
  if (const char* e = std::getenv("RGCN_REL_GROUP")) G = std::atoi(e);
  return G;
}

// the dW-fused variant keeps 2*s*NV float4 of weights + gradient accumulators in registers
bool block_rel_fuse_dw_supported(int d, int s) {
  if (s == 5) {  // group-kernel variant: dH+dW in one walk measured 0.62 ms vs 0.34 + 0.38 ms separate
    const char* e = std::getenv("RGCN_FUSE_DW_S5");
    const int G = rel_group_s5();
    return d <= 512 && !(e && std::atoi(e) == 0) && (G == 4 || G == 2);  // only the group kernel fuses dW
  }
  return s == 4 || s == 8 || s == 16;
}

int launch_block_rel(const WorkItem* items, int n_items, const int32_t* r_row, const int32_t* r_nbr,
                     const float* r_norm, const float* X, int ldx, int d, int s, const float* Wt,
                     float* out, const float* Hrow, int ldh, float* dWt, cudaStream_t st) {
  if (n_items == 0) return RGCN_OK;
  const bool fuse = dWt != nullptr;
  if (fuse && !block_rel_fuse_dw_supported(d, s)) {
    rgcn_set_error("rel-major block kernel: dW fusion unsupported for this block size / kernel choice");
    return RGCN_ERR_INVALID;
  }
  // the dW-fused variant doubles the per-lane register state: it runs with ONE quad per lane (4 column slabs at
  // d = 512; keeps two blocks per SM resident and measured fastest, 11.4 vs 12.6 ms/step, synthetic), the only
  // fused instantiation
#define RLF(S_) \
  return launch_block_rel_t<S_, 1, true>(items, n_items, r_row, r_nbr, r_norm, X, ldx, d, Wt, out, Hrow, ldh, dWt, st)
#define RLN(S_, NV_) \
  return launch_block_rel_t<S_, NV_, false>(items, n_items, r_row, r_nbr, r_norm, X, ldx, d, Wt, out, Hrow, ldh, dWt, st)
  int nv = pick_nv(d);
  if (const char* e = std::getenv("RGCN_REL_NV")) {  // tuning knob: quads per lane (column slabs = d/(128 nv))
    const int v = std::atoi(e);
    if (v >= 1 && v <= 4 && s != 5 && (v * 128) % s == 0) nv = std::min(nv, v);
  }
  if (s == 5) {
    const int G = rel_group_s5();
    if (G == 4 || G == 2) {
      const int groups = RGCN_WARPS_PER_BLOCK / G;
      dim3 grid((n_items + groups - 1) / groups);
      if (G == 4) {
        if (fuse)
          k_block_relg<5, 4, true><<<grid, RGCN_THREADS, 0, st>>>(items, n_items, r_row, r_nbr, r_norm, X, ldx, d, Wt, out, Hrow, ldh, dWt);
        else
          k_block_relg<5, 4, false><<<grid, RGCN_THREADS, 0, st>>>(items, n_items, r_row, r_nbr, r_norm, X, ldx, d, Wt, out, Hrow, ldh, dWt);
      } else {
        if (fuse)
          k_block_relg<5, 2, true><<<grid, RGCN_THREADS, 0, st>>>(items, n_items, r_row, r_nbr, r_norm, X, ldx, d, Wt, out, Hrow, ldh, dWt);
        else
          k_block_relg<5, 2, false><<<grid, RGCN_THREADS, 0, st>>>(items, n_items, r_row, r_nbr, r_norm, X, ldx, d, Wt, out, Hrow, ldh, dWt);
      }
      return check_launch("k_block_relg");
    }
    switch (nv) { case 1: RLN(5, 1); case 2: RLN(5, 2); case 3: RLN(5, 3); default: RLN(5, 4); }
  } else if (fuse) {
    if (s == 4) RLF(4);
    if (s == 8) RLF(8);
    RLF(16);
  } else if (s == 4) {
    switch (nv) { case 1: RLN(4, 1); case 2: RLN(4, 2); case 3: RLN(4, 3); default: RLN(4, 4); }
  } else if (s == 8) {
    if (nv == 1) RLN(8, 1);
    RLN(8, 2);
  } else if (s == 16) {
    RLN(16, 1);
  }
#undef RLF
#undef RLN
  rgcn_set_error("rel-major block kernel: unsupported block size");
  return RGCN_ERR_INVALID;
}

int launch_block_relayout(const float* Wf, const float* Wb, int R, int B, int s, int transpose,
                          float* Wt, cudaStream_t st) {
  const int64_t total = 2 * (int64_t)R * B * s * s;
  k_block_relayout<<<grid_for(total, 256), 256, 0, st>>>(Wf, Wb, R, B, s, transpose, Wt);
  return check_launch("k_block_relayout");
}

int launch_block_unlayout(const float* dWt, int R, int B, int s, float* dWf, float* dWb,
                          int accumulate, int table_t, cudaStream_t st) {
  const int64_t total = 2 * (int64_t)R * B * s * s;
  k_block_unlayout<<<grid_for(total, 256), 256, 0, st>>>(dWt, R, B, s, dWf, dWb, accumulate, table_t);
  return check_launch("k_block_unlayout");
}

template <int BC, int LAYOUT>
static int launch_basis_agg_t(const AggLaunch& a, const float* C, int B, int n_relw, float* Agg,
                              cudaStream_t st) {
  const int nv = pick_nv(a.d);
  const int slabs = (a.d + nv * 128 - 1) / (nv * 128);
  dim3 grid((a.n_items + RGCN_WARPS_PER_BLOCK - 1) / RGCN_WARPS_PER_BLOCK, slabs);
  const int half = n_relw / 2;
  switch (nv) {
    case 1: k_basis_agg<BC, 1, LAYOUT><<<grid, RGCN_THREADS, 0, st>>>(a, C, B, half, Agg); break;
    case 2: k_basis_agg<BC, 2, LAYOUT><<<grid, RGCN_THREADS, 0, st>>>(a, C, B, half, Agg); break;
    case 3: k_basis_agg<BC, 3, LAYOUT><<<grid, RGCN_THREADS, 0, st>>>(a, C, B, half, Agg); break;
    default: k_basis_agg<BC, 4, LAYOUT><<<grid, RGCN_THREADS, 0, st>>>(a, C, B, half, Agg); break;
  }
  return check_launch("k_basis_agg");
}

int launch_basis_agg(const AggLaunch& a, const float* C, int B, int n_relw, int layout, float* Agg,
                     cudaStream_t st) {
  if (a.n_items == 0) return RGCN_OK;
  // bases per pass: all of them when they fit the register budget, else passes of 4
  if (layout == 0) {
    if (B == 1) return launch_basis_agg_t<1, 0>(a, C, B, n_relw, Agg, st);
    if (B == 2) return launch_basis_agg_t<2, 0>(a, C, B, n_relw, Agg, st);
    if (B <= 4) return launch_basis_agg_t<4, 0>(a, C, B, n_relw, Agg, st);
    if (B == 5) return launch_basis_agg_t<5, 0>(a, C, B, n_relw, Agg, st);
    return launch_basis_agg_t<4, 0>(a, C, B, n_relw, Agg, st);
  } else {
    if (B == 1) return launch_basis_agg_t<1, 1>(a, C, B, n_relw, Agg, st);
    if (B == 2) return launch_basis_agg_t<2, 1>(a, C, B, n_relw, Agg, st);
    if (B <= 4) return launch_basis_agg_t<4, 1>(a, C, B, n_relw, Agg, st);
    if (B == 5) return launch_basis_agg_t<5, 1>(a, C, B, n_relw, Agg, st);
    return launch_basis_agg_t<4, 1>(a, C, B, n_relw, Agg, st);
  }
}

template <int BC>
static int launch_basis_dc_t(const AggLaunch& a, const float* dAgg, int B, int n_relw, float* dC,
                             cudaStream_t st) {
  const int nv = pick_nv(a.d);
  const int slabs = (a.d + nv * 128 - 1) / (nv * 128);
  dim3 grid((a.n_items + RGCN_WARPS_PER_BLOCK - 1) / RGCN_WARPS_PER_BLOCK, slabs);
  const int half = n_relw / 2;
  switch (nv) {
    case 1: k_basis_dc<BC, 1><<<grid, RGCN_THREADS, 0, st>>>(a, dAgg, B, half, dC); break;
    case 2: k_basis_dc<BC, 2><<<grid, RGCN_THREADS, 0, st>>>(a, dAgg, B, half, dC); break;
    case 3: k_basis_dc<BC, 3><<<grid, RGCN_THREADS, 0, st>>>(a, dAgg, B, half, dC); break;
    default: k_basis_dc<BC, 4><<<grid, RGCN_THREADS, 0, st>>>(a, dAgg, B, half, dC); break;
  }
  return check_launch("k_basis_dc");
}

int launch_basis_dc(const AggLaunch& a, const float* dAgg, int B, int n_relw, float* dC,
                    cudaStream_t st) {
  if (a.n_items == 0) return RGCN_OK;
  if (B == 1) return launch_basis_dc_t<1>(a, dAgg, B, n_relw, dC, st);
  if (B == 2) return launch_basis_dc_t<2>(a, dAgg, B, n_relw, dC, st);
  if (B == 5) return launch_basis_dc_t<5>(a, dAgg, B, n_relw, dC, st);
  return launch_basis_dc_t<4>(a, dAgg, B, n_relw, dC, st);
}

int launch_grad_prologue(const float* dOut, const float* out, const uint8_t* mask, float inv_keep,
                         int relu, int64_t n, float* G, float* dS, cudaStream_t st) {
  if (n == 0) return RGCN_OK;
  k_grad_prologue<<<grid_for(n / 4, 256), 256, 0, st>>>(dOut, out, mask, inv_keep, relu, n / 4, G, dS);
  return check_launch("k_grad_prologue");
}

int launch_mask_relu(float* x, const uint8_t* mask, float inv_keep, int relu, int64_t n,
                     cudaStream_t st) {
  if (n == 0 || (!mask && !relu)) return RGCN_OK;
  k_mask_relu<<<grid_for(n / 4, 256), 256, 0, st>>>(x, mask, inv_keep, relu, n / 4);
  return check_launch("k_mask_relu");
}

int launch_zero_rows(float* A, int64_t width, const int32_t* rows, int n_rows, cudaStream_t st) {
  if (n_rows == 0) return RGCN_OK;
  k_zero_rows<<<n_rows, 256, 0, st>>>(A, width / 4, rows, n_rows);
  return check_launch("k_zero_rows");
}

int launch_rows_gather(float* dst, const float* src, const int64_t* rows, int64_t n, int d, int max_ctas,
                       cudaStream_t st) {
  if (n == 0) return RGCN_OK;
  int64_t b = (n + 15) / 16;
  const int64_t cap = max_ctas > 0 ? max_ctas : 148 * 8;
  if (b > cap) b = cap;
  k_rows_gather<<<(int)b, 256, 0, st>>>(reinterpret_cast<float4*>(dst), reinterpret_cast<const float4*>(src), rows, n,
                                        d / 4);
  return check_launch("k_rows_gather");
}

int launch_rows_add(float* dst, const int64_t* rows, const float* src, int64_t n, int d, cudaStream_t st) {
  if (n == 0) return RGCN_OK;
  int64_t b = (n + 7) / 8;
  if (b > 148 * 16) b = 148 * 16;
  k_rows_add<<<(int)b, 256, 0, st>>>(dst, rows, src, n, d / 4);
  return check_launch("k_rows_add");
}
