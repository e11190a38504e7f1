// K5 / K6: robust-aggregation baselines on the PS GPU, per parameter tensor.
//
// Geometric median -- reference: `hd.geomedian(np.array(grads), axis=0)` per tensor (hdmedians' Cython
// Weiszfeld loop; src/master/baseline_master.py:271-276).  Here one streaming kernel per Weiszfeld
// iteration: with weights w_i = 1/||g_i - m|| from the previous iteration it forms m_new = sum w_i g_i /
// sum w_i element-wise *and in the same pass* accumulates ||g_i - m_new||^2 for the next iteration plus
// ||m_new - m||^2 for the stopping rule, so every iteration reads the P x D slab exactly once.  A tiny
// `geomed_prep_kernel` turns the accumulated distances into weights and freezes converged tensors.
//
// The product path does better than one pass per iteration: every Weiszfeld iterate is a convex combination
// m = sum_j w_j g_j of the inputs, and for such a point
//     ||g_i - m||^2 = sum_j w_j D_ij - 1/2 sum_jk w_j w_k D_jk          (D_ij = ||g_i - g_j||^2),
// so the whole iteration lives in the P-dimensional weight space once the P(P-1)/2 pairwise distances are known.
// `pair_dist_kernel` (shared with Krum) reads the slab ONCE, `geomed_weights_kernel` iterates to convergence on one
// warp per tensor in fp64, and the weighted combination is formed inside the fused SGD + broadcast kernel
// (aggregate_update MODE 2): two passes over the P x D slab instead of one per iteration.  The streaming
// per-iteration kernels below remain for P > 16.
//
// Krum -- reference: double Python loop of np.linalg.norm per tensor (baseline_master.py:278-296).  Here one
// pass produces all P(P-1)/2 squared distances per tensor, a one-thread-per-tensor kernel scores and selects,
// and the winner row goes through the fused select + SGD + broadcast kernel.
//
// Multi-Krum (Blanchard et al., NeurIPS 2017) shares the distances and the scores: the selection keeps the m rows
// with the lowest scores (ties to the lower slot), and the fused kernel averages them with its select-sum (MODE 0),
// which reads only the selected rows.  m = 1 is Krum.
#include "common.cuh"

#define GM_MAXP DRC_MAX_WORKERS

struct GeoMedArgs {
  const float* grad_in;           // [P][slot_stride]
  long long slot_stride;
  int P;
  TileView tv;
  float* median;                  // [D] current estimate m (in/out)
  const float* weights;           // [T][P]  normalised weights for this iteration
  const int* done;                // [T] tensor converged -> skip
  double* dist2;                  // [T][P] out: ||g_i - m_new||^2 (zero on entry)
  double* move2;                  // [T][2] out: ||m_new - m||^2, ||m_new||^2 (zero on entry)
};

__global__ void __launch_bounds__(DRC_THREADS) geomed_iter_kernel(const __grid_constant__ GeoMedArgs a) {
  __shared__ double s_red[DRC_THREADS / 32];
  for (int tile = blockIdx.x; tile < a.tv.ntiles; tile += gridDim.x) {
    int tensor;
    const int valid = tile_valid(a.tv, tile, tensor);
    if (a.done[tensor]) continue;
    const long long idx = (long long)tile * DRC_TILE + threadIdx.x * 4;
    const bool active = (int)threadIdx.x * 4 < valid;
    float4 m_new = make_float4(0.f, 0.f, 0.f, 0.f), m_old = m_new;
    if (active) {
      m_old = *reinterpret_cast<const float4*>(a.median + idx);
      for (int i = 0; i < a.P; ++i) {
        const float w = a.weights[tensor * a.P + i];
        float4 v = ld_f4(reinterpret_cast<const float4*>(a.grad_in + i * a.slot_stride + idx));
        m_new.x = fmaf(w, v.x, m_new.x); m_new.y = fmaf(w, v.y, m_new.y);
        m_new.z = fmaf(w, v.z, m_new.z); m_new.w = fmaf(w, v.w, m_new.w);
      }
      *reinterpret_cast<float4*>(a.median + idx) = m_new;
    }
    // distances to the new estimate (second read of the slab hits L1/L2: same tile, same CTA)
    for (int i = 0; i <= a.P; ++i) {
      double acc = 0.0;
      if (active) {
        float4 v = (i < a.P) ? ld_f4(reinterpret_cast<const float4*>(a.grad_in + i * a.slot_stride + idx)) : m_old;
        float dx = v.x - m_new.x, dy = v.y - m_new.y, dz = v.z - m_new.z, dw = v.w - m_new.w;
        acc = (double)dx * dx + (double)dy * dy + (double)dz * dz + (double)dw * dw;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = acc;
      __syncthreads();
      if (threadIdx.x == 0) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < DRC_THREADS / 32; ++w) s += s_red[w];
        if (i < a.P) atomicAdd(&a.dist2[tensor * a.P + i], s);
        else atomicAdd(&a.move2[tensor * 2], s);
      }
      __syncthreads();
    }
    {
      double acc = active ? (double)m_new.x * m_new.x + (double)m_new.y * m_new.y + (double)m_new.z * m_new.z +
                                (double)m_new.w * m_new.w : 0.0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = acc;
      __syncthreads();
      if (threadIdx.x == 0) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < DRC_THREADS / 32; ++w) s += s_red[w];
        atomicAdd(&a.move2[tensor * 2 + 1], s);
      }
      __syncthreads();
    }
  }
}

struct GeoMedPrepArgs {
  int T, P;
  double* dist2;                  // [T][P] consumed and zeroed
  double* move2;                  // [T][2] consumed and zeroed
  float* weights;                 // [T][P] out
  int* done;                      // [T] in/out
  int iter;                       // 0: initialise (weights = 1/P -> first estimate is the mean)
  double eps;                     // relative stopping tolerance
};

__global__ void geomed_prep_kernel(const __grid_constant__ GeoMedPrepArgs a) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= a.T) return;
  if (a.iter == 0) {
    for (int i = 0; i < a.P; ++i) { a.weights[t * a.P + i] = 1.0f / a.P; a.dist2[t * a.P + i] = 0.0; }
    a.move2[t * 2] = a.move2[t * 2 + 1] = 0.0;
    a.done[t] = 0;
    return;
  }
  if (a.done[t]) return;
  const double mv = a.move2[t * 2], nm = a.move2[t * 2 + 1];
  if (a.iter > 1 && sqrt(mv) <= a.eps * fmax(1.0, sqrt(nm))) a.done[t] = 1;
  double w[GM_MAXP], sum = 0.0;
  bool all_zero = true;
  for (int i = 0; i < a.P; ++i) {
    double d = sqrt(a.dist2[t * a.P + i]);
    w[i] = d > 1e-300 ? 1.0 / d : 0.0;
    all_zero &= !(d > 1e-300);
    sum += w[i];
    a.dist2[t * a.P + i] = 0.0;
  }
  a.move2[t * 2] = a.move2[t * 2 + 1] = 0.0;
  if (all_zero) { a.done[t] = 1; return; }
  for (int i = 0; i < a.P; ++i) a.weights[t * a.P + i] = (float)(w[i] / sum);
}

extern "C" int drc_geomed_iter(const GeoMedArgs* args, int grid, cudaStream_t stream) {
  geomed_iter_kernel<<<grid, DRC_THREADS, 0, stream>>>(*args);
  return (int)cudaGetLastError();
}
extern "C" int drc_geomed_prep(const GeoMedPrepArgs* args, cudaStream_t stream) {
  if (args->P > GM_MAXP) return (int)cudaErrorInvalidValue;
  geomed_prep_kernel<<<(args->T + 63) / 64, 64, 0, stream>>>(*args);
  return (int)cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Krum
// ---------------------------------------------------------------------------------------------
#define KRUM_MAXP 16
#define KRUM_MAXPAIRS (KRUM_MAXP * (KRUM_MAXP - 1) / 2)

struct PairDistArgs {
  const float* grad_in;
  long long slot_stride;
  int P;
  TileView tv;
  double* pair_d2;                // [T][P*(P-1)/2] zero on entry; pair (i<j) at j*(j-1)/2 + i
};

__global__ void __launch_bounds__(DRC_THREADS) pair_dist_kernel(const __grid_constant__ PairDistArgs a) {
  __shared__ double s_acc[KRUM_MAXPAIRS];
  const int npairs = a.P * (a.P - 1) / 2;
  for (int tile = blockIdx.x; tile < a.tv.ntiles; tile += gridDim.x) {
    int tensor;
    const int valid = tile_valid(a.tv, tile, tensor);
    for (int q = threadIdx.x; q < npairs; q += DRC_THREADS) s_acc[q] = 0.0;
    __syncthreads();
    const long long idx = (long long)tile * DRC_TILE + threadIdx.x * 4;
    const bool active = (int)threadIdx.x * 4 < valid;
    float4 v[KRUM_MAXP];
#pragma unroll
    for (int i = 0; i < KRUM_MAXP; ++i)
      if (i < a.P && active) v[i] = ld_f4(reinterpret_cast<const float4*>(a.grad_in + i * a.slot_stride + idx));
#pragma unroll
    for (int j = 1; j < KRUM_MAXP; ++j) {
#pragma unroll
      for (int i = 0; i < j; ++i) {
        if (j < a.P) {
          float d = 0.f;
          if (active) {
            float dx = v[i].x - v[j].x, dy = v[i].y - v[j].y, dz = v[i].z - v[j].z, dw = v[i].w - v[j].w;
            d = dx * dx + dy * dy + dz * dz + dw * dw;
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
          if ((threadIdx.x & 31) == 0) atomicAdd(&s_acc[j * (j - 1) / 2 + i], (double)d);   // fp64 from the warp level up
        }
      }
    }
    __syncthreads();
    for (int q = threadIdx.x; q < npairs; q += DRC_THREADS)
      atomicAdd(&a.pair_d2[(long long)tensor * npairs + q], s_acc[q]);
    __syncthreads();
  }
}

struct KrumSelectArgs {
  double* pair_d2;                // consumed and zeroed
  int T, P, s;
  int* select;                    // [m][T] selected worker slots, ascending per tensor (m = 1: the Krum winner)
  int m;                          // rows kept (1 <= m <= P)
};

__global__ void krum_select_kernel(const __grid_constant__ KrumSelectArgs a) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= a.T) return;
  const int npairs = a.P * (a.P - 1) / 2;
  double* d2 = a.pair_d2 + (long long)t * npairs;
  int keep = a.P - a.s - 2;
  if (keep < 0) keep = 0;
  double scores[KRUM_MAXP];
  for (int i = 0; i < a.P; ++i) {
    double nb[KRUM_MAXP]; int c = 0;
    for (int j = 0; j < a.P; ++j) {
      if (j == i) continue;
      int lo = i < j ? i : j, hi = i < j ? j : i;
      nb[c++] = d2[hi * (hi - 1) / 2 + lo];
    }
    for (int x = 1; x < c; ++x) { double k = nb[x]; int y = x - 1; while (y >= 0 && nb[y] > k) { nb[y + 1] = nb[y]; --y; } nb[y + 1] = k; }
    double score = 0.0;
    for (int x = 0; x < keep && x < c; ++x) score += nb[x];
    scores[i] = score;
  }
  // m rounds of Krum's argmin (first row, then strictly lower scores) over the rows not taken yet: the first round is
  // exactly the Krum selection, non-finite scores included
  unsigned int taken = 0u;
  for (int r = 0; r < a.m; ++r) {
    double best = 0.0; int best_i = -1;
    for (int i = 0; i < a.P; ++i) {
      if ((taken >> i) & 1u) continue;
      if (best_i < 0 || scores[i] < best) { best = scores[i]; best_i = i; }
    }
    taken |= 1u << best_i;
  }
  for (int i = 0, c = 0; i < a.P; ++i)
    if ((taken >> i) & 1u) a.select[(long long)(c++) * a.T + t] = i;
  for (int q = 0; q < npairs; ++q) d2[q] = 0.0;
}

extern "C" int drc_pair_dist(const PairDistArgs* args, int grid, cudaStream_t stream) {
  if (args->P > KRUM_MAXP) return (int)cudaErrorInvalidValue;
  pair_dist_kernel<<<grid, DRC_THREADS, 0, stream>>>(*args);
  return (int)cudaGetLastError();
}
extern "C" int drc_krum_select(const KrumSelectArgs* args, cudaStream_t stream) {
  if (args->P > KRUM_MAXP || args->m < 1 || args->m > args->P) return (int)cudaErrorInvalidValue;
  krum_select_kernel<<<(args->T + 63) / 64, 64, 0, stream>>>(*args);
  return (int)cudaGetLastError();
}


// ---------------------------------------------------------------------------------------------
// Weiszfeld in weight space (one warp per tensor, lane i owns input i; fp64)
// ---------------------------------------------------------------------------------------------
struct GeoMedWeightsArgs {
  double* pair_d2;                // [T][P(P-1)/2] consumed and zeroed
  int T, P, max_iter;
  double eps;                     // stop when no weight moved by more than eps
  float* weights;                 // [T][P] out, sum to 1
  int* iters;                     // [T] out (optional): iterations used
};

__global__ void geomed_weights_kernel(const __grid_constant__ GeoMedWeightsArgs a) {
  const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (t >= a.T) return;
  const int npairs = a.P * (a.P - 1) / 2;
  double* d2 = a.pair_d2 + (long long)t * npairs;
  double row[KRUM_MAXP];
  double maxd = 0.0;
#pragma unroll
  for (int j = 0; j < KRUM_MAXP; ++j) {
    row[j] = 0.0;
    if (j < a.P && lane < a.P && j != lane) {
      const int lo = lane < j ? lane : j, hi = lane < j ? j : lane;
      row[j] = d2[hi * (hi - 1) / 2 + lo];
      maxd = fmax(maxd, row[j]);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) maxd = fmax(maxd, __shfl_xor_sync(0xffffffffu, maxd, o));
  __syncwarp();
  for (int q = lane; q < npairs; q += 32) d2[q] = 0.0;
  double w = lane < a.P ? 1.0 / a.P : 0.0;            // first estimate: the mean
  int it = 0;
  if (maxd > 0.0) {
    const double floor_d = 1e-12 * sqrt(maxd) + 1e-300;
    for (; it < a.max_iter; ++it) {
      double s = 0.0;
#pragma unroll
      for (int j = 0; j < KRUM_MAXP; ++j)
        if (j < a.P) s = fma(__shfl_sync(0xffffffffu, w, j), row[j], s);
      double q = w * s;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
      const double dist = fmax(sqrt(fmax(s - 0.5 * q, 0.0)), floor_d);
      double wn = lane < a.P ? 1.0 / dist : 0.0;
      double sum = wn;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      wn /= sum;
      double delta = fabs(wn - w);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) delta = fmax(delta, __shfl_xor_sync(0xffffffffu, delta, o));
      w = wn;
      if (delta <= a.eps) { ++it; break; }
    }
  }
  if (lane < a.P) a.weights[t * a.P + lane] = (float)w;
  if (a.iters && lane == 0) a.iters[t] = it;
}

extern "C" int drc_geomed_weights(const GeoMedWeightsArgs* args, cudaStream_t stream) {
  if (args->P > KRUM_MAXP) return (int)cudaErrorInvalidValue;
  geomed_weights_kernel<<<(args->T * 32 + 127) / 128, 128, 0, stream>>>(*args);
  return (int)cudaGetLastError();
}
extern "C" int drc_sizeof_GeoMedWeightsArgs() { return (int)sizeof(GeoMedWeightsArgs); }

extern "C" int drc_sizeof_GeoMedArgs() { return (int)sizeof(GeoMedArgs); }
extern "C" int drc_sizeof_GeoMedPrepArgs() { return (int)sizeof(GeoMedPrepArgs); }
extern "C" int drc_sizeof_PairDistArgs() { return (int)sizeof(PairDistArgs); }
extern "C" int drc_sizeof_KrumSelectArgs() { return (int)sizeof(KrumSelectArgs); }
