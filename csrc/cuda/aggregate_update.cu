// K7 + K8 + K9 (+ the second half of K3 / K4 / K6): fused "aggregate -> optimizer (SGD-momentum | Adam | AMSGrad) -> parameter broadcast".
//
// Reference: the PS first builds the aggregated gradient per tensor (mean: baseline_master.py:267-269; vote
// winners summed per tensor: rep_master.py:154-168 -- here divided by #groups, a documented deviation, DESIGN.md section 7; Krum winner: baseline_master.py:278-296; Fourier recombination
// Re(v^T R)/n: cyclic_master.py:125-129,171-172), then SGDModified.step / AdamModified.step (optim/sgd_modified.py:53-88,
// optim/adam_modified.py:32-92), then
// one MPI.Bcast per tensor (baseline_master.py:180-186).  Here a single streaming kernel per step does all
// three: it reads only the gradient rows that contribute, updates momentum + fp32 master parameters in
// place, and stores the fresh parameters directly into every worker's parameter arena -- with one NVLS
// `multimem.st` through a multicast mapping when available, otherwise with unicast peer stores -- and the
// last CTA raises the step-stamped `params_ready` flag on every worker.  No NCCL call.
//
// MODE 3 adds the coordinate-wise robust rules (Yin et al., ICML 2018): trimmed mean and median.  Each output
// element depends only on the P values at the same position, so the rule runs inside this streaming kernel and
// is bucket-pipelined like the mean.
#include "common.cuh"

struct UpdateArgs {
  // gradient source ---------------------------------------------------------------------------
  int mode;                       // 0: select-sum over `select` table; 1: cyclic recombination; 2: real per-tensor weights;
                                  // 3: coordinate-wise trimmed sum over the K slots (median / trimmed mean)
  const float* grad_in;           // mode 0: [P][slot_stride] fp32 ; mode 1: [n][2*slot_stride] complex64
  long long slot_stride;          // elements (fp32 words for mode 0, complex elements for mode 1)
  const int* select;              // mode 0: [K][T] worker slot to read for (k, tensor); null -> rows 0..K-1 for all tensors
  int K;                          // mode 0: rows summed per tensor ; mode 1: n workers
  float scale;                    // 1/K (mean, vote), 1 (krum, median vector), 1/n (cyclic), 1/(K - 2 trim) (mode 3)
  const float2* recomb;           // mode 1: [T][n] recombination vector v (float2 = complex64); mode 2: float [T][K] weights
  TileView tv;
  // optimizer ---------------------------------------------------------------------------------
  float* params;                  // PS master fp32 [D]
  float* momentum;                // [D] SGD momentum buffer / Adam first moment
  float* exp_avg_sq;              // [D] Adam second moment (null for SGD)
  float* max_exp_avg_sq;          // [D] AMSGrad running maximum (null otherwise)
  const HyperParams* hp;
  const unsigned long long* step_ptr;
  unsigned long long first_step;  // step index at which momentum buffers are created (torch semantics)
  float* grad_out;                // optional: aggregated gradient written out (diagnostics / tests), may be null
  // broadcast ---------------------------------------------------------------------------------
  float* mc_params;               // NVLS multicast pointer to the params arena of every rank, or null
  float* dst[DRC_MAX_DST];        // unicast destinations (peer pointers to workers' params arenas)
  int ndst;
  unsigned int* done_counter;
  FlagList flags;                 // params_ready flags (peer pointers); value written = step + 1
  int tile_begin, tile_end;       // bucket of tiles to update + broadcast (tile_end == 0: whole arena)
  int trim;                       // mode 3: values dropped at each end of every coordinate's sorted column (2 trim < K)
};

// Order-preserving map float -> uint32: unsigned comparison of keys = numeric order of the floats, -0 just below +0.
// Every NaN (either sign, any payload) becomes one canonical key above +Inf, the order of np.sort.  Padding slots of the
// sorting network get 0xffffffff, above every real value including NaN.
#define DRC_KEY_NAN 0xfffffffeu
#define DRC_KEY_PAD 0xffffffffu
__device__ __forceinline__ unsigned int order_key(float x) {
  const unsigned int u = __float_as_uint(x);
  if (x != x) return DRC_KEY_NAN;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_value(unsigned int k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// Batcher's odd-even merge sort on N (a power of two) keys, ascending: 19 compare-exchanges for N = 8, 63 for N = 16.
// The comparator list is built at compile time, so the network unrolls into straight-line min / max pairs on registers.
template <int N>
struct SortNet {
  static constexpr int kMax = N * N;              // more than enough room for the comparators of N <= 16
  int n = 0, lo[kMax] = {}, hi[kMax] = {};
  constexpr SortNet() {
    for (int p = 1; p < N; p <<= 1)
      for (int k = p; k >= 1; k >>= 1)
        for (int j = k % p; j + k < N; j += 2 * k)
          for (int i = 0; i < k && i + j + k < N; ++i)
            if ((i + j) / (2 * p) == (i + j + k) / (2 * p)) { lo[n] = i + j; hi[n] = i + j + k; ++n; }
  }
};

template <int N>
__device__ __forceinline__ void sort_network(unsigned int (&v)[N]) {
  constexpr SortNet<N> net;
#pragma unroll
  for (int c = 0; c < net.n; ++c) {
    const unsigned int x = v[net.lo[c]], y = v[net.hi[c]];
    v[net.lo[c]] = min(x, y);
    v[net.hi[c]] = max(x, y);
  }
}

// MODE 3: sort each of the thread's 4 coordinates over the P = K slots and sum the kept values s_{trim} .. s_{P-trim-1}
// (0-based) in ascending order.  MAXP is the network size (8 or 16), chosen from P by the launcher.
template <int MAXP>
__device__ __forceinline__ float4 trimmed_sum(const float* __restrict__ src, long long stride, int K, int trim) {
  unsigned int key[4][MAXP];
#pragma unroll
  for (int k = 0; k < MAXP; ++k) {
    if (k < K) {
      const float4 v = ld_f4(reinterpret_cast<const float4*>(src + k * stride));
      key[0][k] = order_key(v.x); key[1][k] = order_key(v.y); key[2][k] = order_key(v.z); key[3][k] = order_key(v.w);
    } else {
      key[0][k] = key[1][k] = key[2][k] = key[3][k] = DRC_KEY_PAD;
    }
  }
  // bit k set: s_k is summed (one uniform mask instead of two compares per slot keeps both instantiations free of spills)
  const unsigned int kept = ((1u << (K - trim)) - 1u) & ~((1u << trim) - 1u);
  float s[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    sort_network<MAXP>(key[e]);
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < MAXP; ++k)
      if ((kept >> k) & 1u) acc += key_value(key[e][k]);
    s[e] = acc;
  }
  return make_float4(s[0], s[1], s[2], s[3]);
}

template <int MODE, int MAXP = 0>
__global__ void __launch_bounds__(DRC_THREADS) aggregate_update_kernel(const __grid_constant__ UpdateArgs a) {
  const HyperParams hp = *a.hp;
  const unsigned long long step = *a.step_ptr;
  const bool first = (step == a.first_step);
  // Adam: step count t = updates so far + 1; bias corrections folded into the step size like the reference
  float adam_step_size = 0.f;
  if (hp.optimizer != 0) {
    const double t = (double)(step - a.first_step + 1);
    const double bc1 = 1.0 - pow((double)hp.beta1, t), bc2 = 1.0 - pow((double)hp.beta2, t);
    adam_step_size = (float)((double)hp.lr * sqrt(bc2) / bc1);
  }
  const int tile_end = a.tile_end > 0 ? a.tile_end : a.tv.ntiles;
  for (int tile = a.tile_begin + blockIdx.x; tile < tile_end; tile += gridDim.x) {
    const int tensor = a.tv.tile_tensor[tile];
    const long long idx = (long long)tile * DRC_TILE + threadIdx.x * 4;
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    if (MODE == 0) {
      for (int k = 0; k < a.K; ++k) {
        const int slot = a.select ? a.select[k * a.tv.ntensors + tensor] : k;
        float4 v = ld_f4(reinterpret_cast<const float4*>(a.grad_in + slot * a.slot_stride + idx));
        g.x += v.x; g.y += v.y; g.z += v.z; g.w += v.w;
      }
    } else if constexpr (MODE == 3) {
      g = trimmed_sum<MAXP>(a.grad_in + idx, a.slot_stride, a.K, a.trim);
    } else if (MODE == 2) {
      const float* wts = reinterpret_cast<const float*>(a.recomb);    // geometric median: sum_k w[tensor][k] * g_k
      for (int k = 0; k < a.K; ++k) {
        const float w = wts[tensor * a.K + k];
        float4 v = ld_f4(reinterpret_cast<const float4*>(a.grad_in + k * a.slot_stride + idx));
        g.x = fmaf(w, v.x, g.x); g.y = fmaf(w, v.y, g.y); g.z = fmaf(w, v.z, g.z); g.w = fmaf(w, v.w, g.w);
      }
    } else {
      for (int k = 0; k < a.K; ++k) {
        const float2 v = a.recomb[tensor * a.K + k];
        if (v.x == 0.f && v.y == 0.f) continue;             // rows outside the healthy set
        const float4* src = reinterpret_cast<const float4*>(a.grad_in + 2 * (k * a.slot_stride + idx));
        float4 c0 = ld_f4(src), c1 = ld_f4(src + 1);        // (re0,im0,re1,im1) (re2,im2,re3,im3)
        g.x += v.x * c0.x - v.y * c0.y;
        g.y += v.x * c0.z - v.y * c0.w;
        g.z += v.x * c1.x - v.y * c1.y;
        g.w += v.x * c1.z - v.y * c1.w;
      }
    }
    g.x *= a.scale; g.y *= a.scale; g.z *= a.scale; g.w *= a.scale;
    if (a.grad_out) *reinterpret_cast<float4*>(a.grad_out + idx) = g;

    float4 p = *reinterpret_cast<const float4*>(a.params + idx);
    float4 m = *reinterpret_cast<const float4*>(a.momentum + idx);
    float* gp = &g.x; float* pp = &p.x; float* mp = &m.x;
    if (hp.optimizer == 0) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float d = gp[e];
        if (hp.weight_decay != 0.f) d = fmaf(hp.weight_decay, pp[e], d);
        if (hp.momentum != 0.f) {
          float b = first ? d : fmaf(hp.momentum, mp[e], (1.f - hp.dampening) * d);
          mp[e] = b;
          d = hp.nesterov ? fmaf(hp.momentum, b, d) : b;
        }
        pp[e] = fmaf(-hp.lr, d, pp[e]);
      }
    } else {
      float4 v = *reinterpret_cast<const float4*>(a.exp_avg_sq + idx);
      float4 vm = (hp.optimizer == 2) ? *reinterpret_cast<const float4*>(a.max_exp_avg_sq + idx) : v;
      float* vp = &v.x; float* vmp = &vm.x;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float d = gp[e];
        if (hp.weight_decay != 0.f) d = fmaf(hp.weight_decay, pp[e], d);
        mp[e] = fmaf(hp.beta1, mp[e], (1.f - hp.beta1) * d);
        vp[e] = fmaf(hp.beta2, vp[e], (1.f - hp.beta2) * d * d);
        float vv = vp[e];
        if (hp.optimizer == 2) { vmp[e] = fmaxf(vmp[e], vv); vv = vmp[e]; }
        pp[e] = fmaf(-adam_step_size, mp[e] / (sqrtf(vv) + hp.eps), pp[e]);
      }
      *reinterpret_cast<float4*>(a.exp_avg_sq + idx) = v;
      if (hp.optimizer == 2) *reinterpret_cast<float4*>(a.max_exp_avg_sq + idx) = vm;
    }
    *reinterpret_cast<float4*>(a.momentum + idx) = m;
    *reinterpret_cast<float4*>(a.params + idx) = p;
    if (a.mc_params) {
      multimem_st_f4(reinterpret_cast<float4*>(a.mc_params + idx), p);
    } else {
#pragma unroll 1
      for (int d = 0; d < a.ndst; ++d) st_f4(reinterpret_cast<float4*>(a.dst[d] + idx), p);
    }
  }
  if (grid_last_cta(a.done_counter)) {
    if ((int)threadIdx.x < a.flags.n) st_release_sys(a.flags.ptr[threadIdx.x], step + 1);
  }
}

extern "C" int drc_aggregate_update(const UpdateArgs* args, int grid, cudaStream_t stream) {
  if (args->ndst > DRC_MAX_DST || args->flags.n > DRC_MAX_DST) return (int)cudaErrorInvalidValue;
  if (args->mode == 0) aggregate_update_kernel<0><<<grid, DRC_THREADS, 0, stream>>>(*args);
  else if (args->mode == 2) aggregate_update_kernel<2><<<grid, DRC_THREADS, 0, stream>>>(*args);
  else if (args->mode == 3) {
    if (args->K < 1 || args->trim < 0 || 2 * args->trim >= args->K) return (int)cudaErrorInvalidValue;
    if (args->K <= 8) aggregate_update_kernel<3, 8><<<grid, DRC_THREADS, 0, stream>>>(*args);
    else if (args->K <= 16) aggregate_update_kernel<3, 16><<<grid, DRC_THREADS, 0, stream>>>(*args);
    else return (int)cudaErrorInvalidValue;
  }
  else aggregate_update_kernel<1><<<grid, DRC_THREADS, 0, stream>>>(*args);
  return (int)cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Worker side: refresh the bf16 compute copy of the matrix-like parameters from the fp32 arena the PS
// just wrote (one streaming pass over the tiles flagged bf16).
// ---------------------------------------------------------------------------------------------
struct CastArgs {
  const float* src;
  __nv_bfloat16* dst;
  TileView tv;
};

__global__ void __launch_bounds__(DRC_THREADS) cast_params_kernel(const __grid_constant__ CastArgs a) {
  for (int tile = blockIdx.x; tile < a.tv.ntiles; tile += gridDim.x) {
    const int tensor = a.tv.tile_tensor[tile];
    if (!a.tv.meta[tensor].is_bf16) continue;
    const long long idx = (long long)tile * DRC_TILE + threadIdx.x * 4;
    float4 v = ld_f4(reinterpret_cast<const float4*>(a.src + idx));
    __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 out;
    out.x = *reinterpret_cast<unsigned int*>(&lo);
    out.y = *reinterpret_cast<unsigned int*>(&hi);
    *reinterpret_cast<uint2*>(a.dst + idx) = out;
  }
}

extern "C" int drc_cast_params(const CastArgs* args, int grid, cudaStream_t stream) {
  cast_params_kernel<<<grid, DRC_THREADS, 0, stream>>>(*args);
  return (int)cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Flag / step utilities.  Waiters poll flags in their *own* memory; a watchdog turns a lost peer into a
// host-visible error code instead of a silent hang (the reference blocks forever in MPI waitany).
// ---------------------------------------------------------------------------------------------
struct WaitArgs {
  const unsigned long long* flags[DRC_MAX_WORKERS];
  int n;
  const unsigned long long* step_ptr;
  long long addend;               // wait until flag >= *step_ptr + addend
  unsigned long long timeout_ns;  // 0 = wait forever
  int* error;                     // device int: set to 1 + index of the first flag that timed out
  unsigned long long* stamps;     // optional trace ring [64][2]: %globaltimer at entry / at release (the "Comm" time the
                                  // reference prints per step, src/worker/baseline_worker.py:148-150, measured on the device)
};

__global__ void wait_flags_kernel(const __grid_constant__ WaitArgs a) {
  const int i = threadIdx.x;
  const unsigned long long cur = *a.step_ptr;
  unsigned long long t0 = 0;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0));
  if (i < a.n) {
    const unsigned long long want = cur + a.addend;
    unsigned int backoff = 32;
    while (ld_acquire_sys(a.flags[i]) < want) {
      __nanosleep(backoff);
      if (backoff < 512) backoff <<= 1;
      if (a.timeout_ns) {
        unsigned long long t1;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1));
        if (t1 - t0 > a.timeout_ns) { atomicCAS(a.error, 0, i + 1); break; }
      }
    }
  }
  __syncwarp();
  if (a.stamps && i == 0) {
    unsigned long long t1;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1));
    a.stamps[(cur & 63) * 2] = t0;
    a.stamps[(cur & 63) * 2 + 1] = t1;
  }
}

extern "C" int drc_wait_flags(const WaitArgs* args, cudaStream_t stream) {
  if (args->n > DRC_MAX_WORKERS) return (int)cudaErrorInvalidValue;
  wait_flags_kernel<<<1, 32, 0, stream>>>(*args);
  return (int)cudaGetLastError();
}

__global__ void step_add_kernel(unsigned long long* step, long long delta) { *step += delta; }

extern "C" int drc_step_add(unsigned long long* step, long long delta, cudaStream_t stream) {
  step_add_kernel<<<1, 1, 0, stream>>>(step, delta);
  return (int)cudaGetLastError();
}

// Phase stamp: ring[(step & 63) * 8 + col] = %globaltimer.  One thread; placed at phase boundaries of the captured step so that the
// per-step Comp / Comm / Method / Update times the reference prints (src/worker/cyclic_worker.py:154-156, src/master/
// cyclic_master.py:143) exist in graph mode too, measured on the device with no host synchronisation.
__global__ void stamp_kernel(unsigned long long* ring, const unsigned long long* step_ptr, int col) {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  ring[((*step_ptr) & 63ull) * 8ull + (unsigned long long)col] = t;
}

extern "C" int drc_stamp(unsigned long long* ring, const unsigned long long* step_ptr, int col, cudaStream_t stream) {
  stamp_kernel<<<1, 1, 0, stream>>>(ring, step_ptr, col);
  return (int)cudaGetLastError();
}

struct SetFlagArgs {
  FlagList flags;
  const unsigned long long* step_ptr;
  long long addend;
};

__global__ void set_flags_kernel(const __grid_constant__ SetFlagArgs a) {
  if ((int)threadIdx.x < a.flags.n) {
    fence_sys();
    st_release_sys(a.flags.ptr[threadIdx.x], *a.step_ptr + a.addend);
  }
}

extern "C" int drc_set_flags(const SetFlagArgs* args, cudaStream_t stream) {
  set_flags_kernel<<<1, 32, 0, stream>>>(*args);
  return (int)cudaGetLastError();
}

extern "C" int drc_sizeof_UpdateArgs() { return (int)sizeof(UpdateArgs); }
extern "C" int drc_sizeof_CastArgs() { return (int)sizeof(CastArgs); }
extern "C" int drc_sizeof_WaitArgs() { return (int)sizeof(WaitArgs); }
extern "C" int drc_sizeof_SetFlagArgs() { return (int)sizeof(SetFlagArgs); }
extern "C" int drc_sizeof_TensorMeta() { return (int)sizeof(TensorMeta); }
extern "C" int drc_sizeof_HyperParams() { return (int)sizeof(HyperParams); }
extern "C" int drc_sizeof_TileView() { return (int)sizeof(TileView); }
extern "C" int drc_sizeof_FlagList() { return (int)sizeof(FlagList); }
