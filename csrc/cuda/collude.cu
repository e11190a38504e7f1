// Colluding attacks applied by the parameter server: ALIE ("A Little Is Enough", Baruch et al., NeurIPS 2019) and
// inner-product manipulation (Xie et al., UAI 2019).
//
// Both lies are built from every honest gradient, which only meet at the PS.  So the workers push their honest gradient
// and this kernel, launched on the PS right after the slots of a bucket (or of the whole arena) arrived, overwrites the
// liar slots in place before the aggregation rule reads them:
//     mu_j    = mean over honest slots of x_ij
//     sigma_j = sqrt( sum over honest slots of (x_ij - mu_j)^2 / (h - 1) )         (unbiased, like torch.std)
//     alie: every liar slot <- mu - z * sigma          ipm: every liar slot <- -epsilon * mu
// The liar set is the step's adversary bitmap word, read on the device (like push_encode.cu), so a captured graph picks
// up each step's liars by itself.  Oracle: codes/adversary.py::collude (fp64); here fp32, two passes over the honest
// slots (sum, then squared deviations), each a `#pragma unroll 1` loop over the set bits of the honest mask, so P can go up
// to 32 with no per-P register array.  The second pass re-reads the tile the CTA just read, from L2.
#include "common.cuh"

#define DRC_ATTACK_ALIE 5
#define DRC_ATTACK_IPM 6

struct CollusionArgs {
  float* grad_in;                         // [P][slot_stride] the PS's gradient slab (liar rows rewritten in place)
  long long slot_stride;                  // elements between worker slots
  int P;                                  // worker slots (<= 32: the bitmap width)
  TileView tv;
  int tile_begin, tile_end;               // tiles to process (tile_end == 0: up to the end of the arena)
  const unsigned int* adv_bitmap;         // [adv_len] bit w set = worker slot w lies at that step
  int adv_len;
  const unsigned long long* step_ptr;     // device step counter
  int mode;                               // DRC_ATTACK_ALIE | DRC_ATTACK_IPM
  float param;                            // z (alie) | epsilon (ipm)
};

__global__ void __launch_bounds__(DRC_THREADS) collude_kernel(const __grid_constant__ CollusionArgs a) {
  const unsigned int all = a.P >= 32 ? 0xffffffffu : ((1u << a.P) - 1u);
  const unsigned int liars = a.adv_bitmap[*a.step_ptr % (unsigned long long)a.adv_len] & all;
  const unsigned int honest = all & ~liars;
  if (liars == 0u || honest == 0u) return;                    // uniform over the grid: no lie this step
  const int h = __popc(honest);
  const int tile_end = a.tile_end > 0 ? a.tile_end : a.tv.ntiles;
  for (int tile = a.tile_begin + blockIdx.x; tile < tile_end; tile += gridDim.x) {
    int tensor;
    const int valid = tile_valid(a.tv, tile, tensor);
    const int lane_valid = valid - (int)threadIdx.x * 4;
    if (lane_valid <= 0) continue;                            // padding of every slot stays as it is (zero)
    const long long idx = (long long)tile * DRC_TILE + threadIdx.x * 4;
    float4 mu = make_float4(0.f, 0.f, 0.f, 0.f);
    unsigned int m = honest;
#pragma unroll 1
    while (m) {                                               // ascending slot order
      const int i = __ffs(m) - 1;
      m &= m - 1u;
      const float4 v = ld_f4(reinterpret_cast<const float4*>(a.grad_in + i * a.slot_stride + idx));
      mu.x += v.x; mu.y += v.y; mu.z += v.z; mu.w += v.w;
    }
    mu.x /= (float)h; mu.y /= (float)h; mu.z /= (float)h; mu.w /= (float)h;
    float4 lie;
    if (a.mode == DRC_ATTACK_ALIE) {
      float4 sq = make_float4(0.f, 0.f, 0.f, 0.f);
      m = honest;
#pragma unroll 1
      while (m) {
        const int i = __ffs(m) - 1;
        m &= m - 1u;
        const float4 v = ld_f4(reinterpret_cast<const float4*>(a.grad_in + i * a.slot_stride + idx));
        const float dx = v.x - mu.x, dy = v.y - mu.y, dz = v.z - mu.z, dw = v.w - mu.w;
        sq.x = fmaf(dx, dx, sq.x); sq.y = fmaf(dy, dy, sq.y); sq.z = fmaf(dz, dz, sq.z); sq.w = fmaf(dw, dw, sq.w);
      }
      const float hm1 = (float)(h - 1);
      const float nz = -a.param;
      lie = make_float4(fmaf(nz, sqrtf(sq.x / hm1), mu.x), fmaf(nz, sqrtf(sq.y / hm1), mu.y),
                        fmaf(nz, sqrtf(sq.z / hm1), mu.z), fmaf(nz, sqrtf(sq.w / hm1), mu.w));
    } else {
      const float ne = -a.param;
      lie = make_float4(ne * mu.x, ne * mu.y, ne * mu.z, ne * mu.w);
    }
    if (lane_valid < 4) {                                     // tail of a tensor: the padding lanes stay +0
      if (lane_valid < 2) lie.y = 0.f;
      if (lane_valid < 3) lie.z = 0.f;
      lie.w = 0.f;
    }
    m = liars;
#pragma unroll 1
    while (m) {
      const int i = __ffs(m) - 1;
      m &= m - 1u;
      st_f4(reinterpret_cast<float4*>(a.grad_in + i * a.slot_stride + idx), lie);
    }
  }
}

extern "C" int drc_collude(const CollusionArgs* args, int grid, cudaStream_t stream) {
  if (args->P < 1 || args->P > DRC_MAX_WORKERS || args->adv_len < 1 || !args->adv_bitmap || !args->step_ptr ||
      (args->mode != DRC_ATTACK_ALIE && args->mode != DRC_ATTACK_IPM))
    return (int)cudaErrorInvalidValue;
  collude_kernel<<<grid, DRC_THREADS, 0, stream>>>(*args);
  return (int)cudaGetLastError();
}

extern "C" int drc_sizeof_CollusionArgs() { return (int)sizeof(CollusionArgs); }
