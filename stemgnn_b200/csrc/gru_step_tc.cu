// GRU recurrence for node counts beyond the cluster envelope (N > 480: BASELINE.json configs[4], N = 2048) on tcgen05.
// Reference: models/base_model.py:92,137 (nn.GRU over the node axis) and :154-155 (key / query contraction).
//
// W_hh (3N x N) no longer fits on chip (fp16 hi + lo = 50 MB at N = 2048), so a step is ONE kernel launch whose CTAs
// stream their rows of W_hh from L2 (126 MB: the hi/lo images stay L2-resident across the N steps) through TMA:
//   * CTA (q, grp) owns 40 hidden units (120 rows of W_hh, gate-major) and 32 sequences; per 64-column K chunk a TMA stage
//     carries the A tiles W_hi, W_lo (128 x 64 fp16 each) and the B tile [h_hi (32 rows); h_lo (32 rows)] of h_{s-1};
//   * two M128 x N64 x K16 instructions per 16 hidden units (A = W_hi, A = W_lo) accumulate the four partial products in
//     tensor memory; gh = D00 + 2^-11 (D01 + D10) + 2^-22 D11 (same split-operand scheme as gru_tc.cu: fp32-level parity);
//   * epilogue: tcgen05.ld -> smem transpose -> gate math with the in-kernel input projection (36 FMAs per unit-step) ->
//     fp32 master copy of h, key / query accumulators (unit-major scratch) and the fp16 hi/lo image of h_s that the NEXT
//     launch reads as its B operand (kernel boundary = the grid-wide exchange of h).
// Bound: L2 -> SM streaming of the W_hh images (2 * 3N * N * 2 bytes per step = 50 MB at N = 2048, ~10 us at the measured
// ~5-6 TB/s L2 rate) — DESIGN.md §8.  The round-1 per-step FFMA path (gru_step_kernel) took ~130 us per step.
#include <stdlib.h>

#include "common.cuh"
#include "internal.cuh"
#include "sm100.cuh"

namespace sg {
namespace {

constexpr int ST_U = 40;                // hidden units per CTA
constexpr int ST_SEQ = 32;              // sequences per CTA (B operand: 32 hi rows + 32 lo rows)
constexpr int ST_THREADS = 192;         // warp 0 TMA, warp 1 MMA, warps 2..5 epilogue
constexpr int ST_NSTG = 4;
constexpr uint32_t ST_A_BYTES = 128 * 128;        // one A tile (128 rows x 64 fp16)
constexpr uint32_t ST_B_BYTES = 64 * 128;         // B tile (64 rows x 64 fp16)
constexpr uint32_t ST_STAGE = 2 * ST_A_BYTES + ST_B_BYTES;
constexpr uint32_t ST_TMEM_COLS = 128;
constexpr float ST_LO_INV = 1.0f / F16_LO_SCALE, ST_LO_INV2 = 1.0f / (F16_LO_SCALE * F16_LO_SCALE);
constexpr int ST_SPIN_LOG2 = 26;        // mbarrier polls before a lost arrival traps

constexpr uint32_t ST_IDESC = umma_idesc_m128(UMMA_F16, 64);     // fp16 x fp16 -> fp32, M128 N64

// W_hh (3N, N) fp32 -> image rows [(tile * 2 + arr) * 128 + (gate * 40 + lu)][KP] fp16 (rows 120..127 and pads zero)
__global__ void __launch_bounds__(256) step_pack_whh_kernel(const float* __restrict__ w_hh, unsigned short* __restrict__ img,
                                                             int N, int NT, int KP) {
  const long long total = (long long)NT * 128 * KP;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(idx % KP);
    const int row = (int)((idx / KP) % 128);
    const int q = (int)(idx / ((long long)KP * 128));
    float v = 0.f;
    if (row < 3 * ST_U && k < N) {
      const int gate = row / ST_U, lu = row - gate * ST_U;
      const int u = q * ST_U + lu;
      if (u < N) v = __ldg(w_hh + ((size_t)gate * N + u) * N + k);
    }
    unsigned short hi, lo;
    split_f16_hi_lo_scaled(v, hi, lo);
    img[((size_t)(q * 2 + 0) * 128 + row) * KP + k] = hi;
    img[((size_t)(q * 2 + 1) * 128 + row) * KP + k] = lo;
  }
}

struct StepArgs {
  GruArgs a;
  float* hstate;          // (N, Bp) fp32 master copy of h, unit-major (Bp = groups * 32)
  float* keyT;            // (N, Bp)
  float* queryT;          // (N, Bp)
  unsigned short* himg;   // [2][groups * 64][KP] fp16 images of h (rows 0..31 hi, 32..63 lo per group)
  int s, NCH, KP, Bp;
};

__global__ void __launch_bounds__(ST_THREADS, 1)
gru_step_tc_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_h, StepArgs t) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + smem_pad1024(smem_raw);
  uint8_t* stages = smem;
  float* gh_sm = reinterpret_cast<float*>(stages + ST_NSTG * ST_STAGE);     // [120][32]
  float* wih_sm = gh_sm + 3 * ST_U * ST_SEQ;                                 // [120][W]
  float* bias_sm = wih_sm + 3 * ST_U * t.a.W;                                // [4][40]
  float* x_sm = bias_sm + 4 * ST_U;                                          // [32][W]
  uint8_t* bar_base = reinterpret_cast<uint8_t*>(x_sm + ST_SEQ * t.a.W);
  bar_base += (8u - (smem_u32(bar_base) & 7u)) & 7u;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(bar_base);
  uint64_t* empty_bar = full_bar + ST_NSTG;
  uint64_t* tfull = empty_bar + ST_NSTG;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tfull + 1);

  const GruArgs& a = t.a;
  const int N = a.N, B = a.B, W = a.W, s = t.s;
  const int q = blockIdx.x, grp = blockIdx.y;
  const int u0 = q * ST_U, b0 = grp * ST_SEQ;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cur = s & 1, nxt = cur ^ 1;

  if (threadIdx.x == 0) {
    for (int i = 0; i < ST_NSTG; ++i) {
      mbarrier_init(&full_bar[i], 1);
      mbarrier_init(&empty_bar[i], 1);
    }
    mbarrier_init(tfull, 1);
    fence_mbarrier_init();
  }
  if (warp == 1) {
    tcgen05_alloc(tmem_slot, ST_TMEM_COLS);
    tcgen05_relinquish_alloc_permit();
  }
  if (warp >= 2) {      // step-local constants for the gate phase
    const int et = threadIdx.x - 64;
    for (int i = et; i < 3 * ST_U * W; i += 128) {
      const int row = i / W, tt = i - row * W;
      const int gate = row / ST_U, lu = row - gate * ST_U;
      const int u = u0 + lu;
      wih_sm[i] = u < N ? __ldg(a.w_ih + ((size_t)gate * N + u) * W + tt) : 0.f;
    }
    for (int i = et; i < 4 * ST_U; i += 128) {
      const int gate = i / ST_U, lu = i - gate * ST_U;
      const int u = u0 + lu;
      float v = 0.f;
      if (u < N) {
        if (gate < 2) v = __ldg(a.b_ih + gate * N + u) + __ldg(a.b_hh + gate * N + u);
        else if (gate == 2) v = __ldg(a.b_ih + 2 * N + u);
        else v = __ldg(a.b_hh + 2 * N + u);
      }
      bias_sm[i] = v;
    }
    for (int i = et; i < ST_SEQ * W; i += 128) {
      const int bb = i / W, tt = i - bb * W;
      x_sm[i] = (b0 + bb) < B ? __ldg(a.xs + ((size_t)s * B + b0 + bb) * W + tt) : 0.f;
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one_sync()) {        // ===== TMA producer =====
      for (int c = 0; c < t.NCH; ++c) {
        const int st = c % ST_NSTG;
        const uint32_t ph = (uint32_t)(c / ST_NSTG) & 1u;
        mbarrier_wait<ST_SPIN_LOG2>(&empty_bar[st], ph ^ 1u);
        uint8_t* dst = stages + (size_t)st * ST_STAGE;
        mbarrier_arrive_expect_tx(&full_bar[st], ST_STAGE);
        tma_load_2d(dst, &map_w, &full_bar[st], c * 64, (q * 2 + 0) * 128);
        tma_load_2d(dst + ST_A_BYTES, &map_w, &full_bar[st], c * 64, (q * 2 + 1) * 128);
        tma_load_2d(dst + 2 * ST_A_BYTES, &map_h, &full_bar[st], c * 64, (cur * (int)gridDim.y + grp) * 64);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===== MMA issuer (converged warp, elected lane) =====
    for (int c = 0; c < t.NCH; ++c) {
      const int st = c % ST_NSTG;
      const uint32_t ph = (uint32_t)(c / ST_NSTG) & 1u;
      mbarrier_wait<ST_SPIN_LOG2>(&full_bar[st], ph);
      tcgen05_fence_after();
      if (elect_one_sync()) {
        const uint32_t a_hi = smem_u32(stages + (size_t)st * ST_STAGE), a_lo = a_hi + ST_A_BYTES, bt = a_lo + ST_A_BYTES;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const uint64_t bd = umma_desc_kmajor(bt + kk * 32, 1024, UMMA_SWIZZLE_128B);
          const uint32_t acc = (c > 0 || kk > 0) ? 1u : 0u;
          // W_hi . [h_hi | h_lo], then W_lo . [h_hi | h_lo]
          tcgen05_mma_f16(tmem_base, umma_desc_kmajor(a_hi + kk * 32, 1024, UMMA_SWIZZLE_128B), bd, ST_IDESC, acc);
          tcgen05_mma_f16(tmem_base + 64, umma_desc_kmajor(a_lo + kk * 32, 1024, UMMA_SWIZZLE_128B), bd, ST_IDESC, acc);
        }
        tcgen05_commit(&empty_bar[st]);
        if (c + 1 == t.NCH) tcgen05_commit(tfull);
      }
      __syncwarp();
    }
  } else {
    // ===== epilogue =====
    const int et = threadIdx.x - 64;
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16);
    mbarrier_wait<ST_SPIN_LOG2>(tfull, 0);
    tcgen05_fence_after();
#pragma unroll
    for (int half = 0; half < 2; ++half) {            // 16 sequences at a time; every lane takes part in the aligned loads
      float d00[16], d01[16], d10[16], d11[16];
      tcgen05_ld_32x32b_x16(taddr + half * 16, d00);                   // W_hi.h_hi
      tcgen05_ld_32x32b_x16(taddr + 32 + half * 16, d01);              // W_hi.h_lo
      tcgen05_ld_32x32b_x16(taddr + 64 + half * 16, d10);              // W_lo.h_hi
      tcgen05_ld_32x32b_x16(taddr + 96 + half * 16, d11);              // W_lo.h_lo
      tcgen05_wait_ld();
      if (row < 3 * ST_U) {                            // rows 120..127 hold no unit
#pragma unroll
        for (int j = 0; j < 16; ++j)
          gh_sm[row * ST_SEQ + half * 16 + j] = d00[j] + (d01[j] + d10[j]) * ST_LO_INV + d11[j] * ST_LO_INV2;
      }
    }
    tcgen05_fence_before();
    bar_sync<1, 128>();
    // gate phase: thread -> sequence b = et % 32, units lu = et / 32 + 4 i
    const int bb = et & 31;
    const int bglob = b0 + bb;
    const float wk_s = __ldg(a.wk + s), wq_s = __ldg(a.wq + s);
    unsigned short* hnext = t.himg + ((size_t)(nxt * (int)gridDim.y + grp) * 64) * t.KP;
    for (int lu = et >> 5; lu < ST_U; lu += 4) {
      const int u = u0 + lu;
      float hn = 0.f;
      if (u < N && bglob < B) {
        float gr = bias_sm[lu], gz = bias_sm[ST_U + lu], gn = bias_sm[2 * ST_U + lu];
        const float* xr = x_sm + bb * W;
        const float* wr = wih_sm + (size_t)lu * W;
        const float* wz = wr + (size_t)ST_U * W;
        const float* wn = wz + (size_t)ST_U * W;
        for (int tt = 0; tt < W; ++tt) {
          const float xv = xr[tt];
          gr = fmaf(wr[tt], xv, gr);
          gz = fmaf(wz[tt], xv, gz);
          gn = fmaf(wn[tt], xv, gn);
        }
        const float gh_r = gh_sm[lu * ST_SEQ + bb], gh_z = gh_sm[(ST_U + lu) * ST_SEQ + bb];
        const float gh_n = gh_sm[(2 * ST_U + lu) * ST_SEQ + bb] + bias_sm[3 * ST_U + lu];
        const size_t so = (size_t)u * t.Bp + bglob;
        const float hprev = s > 0 ? t.hstate[so] : 0.f;
        const float r = fast_sigmoid(gr + gh_r), z = fast_sigmoid(gz + gh_z), n = fast_tanh(gn + r * gh_n);
        hn = (1.f - z) * n + z * hprev;
        t.hstate[so] = hn;
        t.keyT[so] = fmaf(hn, wk_s, s > 0 ? t.keyT[so] : 0.f);
        t.queryT[so] = fmaf(hn, wq_s, s > 0 ? t.queryT[so] : 0.f);
        if (a.h_all != nullptr) {
          const size_t o = ((size_t)s * B + bglob) * N + u;
          a.h_all[o] = hn;
          if (a.g_r != nullptr) {
            a.g_r[o] = r; a.g_z[o] = z; a.g_n[o] = n; a.g_hn[o] = gh_n;
          }
        }
      }
      if (u < t.KP) {      // fp16 hi / lo image of h_s: the B operand of the next launch
        unsigned short hi, lo;
        split_f16_hi_lo_scaled(hn, hi, lo);
        hnext[(size_t)bb * t.KP + u] = hi;
        hnext[(size_t)(32 + bb) * t.KP + u] = lo;
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tcgen05_dealloc(tmem_base, ST_TMEM_COLS);
  }
}

// key / query (N, Bp) unit-major scratch -> (B, N)
__global__ void step_finish_kernel(const float* __restrict__ keyT, const float* __restrict__ queryT, float* __restrict__ key,
                                   float* __restrict__ query, int B, int N, int Bp) {
  const long long total = (long long)B * N;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(idx / N), u = (int)(idx % N);
    key[idx] = keyT[(size_t)u * Bp + b];
    query[idx] = queryT[(size_t)u * Bp + b];
  }
}

}  // namespace

// bytes of scratch (inside the `gi` region) the step path needs
size_t gru_step_tc_scratch_bytes(int B, int N) {
  const int NT = ceil_div(N, ST_U), KP = ceil_div(N, 64) * 64, groups = ceil_div(B, ST_SEQ), Bp = groups * ST_SEQ;
  return (size_t)NT * 2 * 128 * KP * 2 + (size_t)2 * groups * 64 * KP * 2 + (size_t)3 * KP * Bp * 4 + 1024;
}

// returns 0 launched, -1 not applicable here (caller falls back), >0 error
int gru_step_tc_forward(const GruArgs& a, uint8_t* scratch, size_t scratch_bytes, int reuse_img, cudaStream_t st) {
  static const bool off = getenv("STEMGNN_GRU_NO_STEP_TC") != nullptr;
  if (off || scratch == nullptr || a.W > 64) return -1;
  if (gru_step_tc_scratch_bytes(a.B, a.N) > scratch_bytes || (reinterpret_cast<uintptr_t>(scratch) & 255)) return -1;
  const int N = a.N, B = a.B;
  const int NT = ceil_div(N, ST_U), NCH = ceil_div(N, 64), KP = NCH * 64, groups = ceil_div(B, ST_SEQ), Bp = groups * ST_SEQ;
  unsigned short* wimg = reinterpret_cast<unsigned short*>(scratch);
  unsigned short* himg = wimg + (size_t)NT * 2 * 128 * KP;
  float* hstate = reinterpret_cast<float*>(himg + (size_t)2 * groups * 64 * KP);
  float* keyT = hstate + (size_t)KP * Bp;
  float* queryT = keyT + (size_t)KP * Bp;
  CUtensorMap mw, mh;
  if (!make_tensor_map_2d(&mw, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, wimg, (uint64_t)NT * 2 * 128, KP, KP * 2ull, 128, 64,
                          CU_TENSOR_MAP_SWIZZLE_128B) ||
      !make_tensor_map_2d(&mh, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, himg, (uint64_t)2 * groups * 64, KP, KP * 2ull, 64, 64,
                          CU_TENSOR_MAP_SWIZZLE_128B))
    return -1;
  const size_t smem = (size_t)ST_NSTG * ST_STAGE + ((size_t)3 * ST_U * ST_SEQ + (size_t)3 * ST_U * a.W + 4 * ST_U +
                                                    (size_t)ST_SEQ * a.W + 2) * sizeof(float) +
                      (2 * ST_NSTG + 1) * 8 + 16 + 1024;
  if (smem > 227 * 1024) return -1;
  SG_CUDA(cudaFuncSetAttribute(gru_step_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (!reuse_img) {
    const long long total = (long long)NT * 128 * KP;
    step_pack_whh_kernel<<<(int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16), 256, 0, st>>>(
        a.w_hh, wimg, N, NT, KP);
    SG_LAUNCH_CHECK("step_pack_whh_kernel");
  }
  SG_CUDA(cudaMemsetAsync(himg, 0, (size_t)2 * groups * 64 * KP * 2, st));      // h_{-1} = 0 and zero padding
  StepArgs t = {};
  t.a = a; t.hstate = hstate; t.keyT = keyT; t.queryT = queryT; t.himg = himg; t.NCH = NCH; t.KP = KP; t.Bp = Bp;
  ProfileHook* hook = profile_hook();
  if (hook->start != nullptr) SG_CUDA(cudaEventRecord(hook->start, st));
  dim3 grid(NT, groups);
  for (int s = 0; s < N; ++s) {
    t.s = s;
    gru_step_tc_kernel<<<grid, ST_THREADS, smem, st>>>(mw, mh, t);
    count_launch();
  }
  SG_LAUNCH_CHECK("gru_step_tc_kernel");
  if (hook->stop != nullptr) SG_CUDA(cudaEventRecord(hook->stop, st));
  step_finish_kernel<<<ceil_div(B * N, 256), 256, 0, st>>>(keyT, queryT, a.key, a.query, B, N, Bp);
  SG_LAUNCH_CHECK("step_finish_kernel");
  return 0;
}

}  // namespace sg
