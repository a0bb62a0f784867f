// Spectral-block GEMMs on tcgen05 with fp32 parity: 3xTF32 split operands, the split done IN the kernel.
//
//   gft_tc        gfted = mul_L[1..3] @ x              (reference models/base_model.py:63, the graph Fourier transform)
//   out_head_tc   igfted -> forecast / backcast heads  (reference :64-72: `weight` contraction, irfft, forecast/backcast
//                                                       Linear layers folded into one map `woutT`, then the sigmoid heads)
//   tc3_gemm      C (+)= alpha A B^T                   (the backward GEMMs of the GLU layers and dW_hh)
//
// One kernel, three epilogues.  kind::tf32 reads 10 mantissa bits of an fp32 operand; a single pass therefore carries
// ~2^-10 relative operand error (round 1's "truncated TF32", which met the 1e-3 / 1e-4 tolerance only at the model
// output).  Here every operand is x = hi + lo with hi = x & 0xffffe000 (what the tensor core reads of the raw fp32 word:
// it truncates, see split_granule) and lo = x - hi (exact in fp32, <= 13 significant bits), and
// each 8-wide K step issues hi.hi into one fp32 accumulator in tensor memory and hi.lo + lo.hi into a SECOND one; the epilogue
// adds the two.  Operand error ~2^-21.  (Why two accumulators: the tensor core truncates the running sum at every accumulating
// MMA — measured, the error of a split product grows linearly with K, 4e-6 of max|C| at K = 480 with all three products in one
// accumulator — and the cross terms are 2^-10 of the main product, so in their own accumulator they are truncated at
// 2^-34 instead of adding two more 2^-24 truncations per K step to the main sum.)
//
// Pipeline per 32-column K block (one 128-byte swizzle row), 320 threads:
//   warp 0        TMA producer: fp32 tiles of A (128 rows) and B (NT rows), 128B-swizzled, K tail / row tail zero-filled
//   warps 2..9    converters: write `lo` to a second tile of the same (swizzled) layout — the transform is elementwise, so
//                 it is layout agnostic; the TMA-written tile itself serves as `hi` (the tensor core truncates it) —
//                 fence.proxy.async, arrive on conv_bar
//   warp 1        converged warp, elected lane issues the tcgen05.mma of a K step; tcgen05.commit frees the stage.
//                 Stage layout [A_hi | A_lo | B_hi | B_lo]: when 2*NT <= 256 the B operand of the first MMA is the STACKED
//                 tile [B_hi; B_lo] (N = 2*NT), so A_hi is read once for hi.hi (columns [0,NT)) and hi.lo (columns [NT,2NT));
//                 the second MMA adds lo.hi onto the cross-term columns: 2 instructions per K step instead of 3.
//   warps 2..9    epilogue from tensor memory (tcgen05.ld 32x32b: thread = accumulator row; the two warps that share a
//                 TMEM lane quarter split the columns).  ncu (profiles/r02_ncu_spec_*): these kernels are bound by
//                 shared-memory bandwidth (TMA fill + split traffic + 3x operand reads) and by the epilogue's latency
//                 chains, not by the tensor pipe — hence 8 worker warps and the stacked B operand.
#include <stdlib.h>

#include "common.cuh"
#include "internal.cuh"
#include "sm100.cuh"

namespace sg {
namespace {

constexpr int S_BM = 128;
constexpr int S_BK = 32;                 // fp32 elements per K block = one 128-byte swizzle row
constexpr int S_THREADS = 320;          // warp 0 TMA, warp 1 MMA issue, warps 2..9 operand split + epilogue
constexpr int S_WORKERS = 256;
constexpr uint32_t S_A_BYTES = S_BM * 128;
constexpr int S_SPIN_LOG2 = 26;         // mbarrier polls before a lost arrival traps

enum { EPI_STORE = 0, EPI_GFT = 1, EPI_HEAD = 2 };

struct Tc3Args {
  int M, K;            // rows of A that exist, reduction length
  int NT;              // columns (rows of the B operand) per CTA: multiple of 16, 16..256
  int nstage;          // smem ring depth
  int split;           // 1: 3xTF32 split products (fp32 parity), 0: one product on the raw fp32 bits
  int stacked;         // split only: [B_hi; B_lo] used as ONE B operand of N = 2*NT (needs 2*NT <= 256)
  uint32_t tmem_cols;  // allocation (power of two >= 32)
  uint32_t lo_col;     // column offset of the cross-term accumulator (split only; NT when stacked)
  // ---- EPI_STORE:  C0/C1[m][n] (+)= alpha * acc;  rows m >= msplit go to C1 (row m - msplit)
  float* C0; float* C1; int ldc, msplit, n_store, atomic; float alpha;
  // ---- EPI_GFT:    row m' = node*3 + k' (INTERLEAVED Chebyshev terms), column c = b*W + t
  //                  -> G[(b*Nn + node)*3W + k'*W + t] = G[b][m'][t] (dense (B, 3Nn, W)) and its 16-bit images
  float* G; unsigned short* g_hi; unsigned short* g_lo; int ldh, bf16, Nn, W, BW;
  // ---- EPI_HEAD:   row = (b, node); columns [0,T) forecast pre-activation, [T,T+W) backcast pre-activation
  const float* bf; const float* wfr; const float* bfr; const float* bb; const float* wsc; const float* bsc;
  const float* x_bnw; float* forecast; float* bc_bnw; float* bc_bwn; float* bc_pad; int ld_pad; float* save_fs; int T;
};

// lo = x - (x & 0xffffe000).  The `hi` tile is NOT rewritten: kind::tf32 truncates its operands to the top 19 bits (measured:
// the error of a single pass on seeded inputs equals the truncation model to 3 digits on every tested shape — 6.42e-4 /
// 9.35e-4 / 7.19e-4 / 7.92e-4 — where round-to-nearest would give 4.18e-4 / 3.83e-4 / 2.76e-4 / 3.78e-4; profiles/README.md),
// so the raw fp32 tile already IS the hi operand.  If a future part rounded instead, tests/test_spec_tc_gpu.py would fail at
// the 1e-4 level; S_MASK_HI = 1 restores the explicit mask (one more 16-byte shared store per granule).
#ifndef S_MASK_HI
#define S_MASK_HI 0
#endif
__device__ __forceinline__ void split_granule(const uint4 v, uint4& h, uint4& l) {
  h.x = v.x & 0xffffe000u; h.y = v.y & 0xffffe000u; h.z = v.z & 0xffffe000u; h.w = v.w & 0xffffe000u;
  l.x = __float_as_uint(__uint_as_float(v.x) - __uint_as_float(h.x));
  l.y = __float_as_uint(__uint_as_float(v.y) - __uint_as_float(h.y));
  l.z = __float_as_uint(__uint_as_float(v.z) - __uint_as_float(h.z));
  l.w = __float_as_uint(__uint_as_float(v.w) - __uint_as_float(h.w));
}

template <int EPI>
__global__ void __launch_bounds__(S_THREADS, 1)
tc3_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, Tc3Args g) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + smem_pad1024(smem_raw);
  const int NT = g.NT, S = g.nstage;
  const uint32_t b_bytes = (uint32_t)NT * 128;
  const bool split = g.split != 0;
  // stage: split [A_hi | A_lo | B_hi | B_lo], otherwise [A | B]
  const uint32_t a_lo_off = S_A_BYTES;
  const uint32_t b_hi_off = split ? 2 * S_A_BYTES : S_A_BYTES;
  const uint32_t b_lo_off = b_hi_off + b_bytes;
  const uint32_t stage_bytes = split ? 2 * (S_A_BYTES + b_bytes) : S_A_BYTES + b_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)S * stage_bytes);
  uint64_t* empty_bar = full_bar + S;
  uint64_t* conv_bar = empty_bar + S;
  uint64_t* tmem_full_bar = conv_bar + S;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);
  float* s_head = reinterpret_cast<float*>(tmem_slot + 2);       // EPI_HEAD only

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * S_BM;
  const int n0 = blockIdx.y * NT;
  const int total_kb = (g.K + S_BK - 1) / S_BK;
  const int per = (total_kb + gridDim.z - 1) / gridDim.z;
  const int kb0 = blockIdx.z * per;
  const int kb1 = min(total_kb, kb0 + per);
  const int num_kb = kb1 - kb0;          // may be <= 0 for trailing K splits: nothing to add

  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbarrier_init(&full_bar[s], 1);
      mbarrier_init(&empty_bar[s], 1);
      mbarrier_init(&conv_bar[s], S_WORKERS);
    }
    mbarrier_init(tmem_full_bar, 1);
    fence_mbarrier_init();
    prefetch_tensormap(&map_a);
    prefetch_tensormap(&map_b);
  }
  if (warp == 1) {
    tcgen05_alloc(tmem_slot, g.tmem_cols);
    tcgen05_relinquish_alloc_permit();
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (num_kb > 0 && elect_one_sync()) {
      for (int i = 0; i < num_kb; ++i) {
        const int s = i % S;
        const uint32_t ph = (uint32_t)(i / S) & 1u;
        mbarrier_wait<S_SPIN_LOG2>(&empty_bar[s], ph ^ 1u);
        uint8_t* st = smem + (size_t)s * stage_bytes;
        mbarrier_arrive_expect_tx(&full_bar[s], S_A_BYTES + b_bytes);
        tma_load_2d(st, &map_a, &full_bar[s], (kb0 + i) * S_BK, m0);
        tma_load_2d(st + b_hi_off, &map_b, &full_bar[s], (kb0 + i) * S_BK, n0);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===== MMA issuer: converged warp, one elected lane =====
    if (num_kb > 0) {
      const uint32_t idesc = umma_idesc_m128(UMMA_TF32, NT);
      const uint32_t idesc2 = umma_idesc_m128(UMMA_TF32, 2 * NT);          // stacked [B_hi; B_lo]
      const uint32_t lo_col = g.lo_col;
      const bool stacked = g.stacked != 0;
      for (int i = 0; i < num_kb; ++i) {
        const int s = i % S;
        const uint32_t ph = (uint32_t)(i / S) & 1u;
        mbarrier_wait<S_SPIN_LOG2>(split ? &conv_bar[s] : &full_bar[s], ph);
        tcgen05_fence_after();
        if (elect_one_sync()) {
          const uint32_t a_hi = smem_u32(smem + (size_t)s * stage_bytes);
          const uint32_t a_lo = a_hi + a_lo_off, b_hi = a_hi + b_hi_off, b_lo = a_hi + b_lo_off;
#pragma unroll
          for (int kk = 0; kk < S_BK / 8; ++kk) {      // 8 tf32 = 32 bytes along K per instruction
            const uint32_t acc = (i > 0 || kk > 0) ? 1u : 0u;
            const uint64_t da = umma_desc_kmajor(a_hi + kk * 32, 1024, UMMA_SWIZZLE_128B);
            const uint64_t db = umma_desc_kmajor(b_hi + kk * 32, 1024, UMMA_SWIZZLE_128B);
            if (!split) {
              tcgen05_mma_tf32(tmem_base, da, db, idesc, acc);
            } else if (stacked) {   // hi.hi -> [0,NT), hi.lo -> [NT,2NT) in one instruction; then lo.hi onto [NT,2NT)
              tcgen05_mma_tf32(tmem_base, da, db, idesc2, acc);
              tcgen05_mma_tf32(tmem_base + lo_col, umma_desc_kmajor(a_lo + kk * 32, 1024, UMMA_SWIZZLE_128B), db, idesc,
                               1u);
            } else {                // cross terms in their own accumulator (file header)
              tcgen05_mma_tf32(tmem_base, da, db, idesc, acc);
              tcgen05_mma_tf32(tmem_base + lo_col, umma_desc_kmajor(a_lo + kk * 32, 1024, UMMA_SWIZZLE_128B), db, idesc,
                               acc);
              tcgen05_mma_tf32(tmem_base + lo_col, da, umma_desc_kmajor(b_lo + kk * 32, 1024, UMMA_SWIZZLE_128B), idesc,
                               1u);
            }
          }
          tcgen05_commit(&empty_bar[s]);
        }
        __syncwarp();
      }
      if (elect_one_sync()) tcgen05_commit(tmem_full_bar);
      __syncwarp();
    }
  } else {
    // ===== warps 2..9: operand split in shared memory, then the epilogue =====
    const int tid = threadIdx.x - 64;                 // 0..255
    float *s_wfr = nullptr, *s_wsc = nullptr, *s_bf = nullptr, *s_bfr = nullptr, *s_bb = nullptr, *s_bsc = nullptr,
          *s_fs = nullptr, *s_pb = nullptr, *s_x = nullptr;
    if (EPI == EPI_HEAD) {
      const int T = g.T, W = g.W;
      s_wfr = s_head;                 // [W][T]   forecast_result.weight
      s_wsc = s_wfr + W * T;          // [W][W]   backcast_short_cut.weight
      s_bf = s_wsc + W * W;           // [T]
      s_bfr = s_bf + T;               // [W]
      s_bb = s_bfr + W;               // [W]
      s_bsc = s_bb + W;               // [W]
      s_fs = s_bsc + W;               // [T][128]  forecast_source of a row (column = row: conflict free)
      s_pb = s_fs + T * 128;          // [W][128]  backcast pre-activation
      s_x = s_pb + W * 128;           // [W][128]  block input row
      for (int i = tid; i < W * T; i += S_WORKERS) s_wfr[i] = __ldg(g.wfr + i);
      for (int i = tid; i < T; i += S_WORKERS) s_bf[i] = __ldg(g.bf + i);
      for (int i = tid; i < W; i += S_WORKERS) s_bfr[i] = __ldg(g.bfr + i);
      if (g.bc_bnw != nullptr) {
        for (int i = tid; i < W * W; i += S_WORKERS) s_wsc[i] = __ldg(g.wsc + i);
        for (int i = tid; i < W; i += S_WORKERS) {
          s_bb[i] = __ldg(g.bb + i);
          s_bsc[i] = __ldg(g.bsc + i);
        }
      }
      bar_sync<1, 256>();
    }
    if (num_kb > 0) {
      if (split) {
        const uint32_t na = S_A_BYTES >> 4, nb = b_bytes >> 4;      // 16-byte granules of the A / B tile
        const uint32_t n16 = na + nb;
        for (int i = 0; i < num_kb; ++i) {
          const int s = i % S;
          const uint32_t ph = (uint32_t)(i / S) & 1u;
          mbarrier_wait<S_SPIN_LOG2>(&full_bar[s], ph);
          uint8_t* st = smem + (size_t)s * stage_bytes;
          for (uint32_t q0 = tid; q0 < n16; q0 += 4 * S_WORKERS) {   // 4 granules in flight per thread
            uint4 v[4];
            uint4* ph_[4];
            uint4* pl_[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const uint32_t q = q0 + u * S_WORKERS;
              const bool ok = q < n16;
              const uint32_t qq = ok ? q : tid;
              const bool isa = qq < na;
              ph_[u] = reinterpret_cast<uint4*>(st + (isa ? 0u : b_hi_off)) + (isa ? qq : qq - na);
              pl_[u] = reinterpret_cast<uint4*>(st + (isa ? a_lo_off : b_lo_off)) + (isa ? qq : qq - na);
              if (!ok) ph_[u] = nullptr;
              v[u] = ok ? *ph_[u] : make_uint4(0, 0, 0, 0);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              if (ph_[u] != nullptr) {
                uint4 h, l;
                split_granule(v[u], h, l);
                if (S_MASK_HI) *ph_[u] = h;
                *pl_[u] = l;
              }
            }
          }
          fence_proxy_async_shared();   // generic writes -> visible to the MMA (async proxy)
          mbarrier_arrive(&conv_bar[s]);
        }
      }
      mbarrier_wait<S_SPIN_LOG2>(tmem_full_bar, 0);
      tcgen05_fence_after();
      const int quarter = warp & 3;                   // TMEM lane quarter this warp may read
      const int half = (warp - 2) >> 2;               // the two warps of a quarter split the columns
      const int rloc = quarter * 32 + lane;
      const int row = m0 + rloc;
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16);
      const uint32_t lo_col = g.lo_col;
      const int nchunk = NT / 16;
      const int c_split = ((nchunk + 1) / 2) * 16;
      const int c_begin = half ? c_split : 0, c_end = half ? NT : c_split;
      // 16 accumulator columns of this thread's row: main (+ cross-term accumulator)
      auto load16 = [&](int c, float (&v)[16]) {
        tcgen05_ld_32x32b_x16(taddr + c, v);
        if (split) {
          float w[16];
          tcgen05_ld_32x32b_x16(taddr + lo_col + c, w);
          tcgen05_wait_ld();
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] += w[j];
        } else {
          tcgen05_wait_ld();
        }
      };

      if (EPI == EPI_STORE) {
        float* crow = nullptr;
        if (row < g.M) crow = row < g.msplit ? g.C0 + (size_t)row * g.ldc : g.C1 + (size_t)(row - g.msplit) * g.ldc;
        for (int c = c_begin; c < c_end; c += 16) {
          float v[16];
          load16(c, v);
          if (crow != nullptr) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int col = n0 + c + j;
              if (col < g.n_store) {
                if (g.atomic) atomicAdd(crow + col, g.alpha * v[j]);
                else crow[col] = g.alpha * v[j];
              }
            }
          }
        }
      } else if (EPI == EPI_GFT) {
        // Stage the tile in shared memory as [b_local][row][t] — with interleaved rows m' = node*3 + k' that IS the layout
        // of G for one batch element (G[b][m'][t], dense) — then write it out with coalesced 16-byte stores.  All MMAs have
        // completed (tmem_full_bar), so the operand ring is free to be reused as the staging buffer.
        const int Nn = g.Nn, W = g.W;
        float* s_out = reinterpret_cast<float*>(smem);
        for (int c = c_begin; c < c_end; c += 16) {
          float v[16];
          load16(c, v);
          int bl = c / W, t = c - bl * W;
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            s_out[(bl * S_BM + rloc) * W + t] = v[j];
            if (++t == W) { t = 0; ++bl; }
          }
        }
        bar_sync<1, 256>();
        const int nv = min(S_BM, g.M - m0);                 // valid rows of this tile
        const int nbl = NT / W;                             // batch elements per tile (NT is a multiple of W)
        const int b0 = n0 / W;
        const bool vec = (W & 3) == 0 && (((size_t)3 * Nn * W) & 3) == 0;
        for (int bl = 0; bl < nbl; ++bl) {
          const int b = b0 + bl;
          if (b * W >= g.BW) break;
          const float* src = s_out + (size_t)bl * S_BM * W;
          if (g.G != nullptr) {
            float* dst = g.G + ((size_t)b * 3 * Nn + m0) * W;
            const int nel = nv * W;
            if (vec) {
              for (int e = tid * 4; e < nel; e += 4 * S_WORKERS)
                *reinterpret_cast<float4*>(dst + e) = *reinterpret_cast<const float4*>(src + e);
            } else {
              for (int e = tid; e < nel; e += S_WORKERS) dst[e] = src[e];
            }
          }
          if (g.g_hi != nullptr) {
            if ((W & 3) == 0 && (g.ldh & 3) == 0) {          // 4 halves = 8 bytes per store
              const int upr = W / 4;                         // units per (row, k') chunk
              for (int it = tid; it < nv * upr; it += S_WORKERS) {
                const int rl = it / upr, u = it - rl * upr;
                const int mp = m0 + rl, node = mp / 3, kp = mp - node * 3;
                const float4 f = *reinterpret_cast<const float4*>(src + rl * W + 4 * u);
                unsigned short h0, h1, h2, h3, l0, l1, l2, l3;
                split_f16_hi_lo(f.x, g.bf16, h0, l0); split_f16_hi_lo(f.y, g.bf16, h1, l1);
                split_f16_hi_lo(f.z, g.bf16, h2, l2); split_f16_hi_lo(f.w, g.bf16, h3, l3);
                const size_t o = ((size_t)b * Nn + node) * g.ldh + kp * W + 4 * u;
                *reinterpret_cast<uint2*>(g.g_hi + o) =
                    make_uint2((uint32_t)h0 | ((uint32_t)h1 << 16), (uint32_t)h2 | ((uint32_t)h3 << 16));
                if (!g.bf16)
                  *reinterpret_cast<uint2*>(g.g_lo + o) =
                      make_uint2((uint32_t)l0 | ((uint32_t)l1 << 16), (uint32_t)l2 | ((uint32_t)l3 << 16));
              }
            } else {
              for (int it = tid; it < nv * W; it += S_WORKERS) {
                const int rl = it / W, t = it - rl * W;
                const int mp = m0 + rl, node = mp / 3, kp = mp - node * 3;
                unsigned short hh, ll;
                split_f16_hi_lo(src[it], g.bf16, hh, ll);
                const size_t o = ((size_t)b * Nn + node) * g.ldh + kp * W + t;
                g.g_hi[o] = hh;
                if (!g.bf16) g.g_lo[o] = ll;
              }
            }
          }
        }
      } else {   // EPI_HEAD
        const int T = g.T, W = g.W;
        const bool valid = row < g.M;
        for (int c = c_begin; c < c_end; c += 16) {
          float v[16];
          load16(c, v);
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int u = c + j;
            if (u < T) {
              const float f = fast_sigmoid(v[j] + s_bf[u]);
              s_fs[u * 128 + rloc] = f;
              if (valid && g.save_fs != nullptr) g.save_fs[(long long)row * T + u] = f;
            } else if (u < T + W) {
              s_pb[(u - T) * 128 + rloc] = v[j];
            }
          }
        }
        const bool has_bc = g.bc_bnw != nullptr;
        if (valid && has_bc && half == 0)
          for (int t = 0; t < W; ++t) s_x[t * 128 + rloc] = g.x_bnw[(long long)row * W + t];
        bar_sync<1, 256>();     // a row's columns were produced by two warps
        if (valid) {
          const int b = row / g.Nn, node = row - b * g.Nn;
          const int o_split = (W + 1) / 2;
          const int o0 = half ? o_split : 0, o1 = half ? W : o_split;   // the two warps of a row split the outputs
          for (int o = o0; o < o1; ++o) {
            float acc = s_bfr[o];
            const float* wr = s_wfr + o * T;
#pragma unroll 4
            for (int u = 0; u < T; ++u) acc = fmaf(s_fs[u * 128 + rloc], wr[u], acc);
            g.forecast[(long long)row * W + o] = acc;
            if (has_bc) {
              float sc = s_bsc[o];
              const float* ws = s_wsc + o * W;
              for (int t = 0; t < W; ++t) sc = fmaf(s_x[t * 128 + rloc], ws[t], sc);
              const float bc = fast_sigmoid(s_pb[o * 128 + rloc] + s_bb[o] - sc);
              g.bc_bnw[(long long)row * W + o] = bc;
              g.bc_bwn[((long long)b * W + o) * g.Nn + node] = bc;
              if (g.bc_pad != nullptr) g.bc_pad[((long long)b * W + o) * g.ld_pad + node] = bc;
            }
          }
        }
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tcgen05_dealloc(tmem_base, g.tmem_cols);
  }
}

uint32_t pow2_cols(int n) {
  uint32_t c = 32;
  while ((int)c < n) c <<= 1;
  return c;
}
// accumulator placement for a tile of NT columns
void plan_tmem(Tc3Args* g) {
  const int NT = g->NT;
  g->stacked = (g->split && 2 * NT <= 256) ? 1 : 0;
  if (!g->split) { g->lo_col = 0; g->tmem_cols = pow2_cols(NT); }
  else if (g->stacked) { g->lo_col = (uint32_t)NT; g->tmem_cols = pow2_cols(2 * NT); }
  else { g->lo_col = pow2_cols(NT); g->tmem_cols = 2 * pow2_cols(NT); }
}

// ring depth and dynamic shared memory for a tile shape; returns 0 stages when it does not fit
int plan_smem(int NT, int split, size_t extra, size_t min_ring, int max_stages, size_t* smem_out) {
  const size_t stage = (size_t)(split ? 2 : 1) * (S_A_BYTES + (size_t)NT * 128);
  const size_t fixed = 1024 /* alignment slack */ + 256 /* barriers + tmem slot */ + extra;
  int s = max_stages;
  while (s >= 2 && fixed + (size_t)s * stage > 227 * 1024) --s;
  if (s < 2 || (size_t)s * stage < min_ring) return 0;
  *smem_out = fixed + (size_t)s * stage;
  return s;
}

template <int EPI>
int launch_tc3(const CUtensorMap& ma, const CUtensorMap& mb, const Tc3Args& g, dim3 grid, size_t smem, cudaStream_t st,
               const char* name) {
  static size_t smem_set_dev[64] = {};   // function attributes are per device
  int dev = 0;
  (void)cudaGetDevice(&dev);
  size_t& smem_set = smem_set_dev[dev & 63];
  if (smem > smem_set) {
    SG_CUDA(cudaFuncSetAttribute(tc3_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  tc3_kernel<EPI><<<grid, S_THREADS, smem, st>>>(ma, mb, g);
  SG_LAUNCH_CHECK(name);
  return 0;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int lcm_i(int a, int b) {
  int x = a, y = b;
  while (y) { const int t = x % y; x = y; y = t; }
  return a / x * b;
}

}  // namespace

// dst[r'][c] = src[r][c] for c < cols (row pitches ld_src / ld_dst): TMA-able (pitch % 4 == 0) copy of an operand, with
// an optional row permutation:  stack_n == 0:  r' = r*row_mul + row_add;   stack_n > 0 (the source is a stack of matrices of
// stack_n rows each, r = k*stack_n + i):  r' = i*row_mul + k + row_add.  (row_mul = 3: the interleaved row order
// node*3 + k' of the graph-Fourier kernel's A operand.)
__global__ void pad_rows_kernel(const float* __restrict__ src, long long rows, int cols, int ld_src,
                                float* __restrict__ dst, int ld_dst, int row_mul, int row_add, int stack_n) {
  const long long total = rows * cols;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long r = idx / cols;
    const int c = (int)(idx - r * cols);
    const long long rd = stack_n > 0 ? (r % stack_n) * row_mul + r / stack_n + row_add : r * row_mul + row_add;
    dst[rd * ld_dst + c] = src[r * ld_src + c];
  }
}
int launch_pad_rows(const float* src, long long rows, int cols, int ld_src, float* dst, int ld_dst, cudaStream_t st,
                    int row_mul, int row_add, int stack_n) {
  const long long total = rows * cols;
  const int blocks = (int)((total + 255) / 256 < 148 * 8 ? (total + 255) / 256 : 148 * 8);
  pad_rows_kernel<<<blocks > 0 ? blocks : 1, 256, 0, st>>>(src, rows, cols, ld_src, dst, ld_dst, row_mul, row_add, stack_n);
  SG_LAUNCH_CHECK("pad_rows_kernel");
  return 0;
}

// generic C0/C1 (+)= alpha A[M,K] B[N,K]^T with split operands (see tc_gemm in glu_tc.cu for the argument meaning)
int tc3_gemm(int M, int N, int K, float alpha, const float* A, int lda, const float* B, int ldb, int n_rows_b, float* C0,
             float* C1, int msplit, int ldc, int n_store, int atomic, int splits, int split_ops, cudaStream_t st) {
  if (N % 16 != 0 || N < 16 || N > 256 || K < 1 || (lda & 3) != 0 || (ldb & 3) != 0) return -1;
  if (!aligned16(A) || !aligned16(B)) return -1;
  CUtensorMap ma, mb;
  if (!make_tensor_map_2d(&ma, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, A, M, K, lda * 4ull, S_BM, S_BK,
                          CU_TENSOR_MAP_SWIZZLE_128B) ||
      !make_tensor_map_2d(&mb, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, B, n_rows_b, K, ldb * 4ull, N, S_BK,
                          CU_TENSOR_MAP_SWIZZLE_128B))
    return -1;
  size_t smem = 0;
  const int ns = plan_smem(N, split_ops, 0, 0, 4, &smem);
  if (ns == 0) return -1;
  Tc3Args g = {};
  g.M = M; g.K = K; g.NT = N; g.nstage = ns; g.split = split_ops;
  plan_tmem(&g);
  g.C0 = C0; g.C1 = C1 != nullptr ? C1 : C0; g.ldc = ldc; g.msplit = C1 != nullptr ? msplit : M;
  g.n_store = n_store; g.atomic = atomic; g.alpha = alpha;
  if (splits < 1) splits = 1;
  return launch_tc3<EPI_STORE>(ma, mb, g, dim3(ceil_div(M, S_BM), 1, splits), smem, st, "tc3_kernel<store>");
}

// gfted rows for the GLU chain: G[(b*N + n)*3W + k'*W + t] = sum_m mul_L[k'+1][n][m] x[b][t][m]  (+ 16-bit images).
// mul_Lp: (3N, ldl) with INTERLEAVED rows, row n*3 + k' = mul_L[k'+1][n][:] (TMA-able pitch); xp: (B*W, ldx).
// Returns -1 when unsupported.
int gft_tc(const float* mul_Lp, int ldl, const float* xp, int ldx, float* G, unsigned short* g_img, int ldh, int bf16,
           int B, int N, int W, int split_ops, cudaStream_t st) {
  static const bool off = getenv("STEMGNN_NO_GFT_TC") != nullptr;
  if (off || mul_Lp == nullptr || xp == nullptr) return -1;
  if ((ldl & 3) != 0 || (ldx & 3) != 0 || !aligned16(mul_Lp) || !aligned16(xp)) return -1;
  if (g_img != nullptr && ((ldh & 1) != 0 || ldh < 3 * W)) return -1;
  // column tile = whole batch elements (the epilogue writes G[b][tile rows][0..W) as one dense block per b)
  const int NT = lcm_i(W, 16);
  if (NT > 128) return -1;
  const int M = 3 * N, BW = B * W;
  CUtensorMap ma, mb;
  if (!make_tensor_map_2d(&ma, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, mul_Lp, M, N, ldl * 4ull, S_BM, S_BK,
                          CU_TENSOR_MAP_SWIZZLE_128B) ||
      !make_tensor_map_2d(&mb, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, xp, BW, N, ldx * 4ull, NT, S_BK,
                          CU_TENSOR_MAP_SWIZZLE_128B))
    return -1;
  size_t smem = 0;
  const int ns = plan_smem(NT, split_ops, 0, (size_t)S_BM * NT * sizeof(float), 4, &smem);   // ring doubles as the staging tile
  if (ns == 0) return -1;
  Tc3Args g = {};
  g.M = M; g.K = N; g.NT = NT; g.nstage = ns; g.split = split_ops;
  plan_tmem(&g);
  g.G = G; g.g_hi = g_img; g.g_lo = g_img != nullptr ? g_img + (size_t)B * N * ldh : nullptr; g.ldh = ldh; g.bf16 = bf16;
  g.Nn = N; g.W = W; g.BW = BW;
  return launch_tc3<EPI_GFT>(ma, mb, g, dim3(ceil_div(M, S_BM), ceil_div(BW, NT), 1), smem, st, "tc3_kernel<gft>");
}

// folded output map + block head in one launch: pre = act3 (R x K) @ woutT (PWp x K)^T stays in tensor memory; the
// epilogue applies base_model.py:68-72.  Returns -1 when the shape does not fit (caller: tc_gemm + block_head_kernel).
int out_head_tc(const float* act3, int K, const float* woutT, int PWp, const HeadArgs& h, float* bc_pad, int ld_pad,
                int split_ops, cudaStream_t st) {
  static const bool off = getenv("STEMGNN_NO_FUSED_HEAD") != nullptr;
  if (off) return -1;
  const int T = h.T, W = h.W, R = h.R;
  if (PWp % 16 != 0 || PWp < 16 || PWp > 256 || (K & 3) != 0 || !aligned16(act3) || !aligned16(woutT)) return -1;
  if (PWp < T + (h.backcast_bnw != nullptr ? W : 0)) return -1;
  CUtensorMap ma, mb;
  if (!make_tensor_map_2d(&ma, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, act3, R, K, K * 4ull, S_BM, S_BK,
                          CU_TENSOR_MAP_SWIZZLE_128B) ||
      !make_tensor_map_2d(&mb, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, woutT, PWp, K, K * 4ull, PWp, S_BK,
                          CU_TENSOR_MAP_SWIZZLE_128B))
    return -1;
  const size_t extra = sizeof(float) * ((size_t)W * T + (size_t)W * W + T + 3 * (size_t)W + (size_t)(T + 2 * W) * 128) + 64;
  size_t smem = 0;
  const int ns = plan_smem(PWp, split_ops, extra, 0, 4, &smem);
  if (ns == 0) return -1;
  Tc3Args g = {};
  g.M = R; g.K = K; g.NT = PWp; g.nstage = ns; g.split = split_ops;
  plan_tmem(&g);
  g.Nn = h.N; g.W = W; g.T = T;
  g.bf = h.bf; g.wfr = h.wfr; g.bfr = h.bfr; g.bb = h.bb; g.wsc = h.wsc; g.bsc = h.bsc;
  g.x_bnw = h.x_bnw; g.forecast = h.forecast; g.bc_bnw = h.backcast_bnw; g.bc_bwn = h.backcast_bwn;
  g.bc_pad = h.backcast_bnw != nullptr ? bc_pad : nullptr; g.ld_pad = ld_pad; g.save_fs = h.save_fs;
  return launch_tc3<EPI_HEAD>(ma, mb, g, dim3(ceil_div(R, S_BM), 1, 1), smem, st, "tc3_kernel<head>");
}

}  // namespace sg
