// GRU recurrence on the 5th-generation tensor cores (reference: models/base_model.py:92,137 and :154-155).
//
// Round-2 rebuild of the dominant kernel (VERDICT r1 item 2).  The recurrence h_s = GRU(x_s, h_{s-1}) is N
// dependent steps of gh = h_{s-1} (G x N) . W_hh^T (N x 3N).  Design:
//   * one thread-block cluster of CS CTAs per group of G <= 8 sequences; CTA q owns U = N/CS (multiple of 8, <= 40)
//     hidden units = 3U <= 120 rows of W_hh, which stay resident in shared memory for all N steps as the
//     tcgen05 A operand (K-major, 128B-swizzled) — W_hh is read from HBM/L2 exactly once per cluster;
//   * fp32 parity on fp16 tensor cores by operand splitting: x = hi + 2^-11 lo with hi = fp16(x),
//     lo = fp16((x - hi) 2^11)  (22 significant bits; h is in (-1,1), weights are far inside the fp16 range).
//     The B operand tile stacks [h_hi (8 rows) ; h_lo (8 rows)] so ONE M128 x N16 x K16 instruction yields both
//     W.h_hi and W.h_lo; two instructions per 16 hidden units (A = W_hi, A = W_lo) give all four partial
//     products: gh = D00 + 2^-11 (D01 + D10) + 2^-22 D11, accumulated in fp32 in tensor memory;
//   * the input projection W_ih x_s + b_ih is computed in-kernel by the gate threads while the MMAs run
//     (36 FMAs per unit-step): the (N.B x 3N) `gi` round trip of round 1 (49 MB written + read) is gone;
//   * per step: MMA thread waits for the h tile (mbarrier) -> 2 x ceil(N/16) tcgen05.mma -> tcgen05.commit;
//     4 epilogue warps: tcgen05.ld -> combine the 4 partials -> smem -> gate math (one thread per (unit, sequence),
//     h / key / query kept in registers) -> fp16 hi/lo split -> 16-byte st.async stores through DSMEM into every
//     cluster CTA's next B tile (already in the swizzled layout the tensor core reads), each signalling the
//     destination's mbarrier.  No cluster barrier on the critical path.
//   * the fp16 hi/lo images of the W_hh slices are produced by gru_pack_whh_kernel (skipped when the caller
//     says the parameters are unchanged) and arrive with cp.async.bulk.
// Envelope: N <= 16*40 with (U, CS) such that the tiles fit 227 KB (N <= 448), W <= 64, G <= 8; everything else
// takes the FFMA2 cluster kernel / per-step path of gru.cu.
#include <cooperative_groups.h>
#include <stdlib.h>

#include "common.cuh"
#include "internal.cuh"
#include "sm100.cuh"

namespace cg = cooperative_groups;

namespace sg {

namespace {

constexpr int GT_ROUNDS = 3;           // MMA warps: warp r consumes the r-th third of the arriving h slices
constexpr int GT_THREADS = (GT_ROUNDS + 4) * 32;   // warps 0..2: MMA issue (warp 0 also allocates TMEM); 4 epilogue warps
constexpr int GT_EPI = 128;
constexpr int GT_GMAX = 8;             // sequences per cluster (rows 0..7 of the B tile = h_hi, 8..15 = h_lo)
constexpr uint32_t GT_TMEM_COLS = 512;    // D (32 columns) + the resident W_hh hi/lo operand
constexpr float GT_LO_INV = 1.0f / F16_LO_SCALE;
constexpr float GT_LO_INV2 = 1.0f / (F16_LO_SCALE * F16_LO_SCALE);
constexpr int GT_SPIN_LOG2 = 24;       // mbarrier polls before a lost signal traps

// kind::f16 instruction descriptor: fp16 A and B, fp32 accumulate, both K-major, M=128, N=16
constexpr uint32_t GT_IDESC = umma_idesc_m128(UMMA_F16, 16);

// byte offset of element (row, k) inside a K-major SWIZZLE_128B fp16 operand whose 64-column chunks are
// `chunk_bytes` apart (16-byte granule index XOR row%8; the tile base is 1024-byte aligned)
__host__ __device__ __forceinline__ uint32_t sw128_off(int row, int k, uint32_t chunk_bytes) {
  const int c = k >> 6, kk = k & 63;
  return (uint32_t)c * chunk_bytes + (uint32_t)row * 128u + (uint32_t)((((kk >> 3) ^ (row & 7)) << 4) + ((kk & 7) << 1));
}

struct GruTcGeom {
  int U;          // hidden units per CTA (multiple of 8, <= 40)
  int CS;         // cluster size
  int NCH;        // 64-column K chunks of the B tile = ceil(CS*U / 64)
  int NKS;        // K steps of 16 = ceil(CS*U / 16)
};
// per-CTA W_hh image (global): uint4 index ((arr * 2 NKS + kg) * 128 + row), arr = hi/lo, kg = k / 8
__host__ __device__ inline uint32_t a_img_bytes(const GruTcGeom& g) { return (uint32_t)g.NKS * 8192u; }
constexpr uint32_t B_CHUNK_BYTES = 16 * 128;     // 16 rows (8 hi + 8 lo) x 64 fp16
constexpr uint32_t GT_TMEM_A0 = 32 * GT_ROUNDS;  // first TMEM column of the resident W_hh operand (accumulator set r: columns 32r..32r+31)

// ---- pack: W_hh (3N, N) fp32 -> per-CTA fp16 hi/lo images in the order the TMEM fill reads them ----------------
// one thread = (row = gate*U + lu, 8 consecutive k): the 8 halves of a uint4 are 4 TMEM columns (2 fp16 each)
__global__ void __launch_bounds__(128) gru_pack_whh_kernel(const float* __restrict__ w_hh, uint4* __restrict__ img,
                                                            int N, GruTcGeom g) {
  const int q = blockIdx.y, kg = blockIdx.x, row = threadIdx.x;
  float v[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = 0.f;
  if (row < 3 * g.U) {
    const int gate = row / g.U, lu = row - gate * g.U;
    const int u = q * g.U + lu;
    if (u < N) {
      const float* src = w_hh + ((size_t)gate * N + u) * N + 8 * kg;
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (8 * kg + i < N) v[i] = __ldg(src + i);
    }
  }
  uint32_t hi[4], lo[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    unsigned short h0, l0, h1, l1;
    split_f16_hi_lo_scaled(v[2 * i], h0, l0);
    split_f16_hi_lo_scaled(v[2 * i + 1], h1, l1);
    hi[i] = (uint32_t)h0 | ((uint32_t)h1 << 16);
    lo[i] = (uint32_t)l0 | ((uint32_t)l1 << 16);
  }
  uint4* base = img + (size_t)q * (a_img_bytes(g) / 16);
  base[(size_t)kg * 128 + row] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  base[(size_t)(2 * g.NKS + kg) * 128 + row] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}

struct GruTcArgs {
  GruArgs a;
  const uint4* img;       // packed W_hh images, one per cluster rank
  GruTcGeom g;
  int G;                  // sequences per cluster
  int x_smem;             // 1: the cluster's x rows are staged in shared memory by bulk copies
  int pipelined;          // 1: MMAs of a K range start as soon as its source CTAs' slices landed
  long long* dbg;         // optional clock64 stamps (STEMGNN_GRU_TC_DBG), null in production
  int dbg_mode;           // 1 both, 2 epilogue stamps only, 3 MMA-warp stamps only
};
// stamps are taken under a WARP-UNIFORM condition and the warp is re-converged right after: a lane that diverges in front of
// elect.sync / tcgen05.ld.sync.aligned breaks those warp-collective instructions (seen as wrong results in early debug builds)
#define GT_STAMP(slot) do { if (dbg_on) { if (lane == 0) ta.dbg[(s - dbg_s0) * 16 + (slot)] = clock64(); __syncwarp(); } } while (0)

// PP = (unit, sequence) pairs per epilogue thread
template <int PP>
__global__ void __launch_bounds__(GT_THREADS, 1) gru_tc_cluster_kernel(GruTcArgs ta) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + smem_pad1024(smem_raw);
  const GruArgs& a = ta.a;
  const GruTcGeom g = ta.g;
  const int U = g.U, CS = g.CS, G = ta.G;
  const int N = a.N, B = a.B, W = a.W;
  const uint32_t b_buf = (uint32_t)g.NCH * B_CHUNK_BYTES;

  uint8_t* B_sm = smem;                                   // [2][NCH][16][128]  h tiles: rows 0..7 hi, 8..15 lo
  float* gh_sm = reinterpret_cast<float*>(B_sm + 2 * b_buf);          // [128][8]
  float* wih_sm = gh_sm + 128 * GT_GMAX;                  // [3U][W]
  float* bias_sm = wih_sm + 3 * U * W;                    // [3U] b_ih (+ b_hh for r,z) and [U] b_hn
  unsigned short* stage_sm = reinterpret_cast<unsigned short*>(bias_sm + 4 * U);      // [2][8][U] (16-byte aligned: U % 8 == 0)
  uint8_t* hbar_base = reinterpret_cast<uint8_t*>(stage_sm + 2 * GT_GMAX * U);
  hbar_base += (8u - (smem_u32(hbar_base) & 7u)) & 7u;
  uint64_t* hbar = reinterpret_cast<uint64_t*>(hbar_base);
  uint64_t* tfull = hbar + 2 * 16;                        // hbar[buf][source]
  uint64_t* xbar = tfull + GT_ROUNDS;                     // tfull[r]: accumulator set r complete
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(xbar + 1);
  uint32_t* rdy_sm = tmem_slot + 2;                       // [16] rdy[r]: K steps of round r, rdy[8 + r]: last arrival index of round r
  uint8_t* xs_base = reinterpret_cast<uint8_t*>(rdy_sm + 16);
  xs_base += (16u - (smem_u32(xs_base) & 15u)) & 15u;
  float* xs_sm = reinterpret_cast<float*>(xs_base);       // [N][G][W]

  cg::cluster_group cluster = cg::this_cluster();
  const int q = (int)cluster.block_rank();
  const int cid = blockIdx.x / CS;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int u0 = q * U;
  const int b0 = cid * G;
  const int nb = min(G, B - b0);                          // real sequences of this cluster

  // ---- one-time setup ------------------------------------------------------------------------------------
  if (tid == 0) {
    for (int i = 0; i < 2 * 16; ++i) mbarrier_init(&hbar[i], 1);
    for (int r = 0; r < GT_ROUNDS; ++r) mbarrier_init(&tfull[r], 1);   // tfull[0] is re-initialised below with the round count
    mbarrier_init(xbar, 1);
    fence_mbarrier_init();
  }
  if (warp == 0) {
    tcgen05_alloc(tmem_slot, GT_TMEM_COLS);
    tcgen05_relinquish_alloc_permit();
  }
  // B tiles (both buffers) start as zeros: h_{-1} = 0, padding columns / unused sequence rows stay zero forever
  for (int i = tid; i < (int)(2 * b_buf / 16); i += GT_THREADS)
    reinterpret_cast<uint4*>(B_sm)[i] = make_uint4(0u, 0u, 0u, 0u);
  for (int i = tid; i < 3 * U * W; i += GT_THREADS) {
    const int row = i / W, t = i - row * W;
    const int gate = row / U, lu = row - gate * U;
    const int u = u0 + lu;
    wih_sm[i] = u < N ? __ldg(a.w_ih + ((size_t)gate * N + u) * W + t) : 0.f;
  }
  for (int i = tid; i < 4 * U; i += GT_THREADS) {
    const int gate = i / U, lu = i - gate * U;
    const int u = u0 + lu;
    float v = 0.f;
    if (u < N) {
      if (gate < 2) v = __ldg(a.b_ih + gate * N + u) + __ldg(a.b_hh + gate * N + u);
      else if (gate == 2) v = __ldg(a.b_ih + 2 * N + u);
      else v = __ldg(a.b_hh + 2 * N + u);
    }
    bias_sm[i] = v;
  }
  if (ta.x_smem) {                     // the cluster's input rows x[s][b0 .. b0+nb) -> smem (16-byte loads, W % 4 == 0)
    const int rowv = nb * W / 4, pitch = G * W / 4;
    const float4* src = reinterpret_cast<const float4*>(a.xs);
    float4* dst = reinterpret_cast<float4*>(xs_sm);
    for (int idx = tid; idx < N * rowv; idx += GT_THREADS) {
      const int ss = idx / rowv, v = idx - ss * rowv;
      dst[(size_t)ss * pitch + v] = __ldg(src + ((size_t)ss * B + b0) * (W / 4) + v);
    }
  }
  fence_proxy_async_shared();                 // generic-proxy zero fill -> visible to the tensor core's async proxy
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t a_cols = (uint32_t)g.NKS * 8u;            // TMEM columns per W_hh array (2 fp16 per column)

  if (warp == 0) {
    if (lane < GT_ROUNDS) {            // round r consumes the slices with arrival index <= last(r); it owns the K steps
      const int R = min(GT_ROUNDS, CS);  // that become complete with them (arrival index of source p here: (q - p) mod CS)
      uint32_t mask = 0;
      int last = -1, prev_last = -1;
      if (lane < R) {
        // even split: a step is bound by the tensor pipe (2 NKS instructions at ~22 cycles) once the first slices are in, so the
        // rounds only need to start early; what matters is that round 0 can begin after a third of the arrivals
        auto last_of = [&](int rr) { return ((rr + 1) * CS + R - 1) / R - 1; };
        last = last_of(lane);
        prev_last = lane == 0 ? -1 : last_of(lane - 1);
        if (!ta.pipelined) { last = lane == 0 ? CS - 1 : -1; prev_last = lane == 0 ? -1 : CS; }
        for (int j = 0; j < g.NKS; ++j) {
          const int p0 = (16 * j) / U, p1 = min((16 * j + 15) / U, CS - 1);
          const int need = max((q - p0 + CS) % CS, (q - p1 + CS) % CS);
          if (need <= last && need > prev_last) mask |= 1u << j;
        }
      }
      rdy_sm[lane] = mask;
      rdy_sm[8 + lane] = (uint32_t)last;
      const uint32_t nz = __ballot_sync((1u << GT_ROUNDS) - 1u, mask != 0u);
      if (lane == 0) {                 // ONE accumulator barrier: every non-empty round commits to it once per step
        rdy_sm[12] = (uint32_t)__popc(nz);
        if (nz != 0u) {
          mbarrier_inval(&tfull[0]);
          mbarrier_init(&tfull[0], (uint32_t)__popc(nz));
          fence_mbarrier_init();
        }
      }
    }
    __syncwarp();
  } else if (warp >= GT_ROUNDS) {
    // W_hh slice -> tensor memory (A operand, resident for all N steps): lane = row, 8 columns = 16 k per store
    const int row = (warp & 3) * 32 + lane;
    (void)row;
    const uint32_t tA = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + GT_TMEM_A0;
    const uint4* src = ta.img + (size_t)q * (a_img_bytes(g) / 16) + row;
    const int nst = 2 * g.NKS;         // [hi: NKS stores][lo: NKS stores], store i covers kg = 2i, 2i+1
#pragma unroll 4
    for (int i = 0; i < nst; ++i) {
      const uint4 v0 = __ldg(src + (size_t)(2 * i) * 128);
      const uint4 v1 = __ldg(src + (size_t)(2 * i + 1) * 128);
      tcgen05_st_32x32b_x8(tA + (uint32_t)i * 8u, v0, v1);
    }
    tcgen05_wait_st();
  }
  tcgen05_fence_before();
  cluster.sync();                      // every CTA's tiles and barriers exist before any remote store
  tcgen05_fence_after();

  const uint32_t src_bytes = (uint32_t)(2 * G * U * 2);    // bytes a CTA receives per step from ONE source CTA

  if (warp < GT_ROUNDS) {
    // ===================== MMA issuers =====================
    // Warp r waits for the slices of its round (lanes wait on different source barriers in parallel), then ONE elected lane
    // makes them visible to the tensor core (fence.proxy.async: the st.async stores are generic-proxy writes and the fence
    // must be executed by the issuing thread itself) and issues the K steps of the round into accumulator set r.
    // * the whole warp runs the loop converged: under `if (lane == 0)` the compiler cannot prove the operands warp-uniform
    //   and wraps every tcgen05.mma in an ELECT/R2UR waterfall loop — 170-260 cycles per instruction against ~20 with
    //   elect.sync (tools/probe/mma_probe.cu, profiles/README.md);
    // * one issuing warp per round: a proxy fence executed by a thread drains the MMAs that thread has in flight, so a
    //   single issuer would serialise arrival -> fence -> MMAs for every round.
    __syncwarp();
    const int r = warp;
    const uint32_t todo0 = rdy_sm[r];
    const int last = (int)rdy_sm[8 + r];
    const int my_p = (q - lane + 16 * CS) % CS;           // source whose slice has arrival index `lane` here
    const int dbg_s0 = N / 2;
    const uint32_t a_hi = tmem_base + GT_TMEM_A0, a_lo = a_hi + a_cols;
    const uint32_t d0 = tmem_base + 32u * (uint32_t)r;
    if (todo0 != 0u) {
      for (int s = 1; s < N; ++s) {
        const int cur = s & 1;
        const uint32_t par = (uint32_t)((s - 1) >> 1) & 1u;
        const bool dbg_on = ta.dbg != nullptr && ta.dbg_mode != 2 && blockIdx.x == 0 && r == GT_ROUNDS - 1 && s >= dbg_s0 && s < dbg_s0 + 4;
        GT_STAMP(0);
        if (lane <= last) {
          // plain (cta-scope) acquire: the cluster-scope form makes ptxas add CCTL.IVALL (an L1 invalidate, 8 % of the
          // kernel's stall samples in profiles/r02_ncu_gru_tc_stalls.txt) although the payload lives in shared memory
          mbarrier_wait<GT_SPIN_LOG2>(&hbar[cur * 16 + my_p], par);                      // slices of h_{s-1} landed in B[cur]
          fence_proxy_async_shared();         // every observer orders the remote generic-proxy stores before async-proxy reads
        }
        __syncwarp();
        GT_STAMP(1);
        if (elect_one_sync()) {
          fence_proxy_async_shared();
          tcgen05_fence_after();
          const uint32_t b_addr = smem_u32(B_sm) + (uint32_t)cur * b_buf;
          uint32_t todo = todo0, acc = 0u;
          while (todo) {
            const int j = __ffs((int)todo) - 1;
            todo &= todo - 1u;
            const uint64_t bd = umma_desc_kmajor(b_addr + (uint32_t)(j >> 2) * B_CHUNK_BYTES + (uint32_t)(j & 3) * 32u, 1024,
                                                 UMMA_SWIZZLE_128B);
            tcgen05_mma_f16_tmem_a(d0, a_hi + (uint32_t)j * 8u, bd, GT_IDESC, acc);           // W_hi . [h_hi | h_lo]
            tcgen05_mma_f16_tmem_a(d0 + 16u, a_lo + (uint32_t)j * 8u, bd, GT_IDESC, acc);     // W_lo . [h_hi | h_lo]
            acc = 1u;
          }
          tcgen05_commit(&tfull[0]);
        }
        __syncwarp();
        GT_STAMP(3);
      }
    }
    __syncwarp();                      // reconverged before the aligned cluster barrier below
  } else {
    // ===================== epilogue: TMEM -> gates -> DSMEM sends =====================
    const int et = tid - 32 * GT_ROUNDS;           // 0..127
    const int quarter = warp & 3;                  // TMEM lane quarter this warp may read
    const int row = quarter * 32 + lane;           // accumulator row = TMEM lane = gate*U + lu
    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16);

    // (unit, sequence) pairs of this thread: pair p = et + 128 i -> b = p / U, lu = p % U
    int p_lu[PP], p_b[PP];
    bool p_ok[PP], p_real[PP];
    float hprev[PP], key_acc[PP], query_acc[PP], gi_r[PP], gi_z[PP], gi_n[PP];
#pragma unroll
    for (int i = 0; i < PP; ++i) {
      const int p = et + GT_EPI * i;
      p_b[i] = p / U;
      p_lu[i] = p - p_b[i] * U;
      p_ok[i] = p < U * G;                                              // pair exists in this cluster
      p_real[i] = p_ok[i] && (u0 + p_lu[i]) < N && (b0 + p_b[i]) < B;   // real unit and real sequence
      hprev[i] = key_acc[i] = query_acc[i] = 0.f;
    }
    auto input_proj = [&](int s, int i, float& r, float& z, float& n) {
      r = z = n = 0.f;
      if (p_real[i]) {
        const float* wr = wih_sm + (size_t)p_lu[i] * W;
        const float* wz = wr + (size_t)U * W;
        const float* wn = wz + (size_t)U * W;
        r = bias_sm[p_lu[i]];
        z = bias_sm[U + p_lu[i]];
        n = bias_sm[2 * U + p_lu[i]];
        if (ta.x_smem) {                     // W % 4 == 0: rows of x and W_ih are 16-byte aligned
          const float4* xp = reinterpret_cast<const float4*>(xs_sm + ((size_t)s * G + p_b[i]) * W);
          const float4* r4 = reinterpret_cast<const float4*>(wr);
          const float4* z4 = reinterpret_cast<const float4*>(wz);
          const float4* n4 = reinterpret_cast<const float4*>(wn);
          for (int t = 0; t < (W >> 2); ++t) {
            const float4 xv = xp[t], a4 = r4[t], b4 = z4[t], c4 = n4[t];
            r = fmaf(a4.x, xv.x, r); r = fmaf(a4.y, xv.y, r); r = fmaf(a4.z, xv.z, r); r = fmaf(a4.w, xv.w, r);
            z = fmaf(b4.x, xv.x, z); z = fmaf(b4.y, xv.y, z); z = fmaf(b4.z, xv.z, z); z = fmaf(b4.w, xv.w, z);
            n = fmaf(c4.x, xv.x, n); n = fmaf(c4.y, xv.y, n); n = fmaf(c4.z, xv.z, n); n = fmaf(c4.w, xv.w, n);
          }
        } else {
          const float* xp = a.xs + ((size_t)s * B + (b0 + p_b[i])) * W;
          for (int t = 0; t < W; ++t) {
            const float xv = __ldg(xp + t);
            r = fmaf(wr[t], xv, r);
            z = fmaf(wz[t], xv, z);
            n = fmaf(wn[t], xv, n);
          }
        }
      }
    };
#pragma unroll
    for (int i = 0; i < PP; ++i) input_proj(0, i, gi_r[i], gi_z[i], gi_n[i]);

    // step-invariant send descriptors.  A granule = 8 consecutive units of one sequence in one array (hi / lo) = 16 bytes of
    // the destination's B tile.  Pair p = et + 128 i maps 8-aligned groups of lanes to granules (U % 8 == 0), so every granule
    // is produced inside ONE warp: the warp that computed it sends it to all CS CTAs after a __syncwarp — no block-wide
    // barrier between the gate math and the sends.  Per (warp, i): 4 lane groups x 2 arrays = 8 granules x CS destinations,
    // visited slot-major in the rotated order (q + slot) % CS so that the slices a CTA receives arrive staggered.
    constexpr int SEND_K = (8 * 16 + 31) / 32;               // sends per lane per i (CS <= 16)
    uint32_t snd_src[PP][SEND_K], snd_dst[PP][SEND_K], snd_bar[PP][SEND_K];
#pragma unroll
    for (int i = 0; i < PP; ++i) {
#pragma unroll
      for (int k = 0; k < SEND_K; ++k) {
        const int j = lane + 32 * k;
        const int slot = j >> 3, gran = j & 7;
        const int arr = gran >> 2;
        const int p0 = 32 * (warp - GT_ROUNDS) + GT_EPI * i + 8 * (gran & 3);     // first pair of the lane group
        snd_src[i][k] = 0xFFFFFFFFu;
        snd_dst[i][k] = snd_bar[i][k] = 0;
        if (slot < CS && p0 < U * G) {
          const int bb = p0 / U, lu0 = p0 - bb * U;
          const int dest = (q + slot) % CS;
          snd_src[i][k] = (uint32_t)(((arr * GT_GMAX + bb) * U + lu0) * 2);                 // bytes into stage_sm
          const uint32_t off = sw128_off(arr * 8 + bb, u0 + lu0, B_CHUNK_BYTES);
          snd_dst[i][k] = mapa_shared_cluster(smem_u32(B_sm) + off, (uint32_t)dest);
          snd_bar[i][k] = mapa_shared_cluster(smem_u32(&hbar[q]), (uint32_t)dest);    // the destination's barrier for source q
        }
      }
    }
    float wk_s = __ldg(a.wk + 0), wq_s = __ldg(a.wq + 0);

    const int dbg_s0 = N / 2;
    for (int s = 0; s < N; ++s) {
      const int nxt = (s & 1) ^ 1;
      const bool dbg_on = ta.dbg != nullptr && ta.dbg_mode != 3 && blockIdx.x == 0 && warp == GT_ROUNDS && s >= dbg_s0 && s < dbg_s0 + 4;
      GT_STAMP(4);
      if (et < CS && s + 1 < N) mbarrier_arrive_expect_tx(&hbar[nxt * 16 + et], src_bytes);   // arm the tile that will receive h_s
      // input projection of the NEXT step while this step's MMAs run
      float nx_r[PP] = {}, nx_z[PP] = {}, nx_n[PP] = {}, nx_wk = 0.f, nx_wq = 0.f;
      if (s + 1 < N) {
        nx_wk = __ldg(a.wk + s + 1);
        nx_wq = __ldg(a.wq + s + 1);
#pragma unroll
        for (int i = 0; i < PP; ++i) input_proj(s + 1, i, nx_r[i], nx_z[i], nx_n[i]);
      }
      GT_STAMP(5);
      if (s > 0) {
        // accumulator set r (columns 32r..): cols 0..7 W_hi.h_hi, 8..15 W_hi.h_lo, 16..23 W_lo.h_hi, 24..31 W_lo.h_lo of the
        // K steps of round r;  gh[b] = sum_r D00 + 2^-11 (D01 + D10) + 2^-22 D11
        float o[8];
#pragma unroll
        for (int b = 0; b < 8; ++b) o[b] = 0.f;
        mbarrier_wait<GT_SPIN_LOG2>(&tfull[0], (uint32_t)(s - 1) & 1u);      // every round's MMAs of this step are complete
        tcgen05_fence_after();
        GT_STAMP(6);
        // all accumulator sets are loaded back to back and waited for once: three dependent load -> wait round trips
        // measured ~430 cycles (profiles/r02_gru_phase_stamps.txt)
        float d[GT_ROUNDS][32];
#pragma unroll
        for (int r = 0; r < GT_ROUNDS; ++r) tcgen05_ld_32x32b_x32(taddr + 32u * (uint32_t)r, d[r]);
        tcgen05_wait_ld();
#pragma unroll
        for (int r = 0; r < GT_ROUNDS; ++r) {
          if (rdy_sm[r] != 0u) {             // a round without K steps never wrote its set
#pragma unroll
            for (int b = 0; b < 8; ++b)
              o[b] += d[r][b] + (d[r][8 + b] + d[r][16 + b]) * GT_LO_INV + d[r][24 + b] * GT_LO_INV2;
          }
        }
        GT_STAMP(7);
        float4* gp = reinterpret_cast<float4*>(gh_sm + row * GT_GMAX);
        gp[0] = make_float4(o[0], o[1], o[2], o[3]);
        gp[1] = make_float4(o[4], o[5], o[6], o[7]);
        tcgen05_fence_before();             // the next step's MMAs (ordered after this thread's sends) overwrite D
        bar_sync<1, 128>();
        GT_STAMP(8);
      }
#pragma unroll
      for (int i = 0; i < PP; ++i) {
        if (p_ok[i]) {
          const int lu = p_lu[i], bb = p_b[i];
          float hn = 0.f;
          if (p_real[i]) {
            float gh_r = 0.f, gh_z = 0.f, gh_n = 0.f;
            if (s > 0) {
              gh_r = gh_sm[lu * GT_GMAX + bb];
              gh_z = gh_sm[(U + lu) * GT_GMAX + bb];
              gh_n = gh_sm[(2 * U + lu) * GT_GMAX + bb];
            }
            const float bhn = bias_sm[3 * U + lu];
            const float r = fast_sigmoid(gi_r[i] + gh_r);
            const float zt = fast_sigmoid(gi_z[i] + gh_z);
            const float nt = fast_tanh(gi_n[i] + r * (gh_n + bhn));
            hn = (1.f - zt) * nt + zt * hprev[i];
            key_acc[i] = fmaf(hn, wk_s, key_acc[i]);
            query_acc[i] = fmaf(hn, wq_s, query_acc[i]);
            if (a.h_all != nullptr) {
              const size_t o = ((size_t)s * B + (b0 + bb)) * N + u0 + lu;
              a.h_all[o] = hn;
              if (a.g_r != nullptr) {
                a.g_r[o] = r; a.g_z[o] = zt; a.g_n[o] = nt; a.g_hn[o] = gh_n + bhn;
              }
            }
            hprev[i] = hn;
          }
          unsigned short hi, lo;
          split_f16_hi_lo_scaled(hn, hi, lo);
          stage_sm[(0 * GT_GMAX + bb) * U + lu] = hi;
          stage_sm[(1 * GT_GMAX + bb) * U + lu] = lo;
        }
        gi_r[i] = nx_r[i]; gi_z[i] = nx_z[i]; gi_n[i] = nx_n[i];
      }
      wk_s = nx_wk; wq_s = nx_wq;
      GT_STAMP(9);
      if (s + 1 < N) {
        __syncwarp();                  // the granules this warp sends were staged by its own lanes
        GT_STAMP(10);
        const uint32_t dst_off = (uint32_t)nxt * b_buf, bar_off = (uint32_t)nxt * 16u * 8u;
#pragma unroll
        for (int k = 0; k < SEND_K; ++k) {
#pragma unroll
          for (int i = 0; i < PP; ++i) {
            if (snd_src[i][k] != 0xFFFFFFFFu) {
              const uint4 v = *reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(stage_sm) + snd_src[i][k]);
              st_async_v4(snd_dst[i][k] + dst_off, v, snd_bar[i][k] + bar_off);
            }
          }
        }
        __syncwarp();                  // stage entries are rewritten by the next step's gate phase of this warp
      }
      GT_STAMP(11);
    }
#pragma unroll
    for (int i = 0; i < PP; ++i) {
      if (p_real[i]) {
        a.key[(size_t)(b0 + p_b[i]) * N + u0 + p_lu[i]] = key_acc[i];
        a.query[(size_t)(b0 + p_b[i]) * N + u0 + p_lu[i]] = query_acc[i];
      }
    }
  }
  tcgen05_fence_before();
  cluster.sync();      // no CTA may exit while peers could still address its shared memory
  if (warp == 0) {
    tcgen05_fence_after();
    tcgen05_dealloc(tmem_base, GT_TMEM_COLS);
  }
}

size_t gru_tc_smem_fixed(const GruTcGeom& g, int W) {
  size_t b = 2 * (size_t)g.NCH * B_CHUNK_BYTES;
  b += (size_t)128 * GT_GMAX * 4 + (size_t)3 * g.U * W * 4 + (size_t)4 * g.U * 4 + (size_t)2 * GT_GMAX * g.U * 2;
  b += 8 + (2 * 16 + GT_ROUNDS + 1) * 8 + 8 + 16 * 4 + 16;
  return b + 1024;     // alignment slack
}

bool pick_geom(int N, int W, GruTcGeom* out) {
  static const int cands[] = {40, 32, 24, 16, 8};
  for (int U : cands) {
    const int CS = ceil_div(N, U);
    if (CS > 16) continue;
    GruTcGeom g;
    g.U = U; g.CS = CS; g.NCH = ceil_div(CS * U, 64); g.NKS = ceil_div(CS * U, 16);
    if (GT_TMEM_A0 + 2 * g.NKS * 8 > 512) continue;          // both W_hh arrays must fit the 512 TMEM columns
    if (gru_tc_smem_fixed(g, W) > 227 * 1024) continue;
    *out = g;
    return true;
  }
  return false;
}

struct PerDev { bool set[3]; int max_clusters[3]; size_t smem[3]; int cs[3]; };
PerDev g_dev[64];

template <int PP>
int launch_tc(const GruTcArgs& ta, size_t smem, cudaStream_t st, int* max_clusters_out, bool probe_only) {
  auto kern = gru_tc_cluster_kernel<PP>;
  int dev = 0;
  SG_CUDA(cudaGetDevice(&dev));
  PerDev& pd = g_dev[dev & 63];
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(GT_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = ta.g.CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  const int slot = PP - 1;
  if (!pd.set[slot] || pd.smem[slot] < smem || pd.cs[slot] != ta.g.CS) {
    SG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (ta.g.CS > 8) SG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cfg.gridDim = dim3(ta.g.CS);
    int mc = 0;
    cudaError_t e = cudaOccupancyMaxActiveClusters(&mc, kern, &cfg);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      mc = 0;
    }
    pd.set[slot] = true; pd.smem[slot] = smem; pd.cs[slot] = ta.g.CS; pd.max_clusters[slot] = mc;
  }
  *max_clusters_out = pd.max_clusters[slot];
  if (pd.max_clusters[slot] < 1) return -1;
  if (probe_only) return 0;
  const int nclusters = ceil_div(ta.a.B, ta.G);
  cfg.gridDim = dim3(nclusters * ta.g.CS);
  ProfileHook* hook = profile_hook();
  if (hook->start != nullptr) SG_CUDA(cudaEventRecord(hook->start, st));
  SG_CUDA(cudaLaunchKernelEx(&cfg, kern, ta));
  if (hook->stop != nullptr) SG_CUDA(cudaEventRecord(hook->stop, st));
  count_launch();
  return 0;
}

}  // namespace

size_t gru_tc_image_bytes(int N, int W) {
  GruTcGeom g;
  if (!pick_geom(N, W, &g)) return 0;
  return (size_t)g.CS * a_img_bytes(g);
}

// returns 0 launched, -1 outside the envelope / not launchable here (caller falls back), >0 error
int gru_tc_forward(const GruArgs& a, uint8_t* img, int reuse_img, cudaStream_t st) {
  static const bool off = getenv("STEMGNN_GRU_NO_TC") != nullptr;
  if (off || img == nullptr) return -1;
  if (a.W > 64 || a.N < 1) return -1;
  GruTcGeom g;
  if (!pick_geom(a.N, a.W, &g)) return -1;
  if ((reinterpret_cast<uintptr_t>(img) & 15) != 0) return -1;
  GruTcArgs ta;
  ta.a = a; ta.img = reinterpret_cast<const uint4*>(img); ta.g = g; ta.G = 1; ta.dbg = nullptr;
  static const bool no_pipe = getenv("STEMGNN_GRU_TC_NOPIPE") != nullptr;
  ta.pipelined = no_pipe ? 0 : 1;
  ta.x_smem = 0;
  static const bool dbg = getenv("STEMGNN_GRU_TC_DBG") != nullptr;
  ta.dbg_mode = dbg ? atoi(getenv("STEMGNN_GRU_TC_DBG")) : 0;
  static long long* dbg_buf = nullptr;
  if (dbg) {
    if (dbg_buf == nullptr) SG_CUDA(cudaMalloc(&dbg_buf, 64 * sizeof(long long)));
    SG_CUDA(cudaMemsetAsync(dbg_buf, 0, 64 * sizeof(long long), st));
    ta.dbg = dbg_buf;
  }
  // sequences per cluster: as few as one wave of resident clusters allows (<= 8), overridable for measurements.
  // The occupancy probe uses the fixed part of the shared memory (the x staging area is optional).
  const size_t smem_fixed = gru_tc_smem_fixed(g, a.W);
  int mc = 0;
  int rc = launch_tc<1>(ta, smem_fixed, st, &mc, true);
  if (rc != 0) return rc;
  int G = ceil_div(a.B, mc);
  if (const char* e = getenv("STEMGNN_GRU_TC_G")) G = atoi(e) > 0 ? atoi(e) : G;
  if (G > GT_GMAX) G = GT_GMAX;
  if (G < 1) G = 1;
  ta.G = G;
  size_t smem = smem_fixed;
  const size_t x_bytes = (size_t)a.N * G * a.W * 4;
  static const bool no_xs = getenv("STEMGNN_GRU_TC_NOXSMEM") != nullptr;
  if (!no_xs && (a.W & 3) == 0 && (reinterpret_cast<uintptr_t>(a.xs) & 15) == 0 && smem_fixed + x_bytes + 16 <= 227 * 1024 &&
      x_bytes < (1u << 20)) {
    ta.x_smem = 1;
    smem = smem_fixed + x_bytes + 16;
  }
  const int pp = ceil_div(g.U * G, GT_EPI);
  if (!reuse_img) {
    dim3 grid(2 * g.NKS, g.CS);
    gru_pack_whh_kernel<<<grid, 128, 0, st>>>(a.w_hh, reinterpret_cast<uint4*>(img), a.N, g);
    SG_LAUNCH_CHECK("gru_pack_whh_kernel");
  }
  int rc2 = -1;
  if (pp == 1) rc2 = launch_tc<1>(ta, smem, st, &mc, false);
  else if (pp == 2) rc2 = launch_tc<2>(ta, smem, st, &mc, false);
  else if (pp == 3) rc2 = launch_tc<3>(ta, smem, st, &mc, false);
  if (dbg && rc2 == 0) {      // measurement only: phase stamps of 4 mid-sequence steps, CTA 0
    long long h[64];
    SG_CUDA(cudaStreamSynchronize(st));
    SG_CUDA(cudaMemcpy(h, dbg_buf, sizeof(h), cudaMemcpyDeviceToHost));
    static const char* names[12] = {"mma:top", "mma:first slice", "mma:all issued", "mma:commit", "epi:top", "epi:in-proj",
                                    "epi:tfull", "epi:tmem ld", "epi:gh bar", "epi:gates+stage", "epi:stage bar", "epi:sent"};
    for (int s = 0; s < 4; ++s) {
      fprintf(stderr, "[gru_tc dbg] step %d (U=%d CS=%d G=%d xsmem=%d pipe=%d):", a.N / 2 + s, g.U, g.CS, G, ta.x_smem,
              ta.pipelined);
      for (int k = 0; k < 12; ++k) fprintf(stderr, " %s=%lld", names[k], h[s * 16 + k] - h[4]);
      fprintf(stderr, "\n");
    }
  }
  return rc2;
}

const char* gru_tc_kernel_name() {
  return "gru_tc_cluster_kernel (GRU recurrence on tcgen05 kind::f16, fp16 hi/lo split operands, fp32 accumulate in TMEM, "
         "W_hh slices resident in smem, DSMEM st.async exchange)";
}

}  // namespace sg
