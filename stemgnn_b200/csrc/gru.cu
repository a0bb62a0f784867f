// GRU over the node axis + key/query contraction  (reference: models/base_model.py:92,137 and
// :154-155; gate equations as in torch.nn.GRU, gate order [r,z,n], h0 = 0) — forward and BPTT.
//
// The recurrence is N dependent steps of h(B x N) . W_hh^T(N x 3N): latency-bound, O(B N^3).
// B200 design (DESIGN.md §5, measurements in profiles/README.md):
//   * batch elements are independent sequences -> one THREAD-BLOCK CLUSTER of 16 CTAs per 4-5
//     sequences (7 clusters x 5 sequences = 112 SMs at B=32: a B200 keeps 7 clusters of 16 resident);
//   * each CTA of a cluster owns ceil(N/16) hidden units: its 3*U rows of W_hh stay resident in
//     shared memory for all N steps (persistent-RNN), so W_hh is read from HBM exactly once;
//   * per step: packed-fp32 (FFMA2) mat-vec in which every W_hh element is read from shared memory
//     once and used for all sequences of the cluster, recursive-halving warp reduction, gate math,
//     then the new hidden slice is sent to every CTA's next-step buffer through DISTRIBUTED SHARED
//     MEMORY with st.async stores that signal a per-buffer mbarrier in the destination CTA (no
//     cluster-wide barrier on the critical path: a CTA starts step s+1 when its 16 slices landed);
//   * the input projection W_ih x_s + b_ih of all steps is one GEMM beforehand (gru_input_proj),
//     prefetched a step ahead; key/query (sum over steps of h_s * w[s]) accumulate in registers, so
//     the (N,B,N) GRU output is never materialised in eval mode;
//   * BPTT (gru_bwd_cluster_kernel) reuses the layout: local gate gradients, partial W_hh^T d_gh over
//     the resident rows, reduce-scatter of the partial sums over DSMEM.
// A generic per-step-launch path covers N > 512 or devices that refuse the 16-CTA cluster.
// Since round 2 this file is the FALLBACK of the tensor-core recurrence (gru_tc.cu, gru_step_tc.cu) and the home of the BPTT.
#include <cooperative_groups.h>
#include <stdlib.h>

#include "common.cuh"
#include "gemm.cuh"
#include "internal.cuh"
#include "sm100.cuh"

namespace cg = cooperative_groups;

namespace sg {


constexpr int GRU_WARPS = 8;
constexpr int GRU_THREADS = GRU_WARPS * 32;
constexpr int GRU_SPIN_LOG2 = 24;       // mbarrier polls before a lost signal traps

// Warp-wide sum of C values per lane (C a power of two <= 32) by recursive halving: after log2(C)
// exchange stages every lane owns ONE column sum; lane l ends with the total of value l / (32/C).
// Costs C-1 + (5 - log2 C) shuffles instead of 5*C.
template <int C>
__device__ __forceinline__ float warp_reduce_scatter(float (&v)[C], int lane) {
  if constexpr (C == 1) {
    float r = v[0];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
    return r;
  } else {
    constexpr int LOG = (C == 32) ? 5 : (C == 16) ? 4 : (C == 8) ? 3 : (C == 4) ? 2 : 1;
    int o = 16;
    int n = C;
#pragma unroll
    for (int st = 0; st < LOG; ++st) {
      const int half = n >> 1;
      const bool up = (lane & o) != 0;
#pragma unroll
      for (int i = 0; i < C / 2; ++i) {
        if (i < half) {
          const float send = up ? v[i] : v[i + half];
          const float keep = up ? v[i + half] : v[i];
          v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
      }
      n = half;
      o >>= 1;
    }
    float r = v[0];
#pragma unroll
    for (int st = LOG; st < 5; ++st) {
      r += __shfl_xor_sync(0xffffffffu, r, o);
      o >>= 1;
    }
    return r;
  }
}

// reduce V = sum of power-of-two chunks; writes the V totals to out[0..V) (one lane per value)
template <int V, int OFF = 0>
__device__ __forceinline__ void warp_reduce_to_smem(const float* vals, float* out, int lane) {
  if constexpr (V > 0) {
    constexpr int C = (V >= 32) ? 32 : (V >= 16) ? 16 : (V >= 8) ? 8 : (V >= 4) ? 4 : (V >= 2) ? 2 : 1;
    float v[C];
#pragma unroll
    for (int i = 0; i < C; ++i) v[i] = vals[OFF + i];
    const float r = warp_reduce_scatter<C>(v, lane);
    if ((lane % (32 / C)) == 0) out[OFF + lane / (32 / C)] = r;
    warp_reduce_to_smem<V - C, OFF + C>(vals, out, lane);
  }
}

// JC: padded h length = 128*JC;  UPW: hidden units per warp;  CS: cluster size;
// NG x G: a cluster owns NG independent groups of G sequences.  With NG = 2 the groups are software
// pipelined: while group A's new hidden slices travel through DSMEM, the CTA computes group B.
template <int JC, int UPW, int CS, int NG, int G>
__global__ void __launch_bounds__(GRU_THREADS, 1) gru_cluster_kernel(GruArgs a) {
  constexpr int KP = 128 * JC;
  constexpr int ULOC = GRU_WARPS * UPW;     // padded units per CTA
  constexpr int ROWS = 3 * UPW;             // W_hh rows per warp
  constexpr int V = ROWS * G;               // dot products per warp per group-step
  constexpr int BC = NG * G;                // sequences per cluster
  static_assert(UPW * G <= 32, "finalising lanes");

  extern __shared__ __align__(16) float smem[];
  float* Wsm = smem;                              // [3*ULOC][KP]
  float* hbuf = Wsm + 3 * ULOC * KP;              // [NG][2][G][KP]
  float* stage = hbuf + NG * 2 * G * KP;          // [NG][5][G][32]: new h, and (training) r, z, n, hn
  float* sums = stage + NG * 5 * G * 32;          // [WARPS][V]
  uint64_t* hbar = reinterpret_cast<uint64_t*>(sums + GRU_WARPS * V + ((GRU_WARPS * V) & 1));   // [NG][2]

  cg::cluster_group cluster = cg::this_cluster();
  const int q = (int)cluster.block_rank();
  const int cid = blockIdx.x / CS;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int N = a.N, B = a.B;
  const int U = (N + CS - 1) / CS;
  const int UP = (U + 3) & ~3;              // slice pitch: every CTA's slice of h is 16-byte aligned
  const int UP4 = UP >> 2;
  const int u0 = q * U;
  const int b0 = cid * BC;

  // ---- one-time: W_hh slice -> smem, h buffers = 0, mbarriers ---------------------------------
  // hidden index k lives at position (k / U) * UP + (k % U) of the padded h vector; the columns of
  // the W_hh slice are permuted the same way (padding columns are zero).
  for (int idx = tid; idx < 3 * ULOC * KP; idx += GRU_THREADS) {
    const int row = idx / KP, kp = idx - row * KP;
    const int lu = row / 3, gate = row - lu * 3;
    const int u = u0 + lu;
    const int src_cta = kp / UP, src_lu = kp - src_cta * UP;
    const int k = src_cta * U + src_lu;
    float v = 0.f;
    if (lu < U && u < N && src_cta < CS && src_lu < U && k < N)
      v = __ldg(a.w_hh + ((long long)gate * N + u) * N + k);
    Wsm[idx] = v;
  }
  for (int idx = tid; idx < NG * 2 * G * KP; idx += GRU_THREADS) hbuf[idx] = 0.f;
  for (int idx = tid; idx < NG * 5 * G * 32; idx += GRU_THREADS) stage[idx] = 0.f;
  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < NG * 2; ++i) mbarrier_init(&hbar[i], 1);
    fence_mbarrier_init();
  }
  const uint32_t tx_bytes = (uint32_t)(CS * G * UP * sizeof(float));   // bytes a CTA receives per group-step

  // step-invariant send descriptors (same for every group up to a constant offset):
  // item -> (float4 inside stage[g][0], remote destination inside hbuf[g][0], remote mbarrier hbar[g][0])
  constexpr int SEND_ITEMS = (CS * G * 8 + GRU_THREADS - 1) / GRU_THREADS;   // UP4 <= 8
  int snd_src[SEND_ITEMS];
  uint32_t snd_dst[SEND_ITEMS], snd_bar[SEND_ITEMS];
#pragma unroll
  for (int it = 0; it < SEND_ITEMS; ++it) {
    const int idx = tid + it * GRU_THREADS;
    snd_src[it] = -1;
    snd_dst[it] = snd_bar[it] = 0;
    if (idx < CS * G * UP4) {
      const int dest = idx / (G * UP4);
      const int rem = idx - dest * (G * UP4);
      const int bb = rem / UP4, i4 = rem - bb * UP4;
      snd_src[it] = bb * 32 + 4 * i4;
      snd_dst[it] = mapa_shared_cluster(smem_u32(hbuf + bb * KP + q * UP + 4 * i4), (uint32_t)dest);
      snd_bar[it] = mapa_shared_cluster(smem_u32(&hbar[0]), (uint32_t)dest);
    }
  }

  // finalising lanes: lane t < UPW*G owns (local unit w*UPW + t/G, sequence t%G of each group)
  const int fi = lane / G, fb = lane - fi * G;
  const int lu = w * UPW + fi;
  const int u = u0 + lu;
  const bool flane = lane < UPW * G;
  const bool fin = flane && (lu < U) && (u < N);
  float bhr = 0.f, bhz = 0.f, bhn = 0.f;
  if (fin) {
    bhr = __ldg(a.b_hh + u);
    bhz = __ldg(a.b_hh + N + u);
    bhn = __ldg(a.b_hh + 2 * N + u);
  }
  float key_acc[NG], query_acc[NG], gi_r[NG], gi_z[NG], gi_n[NG];
  bool bvalid[NG];

  // input projection W_i{r,z,n} x_s + b_i{r,z,n} comes precomputed (gru_input_proj); the values of
  // step s+1 are requested while step s computes so their latency hides behind the mat-vec.
  auto load_gi = [&](int s, int bglob, bool ok, float& gr, float& gz, float& gn) {
    gr = gz = gn = 0.f;
    if (fin && ok) {
      const float* g = a.gi + ((long long)s * B + bglob) * (3 * N) + u;
      gr = __ldg(g);
      gz = __ldg(g + N);
      gn = __ldg(g + 2 * N);
    }
  };
#pragma unroll
  for (int g = 0; g < NG; ++g) {
    key_acc[g] = query_acc[g] = 0.f;
    bvalid[g] = (b0 + g * G + fb) < B;
    load_gi(0, b0 + g * G + fb, bvalid[g], gi_r[g], gi_z[g], gi_n[g]);
  }
  float wk_s = __ldg(a.wk + 0), wq_s = __ldg(a.wq + 0);

  __syncthreads();
  cluster.sync();   // every CTA's buffers and barriers are initialised before any remote write

  for (int s = 0; s < N; ++s) {
    const int cur = s & 1, nxt = cur ^ 1;
    float nx_wk = 0.f, nx_wq = 0.f;
    if (s + 1 < N) {
      nx_wk = __ldg(a.wk + s + 1);
      nx_wq = __ldg(a.wq + s + 1);
    }
#pragma unroll
    for (int g = 0; g < NG; ++g) {
      float* hb_cur = hbuf + ((g * 2 + cur) * G) * KP;
      float* stg = stage + g * 5 * G * 32;
      // arm the barrier of the buffer that will receive h_s, wait until h_{s-1} of this group landed
      if (tid == 0 && s + 1 < N) mbarrier_arrive_expect_tx(&hbar[g * 2 + nxt], tx_bytes * (uint32_t)a.xrep);
      if (s > 0) mbarrier_wait<GRU_SPIN_LOG2>(&hbar[g * 2 + cur], (uint32_t)((s - 1) >> 1) & 1u);
      float nx_r = 0.f, nx_z = 0.f, nx_n = 0.f;
      if (s + 1 < N) load_gi(s + 1, b0 + g * G + fb, bvalid[g], nx_r, nx_z, nx_n);

      // (a)+(b) mat-vec, k-chunk outer / row inner: the lane's slice of h_{s-1} (k' = 128 j + 4 lane + {0..3}
      //     for the G sequences) is loaded chunk by chunk so that the loads of chunk j+1 overlap the FFMA2s of
      //     chunk j.  Each W_hh element is read from shared memory once per group-step (32 lanes x 16 B distinct
      //     per LDS.128) and used for the G sequences; two partial sums per (row, sequence).
      float2 acc[ROWS][G];
#pragma unroll
      for (int r = 0; r < ROWS; ++r)
#pragma unroll
        for (int bb = 0; bb < G; ++bb) acc[r][bb] = make_float2(0.f, 0.f);
      const float* wbase = Wsm + (long long)(w * ROWS) * KP + 4 * lane;
#pragma unroll
      for (int j = 0; j < JC; ++j) {
        float4 h[G];
#pragma unroll
        for (int bb = 0; bb < G; ++bb)
          h[bb] = *reinterpret_cast<const float4*>(hb_cur + bb * KP + 128 * j + 4 * lane);
#pragma unroll
        for (int r = 0; r < ROWS; ++r) {
          const float4 wv = *reinterpret_cast<const float4*>(wbase + r * KP + 128 * j);
#pragma unroll
          for (int bb = 0; bb < G; ++bb) {
            acc[r][bb] = __ffma2_rn(make_float2(wv.x, wv.y), make_float2(h[bb].x, h[bb].y), acc[r][bb]);
            acc[r][bb] = __ffma2_rn(make_float2(wv.z, wv.w), make_float2(h[bb].z, h[bb].w), acc[r][bb]);
          }
        }
      }
      // (c) reduce the V partial dot products over the 32 lanes (recursive halving) -> sums[w][V]
      float part[V];
#pragma unroll
      for (int r = 0; r < ROWS; ++r)
#pragma unroll
        for (int bb = 0; bb < G; ++bb) part[r * G + bb] = acc[r][bb].x + acc[r][bb].y;
      float* wsum = sums + w * V;
      warp_reduce_to_smem<V>(part, wsum, lane);
      __syncwarp();
      // (d) gates for (unit, sequence) on the first UPW*G lanes
      if (flane) {
        float hn = 0.f;
        if (fin) {
          const float gh_r = wsum[(3 * fi + 0) * G + fb];
          const float gh_z = wsum[(3 * fi + 1) * G + fb];
          const float gh_n = wsum[(3 * fi + 2) * G + fb];
          const float hprev = hb_cur[fb * KP + q * UP + lu];
          const float r = fast_sigmoid(gi_r[g] + gh_r + bhr);
          const float zt = fast_sigmoid(gi_z[g] + gh_z + bhz);
          const float nt = fast_tanh(gi_n[g] + r * (gh_n + bhn));
          hn = (1.f - zt) * nt + zt * hprev;
          key_acc[g] = fmaf(hn, wk_s, key_acc[g]);
          query_acc[g] = fmaf(hn, wq_s, query_acc[g]);
          if (a.g_r != nullptr) {   // gate values for BPTT
            stg[(1 * G + fb) * 32 + lu] = r;
            stg[(2 * G + fb) * 32 + lu] = zt;
            stg[(3 * G + fb) * 32 + lu] = nt;
            stg[(4 * G + fb) * 32 + lu] = gh_n + bhn;
          }
        }
        stg[fb * 32 + lu] = hn;
      }
      __syncthreads();
      // (e) send the CTA's new slice to every cluster CTA's next buffer: 16-byte st.async stores through
      //     DSMEM, each signalling the destination's mbarrier (no cluster-wide barrier on the critical path)
      if (s + 1 < N) {
        const uint32_t dst_off = (uint32_t)((g * 2 + nxt) * G * KP * 4);
        const uint32_t bar_off = (uint32_t)((g * 2 + nxt) * 8);
        for (int rep = 1; rep < a.xrep; ++rep)     // measurement knob only (STEMGNN_GRU_XREP)
#pragma unroll
          for (int it = 0; it < SEND_ITEMS; ++it)
            if (snd_src[it] >= 0)
              st_async_v4(snd_dst[it] + dst_off, *reinterpret_cast<const uint4*>(stg + snd_src[it]),
                          snd_bar[it] + bar_off);
#pragma unroll
        for (int it = 0; it < SEND_ITEMS; ++it) {
          if (snd_src[it] >= 0) {
            const uint4 v = *reinterpret_cast<const uint4*>(stg + snd_src[it]);
            st_async_v4(snd_dst[it] + dst_off, v, snd_bar[it] + bar_off);
          }
        }
      }
      if (a.h_all != nullptr && w < G && (b0 + g * G + w) < B && lane < U && (u0 + lane) < N) {
        const long long o = ((long long)s * B + (b0 + g * G + w)) * N + u0 + lane;
        a.h_all[o] = stg[w * 32 + lane];
        if (a.g_r != nullptr) {
          a.g_r[o] = stg[(1 * G + w) * 32 + lane];
          a.g_z[o] = stg[(2 * G + w) * 32 + lane];
          a.g_n[o] = stg[(3 * G + w) * 32 + lane];
          a.g_hn[o] = stg[(4 * G + w) * 32 + lane];
        }
      }
      gi_r[g] = nx_r; gi_z[g] = nx_z; gi_n[g] = nx_n;
      if (NG == 1) __syncthreads();   // stage[] is rewritten by the next step's gate phase
    }
    wk_s = nx_wk; wq_s = nx_wq;
  }
  cluster.sync();      // no CTA may exit while peers could still address its shared memory

#pragma unroll
  for (int g = 0; g < NG; ++g) {
    if (fin && bvalid[g]) {
      a.key[(long long)(b0 + g * G + fb) * N + u] = key_acc[g];
      a.query[(long long)(b0 + g * G + fb) * N + u] = query_acc[g];
    }
  }
}

// returns 0 launched, -1 configuration not launchable here, >0 error
template <int JC, int UPW, int CS, int NG, int G>
static int launch_gru_cluster(const GruArgs& a, cudaStream_t st, int* max_active_out) {
  constexpr int KP = 128 * JC;
  constexpr int ULOC = GRU_WARPS * UPW;
  constexpr int V = 3 * UPW * G;
  const size_t smem = (size_t)(3 * ULOC * KP + NG * 2 * G * KP + NG * 5 * G * 32 + GRU_WARPS * V + 2) * sizeof(float) +
                      NG * 2 * sizeof(uint64_t);
  auto kern = gru_cluster_kernel<JC, UPW, CS, NG, G>;
  static bool attr_set_dev[64] = {};      // function attributes / occupancy are per device (ADVICE r1)
  static int max_clusters_dev[64] = {};
  int dev_ = 0;
  (void)cudaGetDevice(&dev_);
  bool& attr_set = attr_set_dev[dev_ & 63];
  int& max_clusters = max_clusters_dev[dev_ & 63];
  const int nclusters = ceil_div(a.B, NG * G);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(nclusters * CS);
  cfg.blockDim = dim3(GRU_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (!attr_set) {
    if (smem > 227 * 1024) return -1;
    SG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (CS > 8)
      SG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaError_t e = cudaOccupancyMaxActiveClusters(&max_clusters, kern, &cfg);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      max_clusters = 0;
    }
    attr_set = true;
  }
  if (max_active_out != nullptr) *max_active_out = max_clusters;
  if (max_clusters < 1) return -1;
  if (max_active_out != nullptr) return 0;      // probe only
  ProfileHook* hook = profile_hook();
  if (hook->start != nullptr) SG_CUDA(cudaEventRecord(hook->start, st));
  SG_CUDA(cudaLaunchKernelEx(&cfg, kern, a));
  if (hook->stop != nullptr) SG_CUDA(cudaEventRecord(hook->stop, st));
  count_launch();
  return 0;
}

template <int CS, int NG, int G>
static int dispatch_gru_cluster(const GruArgs& a, cudaStream_t st, int* probe) {
  const int U = ceil_div(a.N, CS);
  const int upw = ceil_div(U, GRU_WARPS);
  const int jc = ceil_div(CS * ((U + 3) & ~3), 128);     // padded h vector: CS slices of pitch round4(U)
  if (upw > 4 || jc > 4) return -1;
#define SG_GRU_CASE(J, P) \
  if (jc == J && upw == P) return launch_gru_cluster<J, P, CS, NG, G>(a, st, probe);
  SG_GRU_CASE(1, 1) SG_GRU_CASE(1, 2) SG_GRU_CASE(1, 3) SG_GRU_CASE(1, 4)
  SG_GRU_CASE(2, 1) SG_GRU_CASE(2, 2) SG_GRU_CASE(2, 3) SG_GRU_CASE(2, 4)
  SG_GRU_CASE(3, 1) SG_GRU_CASE(3, 2) SG_GRU_CASE(3, 3) SG_GRU_CASE(3, 4)
  SG_GRU_CASE(4, 1) SG_GRU_CASE(4, 2) SG_GRU_CASE(4, 3) SG_GRU_CASE(4, 4)
#undef SG_GRU_CASE
  return -1;
}

// =================================================================================================
// BPTT through the recurrence on the same cluster layout (backward of base_model.py:137).
//
// Per step s = N-1 .. 0 every CTA (i) sums the 16 partial d h_s slices it received, adds the direct
// key/query terms, and turns them into the gate gradients of ITS hidden units (written to DGH / DGI
// for the weight-gradient GEMMs); (ii) multiplies them with its resident rows of W_hh:
// partial[b][k] = sum_{own rows} d_gh[b][row] W_hh[row][k] for ALL k (lanes own distinct k, so there is
// no cross-lane reduction; the 8 warps' row groups are combined through shared memory); (iii) sends the
// slice of `partial` that belongs to CTA p's units to CTA p (reduce-scatter over DSMEM with st.async +
// mbarrier, same transport as the forward).  W_hh never leaves shared memory: one launch instead of N.
struct GruBwdClusterArgs {
  const float* w_hh; const float* wk; const float* wq;
  const float* d_key; const float* d_query;
  const float* h_all; const float* g_r; const float* g_z; const float* g_n; const float* g_hn;
  float* dgh; float* dgi;            // (S*B, 3N)
  int B, N;
};

template <int JC, int UPW, int CS, int G>
__global__ void __launch_bounds__(GRU_THREADS, 1) gru_bwd_cluster_kernel(GruBwdClusterArgs a) {
  constexpr int KP = 128 * JC;
  constexpr int KQ = KP / 4;                // float4 chunks per padded h vector
  constexpr int ULOC = GRU_WARPS * UPW;
  constexpr int ROWS = 3 * UPW;
  static_assert(UPW * G <= 32, "finalising lanes");

  extern __shared__ __align__(16) float smem[];
  float* Wsm = smem;                                  // [3*ULOC][KP]
  float* red = Wsm + 3 * ULOC * KP;                   // [WARPS][G][KP] per-warp partial products
  float* recv = red + GRU_WARPS * G * KP;             // [2][CS][G][32] received d h slices
  float2* coef = reinterpret_cast<float2*>(recv + 2 * CS * G * 32);   // [3*ULOC][G] {g,g}
  uint64_t* rbar = reinterpret_cast<uint64_t*>(coef + 3 * ULOC * G);  // [2]

  cg::cluster_group cluster = cg::this_cluster();
  const int q = (int)cluster.block_rank();
  const int cid = blockIdx.x / CS;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int N = a.N, B = a.B;
  const int U = (N + CS - 1) / CS;
  const int UP = (U + 3) & ~3;
  const int UP4 = UP >> 2;
  const int u0 = q * U;
  const int b0 = cid * G;

  for (int idx = tid; idx < 3 * ULOC * KP; idx += GRU_THREADS) {
    const int row = idx / KP, kp = idx - row * KP;
    const int lu = row / 3, gate = row - lu * 3;
    const int u = u0 + lu;
    const int src_cta = kp / UP, src_lu = kp - src_cta * UP;
    const int k = src_cta * U + src_lu;
    float v = 0.f;
    if (lu < U && u < N && src_cta < CS && src_lu < U && k < N)
      v = __ldg(a.w_hh + ((long long)gate * N + u) * N + k);
    Wsm[idx] = v;
  }
  for (int idx = tid; idx < 2 * CS * G * 32; idx += GRU_THREADS) recv[idx] = 0.f;
  for (int idx = tid; idx < 3 * ULOC * G; idx += GRU_THREADS) coef[idx] = make_float2(0.f, 0.f);
  if (tid == 0) {
    mbarrier_init(&rbar[0], 1);
    mbarrier_init(&rbar[1], 1);
    fence_mbarrier_init();
  }
  const uint32_t tx_bytes = (uint32_t)(CS * G * UP * sizeof(float));

  // reduce-scatter descriptors: this thread combines float4 chunk (b, kq) of the 8 warp partials and
  // sends it to the CTA that owns hidden positions [4kq, 4kq+4)
  constexpr int ITEMS = (G * KQ + GRU_THREADS - 1) / GRU_THREADS;
  int it_off[ITEMS];
  uint32_t it_dst[ITEMS], it_bar[ITEMS];
#pragma unroll
  for (int it = 0; it < ITEMS; ++it) {
    const int c = tid + it * GRU_THREADS;
    it_off[it] = -1;
    it_dst[it] = it_bar[it] = 0;
    if (c < G * KQ) {
      const int bb = c / KQ, kq = c - bb * KQ;
      const int dest = kq / UP4, i4 = kq - dest * UP4;
      if (dest < CS) {
        it_off[it] = bb * KP + 4 * kq;
        it_dst[it] = mapa_shared_cluster(smem_u32(recv + (q * G + bb) * 32 + 4 * i4), (uint32_t)dest);
        it_bar[it] = mapa_shared_cluster(smem_u32(&rbar[0]), (uint32_t)dest);
      }
    }
  }

  // finalising lanes: lane t < UPW*G owns (local unit w*UPW + t/G, sequence t%G)
  const int fi = lane / G, fb = lane - fi * G;
  const int lu = w * UPW + fi;
  const int u = u0 + lu;
  const bool flane = lane < UPW * G;
  const bool bvalid = (b0 + fb) < B;
  const bool fin = flane && (lu < U) && (u < N) && bvalid;
  float dk = 0.f, dq = 0.f;
  if (fin) {
    dk = __ldg(a.d_key + (long long)(b0 + fb) * N + u);
    dq = __ldg(a.d_query + (long long)(b0 + fb) * N + u);
  }
  // saved gates of step s for this lane, requested one step ahead
  auto load_gates = [&](int s, float& r, float& z, float& n, float& hn, float& hp) {
    r = z = n = hn = hp = 0.f;
    if (fin) {
      const long long e = ((long long)s * B + (b0 + fb)) * N + u;
      r = __ldg(a.g_r + e); z = __ldg(a.g_z + e); n = __ldg(a.g_n + e); hn = __ldg(a.g_hn + e);
      if (s > 0) hp = __ldg(a.h_all + e - (long long)B * N);
    }
  };
  float gr, gz, gn, ghn, ghp;
  load_gates(N - 1, gr, gz, gn, ghn, ghp);
  float carry = 0.f;       // dh_s * z_s : direct path into dh_{s-1} of the same (unit, sequence)

  __syncthreads();
  cluster.sync();

  for (int s = N - 1; s >= 0; --s) {
    const int cur = s & 1, nxt = cur ^ 1;
    if (tid == 0 && s > 0) mbarrier_arrive_expect_tx(&rbar[nxt], tx_bytes);
    if (s < N - 1) mbarrier_wait<GRU_SPIN_LOG2>(&rbar[cur], (uint32_t)((N - 2 - s) >> 1) & 1u);
    float nr = 0.f, nz = 0.f, nn = 0.f, nhn = 0.f, nhp = 0.f;
    if (s > 0) load_gates(s - 1, nr, nz, nn, nhn, nhp);
    // (i) gate gradients of the own units
    if (flane) {
      float d_r = 0.f, d_z = 0.f, d_np = 0.f, d_hn = 0.f;
      if (fin) {
        float dh = carry + dk * __ldg(a.wk + s) + dq * __ldg(a.wq + s);
        if (s < N - 1) {
          const float* rp = recv + (cur * CS * G + fb) * 32 + lu;
#pragma unroll
          for (int src = 0; src < CS; ++src) dh += rp[src * G * 32];
        }
        const float dn = dh * (1.f - gz);
        d_np = dn * (1.f - gn * gn);
        d_z = dh * (ghp - gn) * gz * (1.f - gz);
        d_r = d_np * ghn * gr * (1.f - gr);
        d_hn = d_np * gr;
        carry = dh * gz;
        const long long o = ((long long)s * B + (b0 + fb)) * 3 * N + u;
        a.dgh[o] = d_r; a.dgh[o + N] = d_z; a.dgh[o + 2 * N] = d_hn;
        a.dgi[o] = d_r; a.dgi[o + N] = d_z; a.dgi[o + 2 * N] = d_np;
      }
      coef[(lu * 3 + 0) * G + fb] = make_float2(d_r, d_r);
      coef[(lu * 3 + 1) * G + fb] = make_float2(d_z, d_z);
      coef[(lu * 3 + 2) * G + fb] = make_float2(d_hn, d_hn);
    }
    gr = nr; gz = nz; gn = nn; ghn = nhn; ghp = nhp;
    if (s == 0) break;                      // dh_{-1} is not needed
    __syncthreads();
    // (ii) partial[b][k] over this warp's rows; lane owns k' = 128 j + 4 lane + {0..3}
    float2 acc[G][JC][2];
#pragma unroll
    for (int bb = 0; bb < G; ++bb)
#pragma unroll
      for (int j = 0; j < JC; ++j) acc[bb][j][0] = acc[bb][j][1] = make_float2(0.f, 0.f);
    const float* wbase = Wsm + (long long)(w * ROWS) * KP + 4 * lane;
    const float2* cbase = coef + (w * ROWS) * G;
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
      float4 wv[JC];
#pragma unroll
      for (int j = 0; j < JC; ++j) wv[j] = *reinterpret_cast<const float4*>(wbase + r * KP + 128 * j);
#pragma unroll
      for (int bb = 0; bb < G; ++bb) {
        const float2 g2 = cbase[r * G + bb];
#pragma unroll
        for (int j = 0; j < JC; ++j) {
          acc[bb][j][0] = __ffma2_rn(make_float2(wv[j].x, wv[j].y), g2, acc[bb][j][0]);
          acc[bb][j][1] = __ffma2_rn(make_float2(wv[j].z, wv[j].w), g2, acc[bb][j][1]);
        }
      }
    }
    float* myred = red + (long long)w * G * KP + 4 * lane;
#pragma unroll
    for (int bb = 0; bb < G; ++bb)
#pragma unroll
      for (int j = 0; j < JC; ++j)
        *reinterpret_cast<float4*>(myred + bb * KP + 128 * j) =
            make_float4(acc[bb][j][0].x, acc[bb][j][0].y, acc[bb][j][1].x, acc[bb][j][1].y);
    __syncthreads();
    // (iii) combine the 8 row groups and reduce-scatter to the owners of each hidden slice
#pragma unroll
    for (int it = 0; it < ITEMS; ++it) {
      if (it_off[it] >= 0) {
        float4 v = *reinterpret_cast<const float4*>(red + it_off[it]);
#pragma unroll
        for (int ww = 1; ww < GRU_WARPS; ++ww) {
          const float4 t = *reinterpret_cast<const float4*>(red + (long long)ww * G * KP + it_off[it]);
          v.x += t.x; v.y += t.y; v.z += t.z; v.w += t.w;
        }
        st_async_v4(it_dst[it] + (uint32_t)nxt * (CS * G * 32 * 4),
                    make_uint4(__float_as_uint(v.x), __float_as_uint(v.y), __float_as_uint(v.z), __float_as_uint(v.w)),
                    it_bar[it] + (uint32_t)nxt * 8);
      }
    }
  }
  cluster.sync();
}

template <int JC, int UPW, int CS, int G>
static int launch_gru_bwd_cluster(const GruBwdClusterArgs& a, cudaStream_t st) {
  constexpr int KP = 128 * JC;
  constexpr int ULOC = GRU_WARPS * UPW;
  const size_t smem = (size_t)(3 * ULOC * KP + GRU_WARPS * G * KP + 2 * CS * G * 32 + 2 * 3 * ULOC * G) * sizeof(float) +
                      2 * sizeof(uint64_t);
  if (smem > 227 * 1024) return -1;
  auto kern = gru_bwd_cluster_kernel<JC, UPW, CS, G>;
  static bool attr_set_dev[64] = {};
  static int max_clusters_dev[64] = {};
  int dev_ = 0;
  (void)cudaGetDevice(&dev_);
  bool& attr_set = attr_set_dev[dev_ & 63];
  int& max_clusters = max_clusters_dev[dev_ & 63];
  const int nclusters = ceil_div(a.B, G);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(nclusters * CS);
  cfg.blockDim = dim3(GRU_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (!attr_set) {
    SG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (CS > 8) SG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaError_t e = cudaOccupancyMaxActiveClusters(&max_clusters, kern, &cfg);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      max_clusters = 0;
    }
    attr_set = true;
  }
  if (max_clusters < 1) return -1;
  SG_CUDA(cudaLaunchKernelEx(&cfg, kern, a));
  count_launch();
  return 0;
}

// returns 0 launched, -1 unsupported here (caller falls back to the per-step kernels), >0 error
int gru_bwd_cluster(const float* w_hh, const float* wk, const float* wq, const float* d_key,
                    const float* d_query, const float* h_all, const float* g_r, const float* g_z,
                    const float* g_n, const float* g_hn, float* dgh, float* dgi, int B, int N,
                    cudaStream_t st) {
  if (getenv("STEMGNN_BPTT_STEPWISE") != nullptr) return -1;
  constexpr int CS = 16;
  GruBwdClusterArgs a = {w_hh, wk, wq, d_key, d_query, h_all, g_r, g_z, g_n, g_hn, dgh, dgi, B, N};
  const int U = ceil_div(N, CS);
  const int upw = ceil_div(U, GRU_WARPS);
  const int jc = ceil_div(CS * ((U + 3) & ~3), 128);
  if (upw > 4 || jc > 4) return -1;
  const bool g5 = ceil_div(B, 4) > 7 && ceil_div(B, 5) <= 7;     // same wave rule as the forward
#define SG_BWD_CASE(J, P)                                                        \
  if (jc == J && upw == P) {                                                     \
    if (g5) {                                                                    \
      const int rc = launch_gru_bwd_cluster<J, P, CS, 5>(a, st);                 \
      if (rc >= 0) return rc;                                                    \
    }                                                                            \
    return launch_gru_bwd_cluster<J, P, CS, 4>(a, st);                           \
  }
  SG_BWD_CASE(1, 1) SG_BWD_CASE(1, 2) SG_BWD_CASE(2, 1) SG_BWD_CASE(2, 2) SG_BWD_CASE(2, 3)
  SG_BWD_CASE(3, 2) SG_BWD_CASE(3, 3) SG_BWD_CASE(3, 4) SG_BWD_CASE(4, 3) SG_BWD_CASE(4, 4)
  SG_BWD_CASE(1, 3) SG_BWD_CASE(1, 4) SG_BWD_CASE(2, 4) SG_BWD_CASE(3, 1) SG_BWD_CASE(4, 1) SG_BWD_CASE(4, 2)
#undef SG_BWD_CASE
  return -1;
}

// ---- generic path: one launch per step, W_hh streamed from L2 --------------------------------
// grid.x = ceil(N / 4) (one warp per hidden unit), loops over the batch in chunks of 4.
__global__ void __launch_bounds__(128) gru_step_kernel(GruArgs a, int s, const float* __restrict__ h_prev,
                                                       float* __restrict__ h_next) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int u = blockIdx.x * 4 + wid;
  const int N = a.N, B = a.B;
  if (u >= N) return;
  const float* wr = a.w_hh + (long long)u * N;
  const float* wz = a.w_hh + (long long)(N + u) * N;
  const float* wn = a.w_hh + (long long)(2 * N + u) * N;
  const float wk_s = __ldg(a.wk + s), wq_s = __ldg(a.wq + s);
  for (int bb = 0; bb < B; bb += 4) {
    float acc[3][4];
#pragma unroll
    for (int g = 0; g < 3; ++g)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[g][j] = 0.f;
    for (int k = lane; k < N; k += 32) {
      const float r = __ldg(wr + k), z = __ldg(wz + k), n = __ldg(wn + k);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float hv = (bb + j < B) ? h_prev[(long long)(bb + j) * N + k] : 0.f;
        acc[0][j] = fmaf(r, hv, acc[0][j]);
        acc[1][j] = fmaf(z, hv, acc[1][j]);
        acc[2][j] = fmaf(n, hv, acc[2][j]);
      }
    }
#pragma unroll
    for (int g = 0; g < 3; ++g)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[g][j] = warp_sum(acc[g][j]);
    if (lane < 4 && bb + lane < B) {
      const int bi = bb + lane;
      float gh_r = 0.f, gh_z = 0.f, gh_n = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (lane == j) { gh_r = acc[0][j]; gh_z = acc[1][j]; gh_n = acc[2][j]; }
      const float* gp = a.gi + ((long long)s * B + bi) * (3 * N) + u;
      const float gr = __ldg(gp), gz = __ldg(gp + N), gn = __ldg(gp + 2 * N);
      const float r = sigmoidf_(gr + gh_r + __ldg(a.b_hh + u));
      const float zt = sigmoidf_(gz + gh_z + __ldg(a.b_hh + N + u));
      const float nt = tanhf(gn + r * (gh_n + __ldg(a.b_hh + 2 * N + u)));
      const float hn = (1.f - zt) * nt + zt * h_prev[(long long)bi * N + u];
      h_next[(long long)bi * N + u] = hn;
      if (a.h_all != nullptr) a.h_all[((long long)s * B + bi) * N + u] = hn;
      if (a.g_r != nullptr) {
        const long long o = ((long long)s * B + bi) * N + u;
        a.g_r[o] = r; a.g_z[o] = zt; a.g_n[o] = nt; a.g_hn[o] = gh_n + __ldg(a.b_hh + 2 * N + u);
      }
      // key/query accumulate in place (this thread is the only writer of (bi,u))
      a.key[(long long)bi * N + u] = fmaf(hn, wk_s, a.key[(long long)bi * N + u]);
      a.query[(long long)bi * N + u] = fmaf(hn, wq_s, a.query[(long long)bi * N + u]);
    }
  }
}

// gi[(s*B+b)][g*N+u] = W_i{g} x_s[b] + b_i{g}   for all steps at once: (N*B x W) . (W x 3N).
// K = W is tiny (12): the product is bound by writing the (N*B x 3N) result (49 MB at cfg2), so each thread keeps
// one row of W_ih in registers and streams over a tile of 64 x-rows held in shared memory (coalesced stores).
template <int WMAX>
__global__ void __launch_bounds__(256) gru_input_proj_kernel(const float* __restrict__ xs, const float* __restrict__ w_ih,
                                                             const float* __restrict__ b_ih, float* __restrict__ gi,
                                                             int SB, int N3, int W) {
  __shared__ float xt[64][WMAX];
  const int row = blockIdx.x * 256 + threadIdx.x;
  const int r0 = blockIdx.y * 64;
  const int nr = min(64, SB - r0);
  for (int i = threadIdx.x; i < 64 * WMAX; i += 256) {      // padded taps must be finite zeros
    const int r = i / WMAX, t = i % WMAX;
    xt[r][t] = (r < nr && t < W) ? xs[(long long)(r0 + r) * W + t] : 0.f;
  }
  float wr[WMAX];
  float bias = 0.f;
  if (row < N3) {
    bias = __ldg(b_ih + row);
#pragma unroll
    for (int t = 0; t < WMAX; ++t) wr[t] = t < W ? __ldg(w_ih + (long long)row * W + t) : 0.f;
  }
  __syncthreads();
  if (row >= N3) return;
  for (int r = 0; r < nr; ++r) {
    float acc = bias;
#pragma unroll
    for (int t = 0; t < WMAX; ++t) acc = fmaf(wr[t], xt[r][t], acc);     // padded taps multiply zeros
    gi[(long long)(r0 + r) * N3 + row] = acc;
  }
}

int gru_input_proj(const GruArgs& a, cudaStream_t st) {
  const int SB = a.N * a.B, N3 = 3 * a.N;
  if (a.W <= 16) {
    dim3 grid(ceil_div(N3, 256), ceil_div(SB, 64));
    gru_input_proj_kernel<16><<<grid, 256, 0, st>>>(a.xs, a.w_ih, a.b_ih, a.gi, SB, N3, a.W);
    SG_LAUNCH_CHECK("gru_input_proj_kernel");
    return 0;
  }
  GemmOperands g = {a.xs, a.W, 0, a.w_ih, a.W, 0, nullptr, SB, N3, a.W};
  EpiBias<0> epi = {a.gi, N3, 0, a.b_ih, 0};
  return launch_sgemm<false, true, false>(g, epi, 1, st, "gru_input_proj");
}

// scratch: 2*B*N floats (ping-pong hidden state) for the generic path
int gru_keyquery_forward(const GruArgs& a_in, int path, float* scratch, cudaStream_t st) {
  GruArgs a = a_in;
  SG_CHECK(a.B > 0 && a.N > 0 && a.W > 0, "gru: bad dims B=%d N=%d W=%d", a.B, a.N, a.W);
  a.xrep = 1;
  if (const char* e = getenv("STEMGNN_GRU_XREP")) a.xrep = atoi(e) > 0 ? atoi(e) : 1;
  if (path == 0 || path == 3) {
    // tensor-core recurrence (gru_tc.cu): input projection in-kernel, packed W_hh images live at the start of `gi`
    const int rc = gru_tc_forward(a, reinterpret_cast<uint8_t*>(a.gi), a.tc_reuse, st);
    if (rc == 0) return 0;
    if (rc > 0) return rc;
    if (a.N > 512) {      // beyond every cluster kernel: one tensor-core launch per step, W_hh streamed from L2
      const int rc2 = gru_step_tc_forward(a, reinterpret_cast<uint8_t*>(a.gi), (size_t)3 * a.N * a.N * a.B * sizeof(float),
                                          a.tc_reuse, st);
      if (rc2 == 0) return 0;
      if (rc2 > 0) return rc2;
    }
    SG_CHECK(path != 3, "gru: tensor-core path unavailable for N=%d W=%d on this device", a.N, a.W);
  }
  SG_TRY(gru_input_proj(a, st));
  if (path != 1) {
    // 16-CTA clusters with one group of 4 (or 5, to stay within the 7 resident clusters of a B200) sequences each.
    // (The two-group software-pipelined and the unit-wise variants of round 1 measured slower and were removed;
    // profiles/README.md keeps their numbers.)
    int max_active = 0;
    int rc = dispatch_gru_cluster<16, 1, 4>(a, st, &max_active);
    if (rc == 0) {
      const int mx = max_active > 0 ? max_active : 1;
      const bool g5 = ceil_div(a.B, 4) > mx && ceil_div(a.B, 5) <= mx;     // one wave beats two
      rc = g5 ? dispatch_gru_cluster<16, 1, 5>(a, st, nullptr) : dispatch_gru_cluster<16, 1, 4>(a, st, nullptr);
      if (rc < 0) rc = dispatch_gru_cluster<16, 1, 4>(a, st, nullptr);
      if (rc == 0) return 0;
      if (rc > 0) return rc;
    } else if (rc > 0) {
      return rc;
    }
    if (a.N <= 256) {
      rc = dispatch_gru_cluster<8, 1, 4>(a, st, nullptr);
      if (rc == 0) return 0;
      if (rc > 0) return rc;
    }
    SG_CHECK(path != 2, "gru: cluster path unavailable for N=%d on this device", a.N);
  }
  const size_t bn = (size_t)a.B * a.N;
  SG_CUDA(cudaMemsetAsync(scratch, 0, 2 * bn * sizeof(float), st));
  SG_CUDA(cudaMemsetAsync(a.key, 0, bn * sizeof(float), st));
  SG_CUDA(cudaMemsetAsync(a.query, 0, bn * sizeof(float), st));
  for (int s = 0; s < a.N; ++s) {
    const float* hp = scratch + (size_t)(s & 1) * bn;
    float* hn = scratch + (size_t)((s & 1) ^ 1) * bn;
    gru_step_kernel<<<ceil_div(a.N, 4), 128, 0, st>>>(a, s, hp, hn);
    count_launch();
  }
  SG_LAUNCH_CHECK("gru_step_kernel");
  return 0;
}

}  // namespace sg
