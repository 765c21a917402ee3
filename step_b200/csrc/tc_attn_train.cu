// Stage-1 (TSFormer pre-training) attention on the 5th-generation tensor cores: forward with the statistics the
// backward needs, and the backward itself.  bf16 operands, fp32 accumulation in TMEM, fp32 softmax statistics.
//
// Operands are the per-(sequence, head) images of tc_encoder.cu's attention (see step_tc_qkv): Q pre-scaled by
// log2(e)/sqrt(24) as [RT row tiles][3 chunks][128 rows][8] (odd heads' last tile of <= 64 queries at rows 64..),
// K and V as [3 chunks][Pk rows][8], Pk = P rounded up to 16.  Head dim 24 is padded to 32 by a shared zero chunk.
//
// Forward, one CTA per (sequence, head), per 128-query tile:  S = Q K^T (TMEM), exact row max and
// l = sum 2^(s - m) in fp32, P = bf16(2^(s - m)) with dropout -> K-major image in smem, O = P V (TMEM);
// writes O / l as fp32 rows [S*P, 96] and the log2-sum-exp L = m + log2(l) [S, 4, P].
//
// Backward, one CTA per (sequence, head), for every (128-key tile kt, 128-query tile qc):
//   S^T = K_kt Q_qc^T, dP^T = V_kt dO_qc^T                      (M = keys, N = queries, K = 32)
//   thread = key j:  p = 2^(s - L_i), keep = mask(i, j), dS = p (keep dP / (1 - p) - D_i)
//   dV_kt += (p keep / (1 - p))^T dO_qc,  dK_kt += dS^T Q_qc    (M = keys, K = queries)
//   dQ_qc += dS K_kt                                             (M = queries, K = keys: the dS^T image read MN-major)
// D_i = dO_i . O_i is formed in fp32 from the fp32 rows before dO is rounded to bf16.
//
// Synchronisation: one thread issues every TMA copy and MMA; each batch of MMAs ends in one tcgen05.commit on an
// mbarrier that all 128 threads wait on (bounded, traps).  tcgen05 operations of one issuing thread complete in
// order, so the wait that precedes the softmax / gradient pass of a step also guarantees that the MMAs of the
// previous step no longer read the smem images that pass overwrites.
#include "common.cuh"
#include "tc_common.cuh"

namespace stepk {
using namespace tc;

constexpr int TAT_THREADS = 128;                       // four warps: one per TMEM lane quadrant
constexpr int TAT_HD = 24;
constexpr int TAT_PMAX = 352;
constexpr float TAT_QSCALE = 0.20412414523193154f * 1.4426950408889634f;   // log2(e) / sqrt(24)

// Keep decisions of the training attention: one 32-bit word per pair of keys (2c, 2c+1) of a query row
// (rowid = (sequence * 4 + head) * P + query); half j & 1 of it, read as a bf16 number, is compared with the threshold
// (keep_mask_bf16x2: keep probability exactly 1 - floor(65536 p) / 65536).  Forward (thread = query) and backward
// (thread = key) evaluate the same function.
__device__ __forceinline__ uint32_t attn_pair_word(uint64_t rowid, int j, uint32_t salt) {
  const uint64_t w = rowid * 256u + (uint32_t)(j >> 1);
  return hash32((uint32_t)w ^ salt ^ ((uint32_t)(w >> 32) * 0x85EBCA6Bu));
}
__device__ __forceinline__ bool attn_keep(uint64_t rowid, int j, uint32_t salt, uint32_t thr2) {
  return ((keep_mask_bf16x2(attn_pair_word(rowid, j, salt), thr2) >> ((j & 1) * 16)) & 1u) != 0;
}
__host__ __device__ __forceinline__ uint32_t attn_salt(uint64_t key) {
  return (uint32_t)key ^ ((uint32_t)(key >> 32) * 0x9E3779B9u);
}

__device__ __forceinline__ void zero_smem(uint8_t *p, uint32_t bytes) {
  for (uint32_t i = threadIdx.x; i < bytes / 16; i += blockDim.x) reinterpret_cast<uint4 *>(p)[i] = make_uint4(0, 0, 0, 0);
}

// ===========================================================================
// fp32 qkv rows [S*P, 288] (q | k | v, head h at columns h*24..) -> Q / K / V operand images; pads are zero
// ===========================================================================
__global__ void tc_attn_pack_kernel(const float *__restrict__ qkv, int S, int P, int Pk, int RT, uint4 *__restrict__ q_img,
                                    uint4 *__restrict__ k_img, uint4 *__restrict__ v_img, float *__restrict__ bound) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // (sequence, head, slot), slot fastest
  const int slots = RT * 128;
  if (idx >= (long long)S * 4 * slots) return;                              // slots is a multiple of 32: whole warps leave
  const int slot = (int)(idx % slots);
  const long long sh = idx / slots;
  const int h = (int)(sh & 3);
  const long long seq = sh >> 2;
  const float *base = qkv + (size_t)seq * P * 288 + h * TAT_HD;
  // Q: tile rt, image row r
  {
    const int rt = slot >> 7, r = slot & 127;
    const int p = rt * 128 + r - q_tail_offset(P, rt, h);
    const bool valid = r >= q_tail_offset(P, rt, h) && p < P;
    uint4 *o = q_img + ((size_t)sh * RT + rt) * 3 * 128 + r;
    float n2 = 0.f;
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) {
      float x[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) { x[j] = valid ? base[(size_t)p * 288 + cc * 8 + j] * TAT_QSCALE : 0.f; n2 = fmaf(x[j], x[j], n2); }
      o[cc * 128] = pack8_bf16(x);
    }
    if (bound != nullptr && valid) bound[(size_t)S * 4 + (size_t)sh * P + p] = sqrtf(n2);
  }
  // K, V: key row `slot`
  float kn = 0.f;
  if (slot < Pk) {
    const bool valid = slot < P;
    uint4 *ok = k_img + (size_t)sh * 3 * Pk + slot, *ov = v_img + (size_t)sh * 3 * Pk + slot;
    float n2 = 0.f;
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) {
      float xk[8], xv[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        xk[j] = valid ? base[(size_t)slot * 288 + 96 + cc * 8 + j] : 0.f;
        xv[j] = valid ? base[(size_t)slot * 288 + 192 + cc * 8 + j] : 0.f;
        n2 = fmaf(xk[j], xk[j], n2);
      }
      ok[(size_t)cc * Pk] = pack8_bf16(xk);
      ov[(size_t)cc * Pk] = pack8_bf16(xv);
    }
    kn = sqrtf(n2);
  }
  if (bound != nullptr) {
    // max_j |k_j| per (sequence, head): a warp holds 32 slots of one (sequence, head); non-negative floats order like
    // their bit patterns -> integer atomicMax
    kn = warp_max(kn);
    if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<uint32_t *>(bound) + sh, __float_as_uint(kn));
  }
}

// ===========================================================================
// forward
// ===========================================================================
struct TatFwdArgs {
  const uint8_t *q_img, *k_img, *v_img;
  float *out, *lse;
  int S, P, Pk, RT, tmem_cols;
  uint32_t thr2; float dscale; uint32_t salt;
};

__host__ __device__ inline uint32_t tat_fwd_smem(int Pk, int RT) {
  const uint32_t zrows = Pk > 128 ? Pk : 128;
  return RT * 6144u + 2u * 3u * Pk * 16u + zrows * 16u + (uint32_t)(Pk / 8) * 2048u + 64u;
}
__host__ __device__ inline int tat_fwd_tmem_cols(int Pk) { return Pk + 32 <= 128 ? 128 : Pk + 32 <= 256 ? 256 : 512; }

template <bool DROP>
__global__ void __launch_bounds__(TAT_THREADS) tc_attn_train_fwd_kernel(TatFwdArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int P = a.P, Pk = a.Pk, RT = a.RT;
  const int sh = blockIdx.x, h = sh & 3, seq = sh >> 2;
  const uint32_t KVB = 3u * Pk * 16u;
  uint8_t *sQ = smem;                       // RT x [3][128][8]
  uint8_t *sK = sQ + RT * 6144;             // [3][Pk][8]
  uint8_t *sV = sK + KVB;                   // [3][Pk][8]; the zero chunk right behind it is V's 4th (head dims 24..31) group
  uint8_t *sZ = sV + KVB;                   // zero chunk: max(128, Pk) rows x 16 B
  const uint32_t zrows = Pk > 128 ? Pk : 128;
  uint8_t *sP = sZ + zrows * 16;            // [Pk/8][128][8] probabilities
  uint64_t *bars = reinterpret_cast<uint64_t *>(sP + (size_t)(Pk / 8) * 2048);
  uint64_t *ld_bar = bars, *mma_bar = bars + 1;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2);
  const int warp = threadIdx.x >> 5, row = threadIdx.x;

  if (threadIdx.x == 0) {
    mbar_init(ld_bar, 1); mbar_init(mma_bar, 1);
    fence_barrier_init();
  }
  zero_smem(sZ, zrows * 16);
  fence_proxy_async();
  if (warp == 0) tmem_alloc(tmem_slot, a.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot, ocol = a.tmem_cols - 32;
  const uint32_t lane_base = (uint32_t)(warp * 32) << 16;

  if (threadIdx.x == 0) {
    mbar_expect_tx(ld_bar, RT * 6144u + 2u * KVB);
    tma_bulk_g2s(sQ, a.q_img + (size_t)sh * RT * 6144, RT * 6144u, ld_bar);
    tma_bulk_g2s(sK, a.k_img + (size_t)sh * KVB, KVB, ld_bar);
    tma_bulk_g2s(sV, a.v_img + (size_t)sh * KVB, KVB, ld_bar);
  }
  mbar_wait(ld_bar, 0);
  const uint32_t zaddr = smem_u32(sZ), ka = smem_u32(sK), va = smem_u32(sV), pa = smem_u32(sP);
  uint32_t phase = 0;
  for (int rt = 0; rt < RT; ++rt) {
    // ---- S = Q_rt K^T: N = Pk in pieces of <= 256 columns; k-step 1 = head dims 16..23 + the zero chunk ----
    if (threadIdx.x == 0) {
      tc_fence_after();
      const uint32_t qa = smem_u32(sQ + rt * 6144);
      for (int n0 = 0; n0 < Pk; n0 += 256) {
        const int nn = Pk - n0 < 256 ? Pk - n0 : 256;
        const uint32_t idesc = umma_idesc_bf16(128, nn, 0, 0), kb = ka + n0 * 16, kb2 = kb + 2 * Pk * 16;
        umma_bf16(tmem + n0, umma_desc(qa, 2048, 128), umma_desc(kb, Pk * 16, 128), idesc, 0u);
        umma_bf16(tmem + n0, umma_desc(qa + 4096, zaddr - (qa + 4096), 128), umma_desc(kb2, zaddr - kb2, 128), idesc, 1u);
      }
      umma_commit(mma_bar);
    }
    mbar_wait(mma_bar, phase); phase ^= 1;
    tc_fence_after();
    // ---- softmax of row `row` (TMEM lane): exact max, then p = 2^(s - m), fp32 row sum, bf16 image with dropout ----
    const int roff = q_tail_offset(P, rt, h), lrow = row - roff, p_row = rt * 128 + lrow;
    const bool valid = lrow >= 0 && p_row < P;
    float m = -INFINITY;
    for (int c0 = 0; c0 < Pk; c0 += 16) {
      float t[16];
      tmem_ld16(tmem + lane_base + c0, t);
#pragma unroll
      for (int c = 0; c < 16; ++c) if (c0 + c < P) m = fmaxf(m, t[c]);
    }
    const uint64_t rowid = ((uint64_t)sh * P + (uint32_t)p_row);
    float l0 = 0.f, l1 = 0.f;
    uint4 *prow = reinterpret_cast<uint4 *>(sP) + row;
    for (int c0 = 0; c0 < Pk; c0 += 16) {
      float t[16];
      tmem_ld16(tmem + lane_base + c0, t);
      uint32_t w[8];
#pragma unroll
      for (int c = 0; c < 16; c += 2) {
        const float e0 = c0 + c < P ? fast_exp2(t[c] - m) : 0.f;
        const float e1 = c0 + c + 1 < P ? fast_exp2(t[c + 1] - m) : 0.f;
        l0 += e0; l1 += e1;
        w[c / 2] = pack_bf16(e0, e1);
        if (DROP) w[c / 2] &= keep_mask_bf16x2(attn_pair_word(rowid, c0 + c, a.salt), a.thr2);
      }
      prow[(size_t)(c0 / 8) * 128] = make_uint4(w[0], w[1], w[2], w[3]);
      prow[(size_t)(c0 / 8 + 1) * 128] = make_uint4(w[4], w[5], w[6], w[7]);
    }
    const float l = l0 + l1;
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    // ---- O = P V: V is the MN-major B operand (N = 32 head dims, K = keys) ----
    if (threadIdx.x == 0) {
      tc_fence_after();
      const uint32_t idesc = umma_idesc_bf16(128, 32, 0, 1);
      for (int kk = 0; kk < Pk / 16; ++kk)
        umma_bf16(tmem + ocol, umma_desc(pa + kk * 4096, 2048, 128), umma_desc(va + kk * 256, 128, Pk * 16), idesc, kk != 0 ? 1u : 0u);
      umma_commit(mma_bar);
    }
    mbar_wait(mma_bar, phase); phase ^= 1;
    tc_fence_after();
    float o[32];
    tmem_ld32(tmem + lane_base + ocol, o);
    tc_fence_before();
    if (valid) {
      const float inv = a.dscale / l;
      float *dst = a.out + ((size_t)seq * P + p_row) * 96 + h * TAT_HD;
#pragma unroll
      for (int c = 0; c < TAT_HD; c += 4) *reinterpret_cast<float4 *>(dst + c) = make_float4(o[c] * inv, o[c + 1] * inv, o[c + 2] * inv, o[c + 3] * inv);
      a.lse[(size_t)sh * P + p_row] = m + __log2f(l);
    }
    // every thread has passed this phase of mma_bar before the next commit can complete another one
    __syncthreads();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, a.tmem_cols);
}

// ===========================================================================
// backward
// ===========================================================================
struct TatBwdArgs {
  const uint8_t *q_img, *k_img, *v_img;
  const float *out, *lse, *dout;
  float *dqkv;
  int S, P, Pk, RT;
  uint32_t thr2; float dscale; uint32_t salt;
};

__host__ __device__ inline uint32_t tat_bwd_smem(int RT) {
  // Q, dO tiles; K, V as [3][RT*128][8]; zero chunk; P^T and dS^T images [16][128][8]; L, D per query slot; barriers
  return 2u * RT * 6144u + 2u * 3u * RT * 128u * 16u + 2048u + 2u * 32768u + 2u * RT * 128u * 4u + 64u;
}

template <bool DROP>
__global__ void __launch_bounds__(TAT_THREADS) tc_attn_train_bwd_kernel(TatBwdArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int P = a.P, Pk = a.Pk, RT = a.RT, PR = RT * 128;
  const int sh = blockIdx.x, h = sh & 3, seq = sh >> 2;
  uint8_t *sQ = smem;                              // RT x [3][128][8]
  uint8_t *sO = sQ + RT * 6144;                    // dO, same layout as Q
  uint8_t *sK = sO + RT * 6144;                    // [3][PR][8]
  uint8_t *sV = sK + 3 * PR * 16;                  // [3][PR][8]
  uint8_t *sZ = sV + 3 * PR * 16;                  // zero chunk, 128 rows
  uint8_t *sPT = sZ + 2048;                        // [16 query chunks][128 keys][8]: (p keep / (1 - p))^T
  uint8_t *sDS = sPT + 32768;                      // same layout: dS^T
  float *sL = reinterpret_cast<float *>(sDS + 32768);    // [PR] per query slot: L (+inf on pad slots)
  float *sD = sL + PR;                                    // [PR] D
  uint64_t *bars = reinterpret_cast<uint64_t *>(sD + PR);
  uint64_t *ld_bar = bars, *mma_bar = bars + 1;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2);
  const int warp = threadIdx.x >> 5, row = threadIdx.x;
  // TMEM columns: S^T [0,128), dP^T [128,256), dV 256.., dK 288.., dQ of query tile qc at 320 + 32 qc
  constexpr uint32_t C_DP = 128, C_DV = 256, C_DK = 288, C_DQ = 320;

  if (threadIdx.x == 0) {
    mbar_init(ld_bar, 1); mbar_init(mma_bar, 1);
    fence_barrier_init();
  }
  zero_smem(sZ, 2048);
  // key rows [Pk, PR) of K and V (rows [P, Pk) arrive as zeros from the pack kernel)
  for (int i = threadIdx.x; i < 2 * 3 * (PR - Pk); i += blockDim.x) {
    const int n = PR - Pk, which = i / (3 * n), cc = (i / n) % 3, r = Pk + i % n;
    reinterpret_cast<uint4 *>(which ? sV : sK)[(size_t)cc * PR + r] = make_uint4(0, 0, 0, 0);
  }
  if (warp == 0) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t lane_base = (uint32_t)(warp * 32) << 16;

  if (threadIdx.x == 0) {
    const uint32_t kvc = (uint32_t)Pk * 16;
    mbar_expect_tx(ld_bar, RT * 6144u + 6u * kvc);
    tma_bulk_g2s(sQ, a.q_img + (size_t)sh * RT * 6144, RT * 6144u, ld_bar);
    for (int cc = 0; cc < 3; ++cc) {
      tma_bulk_g2s(sK + cc * PR * 16, a.k_img + (size_t)sh * 3 * kvc + cc * kvc, kvc, ld_bar);
      tma_bulk_g2s(sV + cc * PR * 16, a.v_img + (size_t)sh * 3 * kvc + cc * kvc, kvc, ld_bar);
    }
  }
  // dO tiles (bf16, same row placement as Q), L and D = dO . O (fp32) per query slot
  for (int slot = threadIdx.x; slot < PR; slot += blockDim.x) {
    const int rt = slot >> 7, r = slot & 127, roff = q_tail_offset(P, rt, h);
    const int p = rt * 128 + r - roff;
    const bool valid = r >= roff && p < P;
    uint4 *dst = reinterpret_cast<uint4 *>(sO) + rt * 3 * 128 + r;
    float d = 0.f;
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) {
      float g[8];
      if (valid) {
        const float4 *gp = reinterpret_cast<const float4 *>(a.dout + ((size_t)seq * P + p) * 96 + h * TAT_HD + cc * 8);
        const float4 *op = reinterpret_cast<const float4 *>(a.out + ((size_t)seq * P + p) * 96 + h * TAT_HD + cc * 8);
        const float4 g0 = gp[0], g1 = gp[1], o0 = op[0], o1 = op[1];
        g[0] = g0.x; g[1] = g0.y; g[2] = g0.z; g[3] = g0.w; g[4] = g1.x; g[5] = g1.y; g[6] = g1.z; g[7] = g1.w;
        d = fmaf(g0.x, o0.x, d); d = fmaf(g0.y, o0.y, d); d = fmaf(g0.z, o0.z, d); d = fmaf(g0.w, o0.w, d);
        d = fmaf(g1.x, o1.x, d); d = fmaf(g1.y, o1.y, d); d = fmaf(g1.z, o1.z, d); d = fmaf(g1.w, o1.w, d);
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) g[j] = 0.f;
      }
      dst[cc * 128] = pack8_bf16(g);
    }
    sL[slot] = valid ? a.lse[(size_t)sh * P + p] : INFINITY;
    sD[slot] = d;
  }
  fence_proxy_async();
  __syncthreads();
  mbar_wait(ld_bar, 0);

  const uint32_t zaddr = smem_u32(sZ), qa0 = smem_u32(sQ), oa0 = smem_u32(sO), ka0 = smem_u32(sK), va0 = smem_u32(sV);
  const uint32_t pta = smem_u32(sPT), dsa = smem_u32(sDS);
  const uint32_t idesc_s = umma_idesc_bf16(128, 128, 0, 0);
  const uint32_t idesc_kn = umma_idesc_bf16(128, 32, 0, 1);     // A K-major, B MN-major (dV, dK)
  const uint32_t idesc_mn = umma_idesc_bf16(128, 32, 1, 1);     // A MN-major, B MN-major (dQ)
  uint32_t phase = 0;
  for (int kt = 0; kt < RT; ++kt) {
    const int key = kt * 128 + row;
    const bool kvalid = key < P;
    for (int qc = 0; qc < RT; ++qc) {
      // ---- S^T = K_kt Q_qc^T and dP^T = V_kt dO_qc^T (M = 128 keys, N = 128 query slots, K = 24 + zero chunk) ----
      if (threadIdx.x == 0) {
        tc_fence_after();
#pragma unroll
        for (int which = 0; which < 2; ++which) {
          const uint32_t aa = (which ? va0 : ka0) + kt * 2048, a2 = aa + 2 * PR * 16;
          const uint32_t ba = (which ? oa0 : qa0) + qc * 6144, b2 = ba + 4096;
          const uint32_t d = tmem + (which ? C_DP : 0u);
          umma_bf16(d, umma_desc(aa, PR * 16, 128), umma_desc(ba, 2048, 128), idesc_s, 0u);
          umma_bf16(d, umma_desc(a2, zaddr - a2, 128), umma_desc(b2, zaddr - b2, 128), idesc_s, 1u);
        }
        umma_commit(mma_bar);
      }
      mbar_wait(mma_bar, phase); phase ^= 1;
      tc_fence_after();
      // ---- per key row: probabilities and dS for the 128 query slots ----
      const int roff = q_tail_offset(P, qc, h);
      const uint64_t rowid0 = (uint64_t)sh * P + (uint64_t)(qc * 128 - roff);    // rowid of slot 0 (slot c -> + c)
      const float *Lq = sL + qc * 128, *Dq = sD + qc * 128;
      uint4 *ptrow = reinterpret_cast<uint4 *>(sPT) + row, *dsrow = reinterpret_cast<uint4 *>(sDS) + row;
      for (int c0 = 0; c0 < 128; c0 += 16) {
        float s[16], dp[16];
        tmem_ld16(tmem + lane_base + c0, s);
        tmem_ld16(tmem + lane_base + C_DP + c0, dp);
        uint32_t wp[8], wd[8];
#pragma unroll
        for (int c = 0; c < 16; c += 2) {
          float pk[2], ds[2];
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int cs = c0 + c + e;
            const float pr = fast_exp2(s[c + e] - Lq[cs]);
            float g = dp[c + e] * a.dscale, pd = pr * a.dscale;
            if (DROP && !attn_keep(rowid0 + cs, key, a.salt, a.thr2)) { g = 0.f; pd = 0.f; }
            pk[e] = kvalid ? pd : 0.f;
            ds[e] = kvalid ? pr * (g - Dq[cs]) : 0.f;
          }
          wp[c / 2] = pack_bf16(pk[0], pk[1]);
          wd[c / 2] = pack_bf16(ds[0], ds[1]);
        }
        ptrow[(size_t)(c0 / 8) * 128] = make_uint4(wp[0], wp[1], wp[2], wp[3]);
        ptrow[(size_t)(c0 / 8 + 1) * 128] = make_uint4(wp[4], wp[5], wp[6], wp[7]);
        dsrow[(size_t)(c0 / 8) * 128] = make_uint4(wd[0], wd[1], wd[2], wd[3]);
        dsrow[(size_t)(c0 / 8 + 1) * 128] = make_uint4(wd[4], wd[5], wd[6], wd[7]);
      }
      fence_proxy_async();
      tc_fence_before();
      __syncthreads();
      // ---- dV_kt += P~^T dO_qc, dK_kt += dS^T Q_qc (K = 128 query slots), dQ_qc += dS K_kt (K = 128 keys) ----
      if (threadIdx.x == 0) {
        tc_fence_after();
        const uint32_t qa = qa0 + qc * 6144, oa = oa0 + qc * 6144;
        for (int kk = 0; kk < 8; ++kk) {
          const uint32_t acc = (qc | kk) != 0 ? 1u : 0u;
          umma_bf16(tmem + C_DV, umma_desc(pta + kk * 4096, 2048, 128), umma_desc(oa + kk * 256, 128, 2048), idesc_kn, acc);
          umma_bf16(tmem + C_DK, umma_desc(dsa + kk * 4096, 2048, 128), umma_desc(qa + kk * 256, 128, 2048), idesc_kn, acc);
          umma_bf16(tmem + C_DQ + qc * 32, umma_desc(dsa + kk * 256, 128, 2048),
                    umma_desc(ka0 + (kt * 128 + kk * 16) * 16, 128, PR * 16), idesc_mn, (kt | kk) != 0 ? 1u : 0u);
        }
        if (qc == RT - 1) umma_commit(mma_bar);
      }
    }
    // ---- dK, dV of this key tile ----
    mbar_wait(mma_bar, phase); phase ^= 1;
    tc_fence_after();
    float dv[32], dk[32];
    tmem_ld32(tmem + lane_base + C_DV, dv);
    tmem_ld32(tmem + lane_base + C_DK, dk);
    tc_fence_before();
    __syncthreads();         // all threads are past this phase of mma_bar (and done reading dV / dK) before the next commit
    if (kvalid) {
      float *dst = a.dqkv + ((size_t)seq * P + key) * 288 + h * TAT_HD;
      const float kscale = 0.69314718055994531f;    // dK = dS^T Q / sqrt(24) = ln(2) dS^T (Q log2(e) / sqrt(24))
#pragma unroll
      for (int c = 0; c < TAT_HD; c += 4) {
        *reinterpret_cast<float4 *>(dst + 96 + c) = make_float4(dk[c] * kscale, dk[c + 1] * kscale, dk[c + 2] * kscale, dk[c + 3] * kscale);
        *reinterpret_cast<float4 *>(dst + 192 + c) = make_float4(dv[c], dv[c + 1], dv[c + 2], dv[c + 3]);
      }
    }
  }
  // ---- dQ (every MMA completed before the last wait) ----
  for (int qc = 0; qc < RT; ++qc) {
    float dq[32];
    tmem_ld32(tmem + lane_base + C_DQ + qc * 32, dq);
    const int roff = q_tail_offset(P, qc, h), p = qc * 128 + row - roff;
    if (row >= roff && p < P) {
      float *dst = a.dqkv + ((size_t)seq * P + p) * 288 + h * TAT_HD;
      const float qs = 0.20412414523193154f;          // 1 / sqrt(24)
#pragma unroll
      for (int c = 0; c < TAT_HD; c += 4) *reinterpret_cast<float4 *>(dst + c) = make_float4(dq[c] * qs, dq[c + 1] * qs, dq[c + 2] * qs, dq[c + 3] * qs);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

// test helper: the keep decision of every (sequence, head, query, key)
__global__ void tc_attn_keep_mask_kernel(int S, int P, uint32_t thr2, uint32_t salt, uint8_t *__restrict__ mask) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)S * 4 * P * P) return;
  const int j = (int)(idx % P);
  mask[idx] = attn_keep((uint64_t)(idx / P), j, salt, thr2) ? 1 : 0;
}

struct DropCfg { uint32_t thr2; float dscale; uint32_t salt; bool live; };
static DropCfg drop_cfg(float drop_p, unsigned long long seed) {
  DropCfg c{0u, 1.f, attn_salt(rng_key(seed, 0)), false};
  if (drop_p > 0.f) { c.thr2 = drop_thr_bf16x2((uint32_t)(drop_p * 65536.0f)); c.dscale = 1.f / (1.f - drop_p); c.live = true; }
  return c;
}

}  // namespace stepk

using namespace stepk;

#define TAT_CHECK_SHAPE(what)                                                                                   \
  STEP_REQUIRE(S > 0 && P >= 1 && P <= TAT_PMAX, what ": S must be > 0 and P in [1, 352]");                     \
  STEP_REQUIRE(drop_p >= 0.f && drop_p < 1.f, what ": drop_p must be in [0, 1)")

extern "C" size_t step_tc_attn_train_lse_bytes(int S, int P) {
  if (S <= 0 || P <= 0) return 0;
  return (size_t)S * 4 * P * sizeof(float);
}

extern "C" int step_tc_attn_train_pack(const float *qkv, int S, int P, void *q_img, void *k_img, void *v_img, float *bound,
                                       void *stream) {
  STEP_REQUIRE(qkv && q_img && k_img && v_img, "tc_attn_train_pack: null pointer");
  STEP_REQUIRE(S > 0 && P >= 1 && P <= TAT_PMAX, "tc_attn_train_pack: S must be > 0 and P in [1, 352]");
  const cudaStream_t st = (cudaStream_t)stream;
  if (bound != nullptr) {
    const cudaError_t e = cudaMemsetAsync(bound, 0, (size_t)S * 4 * sizeof(float), st);
    if (e != cudaSuccess) return fail_msg((int)e, cudaGetErrorString(e));
  }
  const int Pk = (P + 15) / 16 * 16, RT = (P + 127) / 128;
  const long long n = (long long)S * 4 * RT * 128;
  tc_attn_pack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(qkv, S, P, Pk, RT, reinterpret_cast<uint4 *>(q_img),
                                                                   reinterpret_cast<uint4 *>(k_img), reinterpret_cast<uint4 *>(v_img), bound);
  return check_launch("tc_attn_pack_kernel");
}

extern "C" int step_tc_attn_train_fwd(const void *q_img, const void *k_img, const void *v_img, int S, int P, float drop_p,
                                      unsigned long long seed, float *out, float *lse, void *stream) {
  STEP_REQUIRE(q_img && k_img && v_img && out && lse, "tc_attn_train_fwd: null pointer");
  TAT_CHECK_SHAPE("tc_attn_train_fwd");
  TatFwdArgs a{};
  a.q_img = (const uint8_t *)q_img; a.k_img = (const uint8_t *)k_img; a.v_img = (const uint8_t *)v_img;
  a.out = out; a.lse = lse;
  a.S = S; a.P = P; a.Pk = (P + 15) / 16 * 16; a.RT = (P + 127) / 128; a.tmem_cols = tat_fwd_tmem_cols(a.Pk);
  const DropCfg d = drop_cfg(drop_p, seed);
  a.thr2 = d.thr2; a.dscale = d.dscale; a.salt = d.salt;
  const size_t smem = tat_fwd_smem(a.Pk, a.RT);
  const cudaStream_t st = (cudaStream_t)stream;
  int rc;
  if (d.live) {
    if ((rc = allow_smem(tc_attn_train_fwd_kernel<true>, smem))) return rc;
    tc_attn_train_fwd_kernel<true><<<S * 4, TAT_THREADS, smem, st>>>(a);
  } else {
    if ((rc = allow_smem(tc_attn_train_fwd_kernel<false>, smem))) return rc;
    tc_attn_train_fwd_kernel<false><<<S * 4, TAT_THREADS, smem, st>>>(a);
  }
  return check_launch("tc_attn_train_fwd_kernel");
}

extern "C" int step_tc_attn_train_bwd(const void *q_img, const void *k_img, const void *v_img, const float *out, const float *lse,
                                      const float *dout, int S, int P, float drop_p, unsigned long long seed, float *dqkv,
                                      void *stream) {
  STEP_REQUIRE(q_img && k_img && v_img && out && lse && dout && dqkv, "tc_attn_train_bwd: null pointer");
  TAT_CHECK_SHAPE("tc_attn_train_bwd");
  TatBwdArgs a{};
  a.q_img = (const uint8_t *)q_img; a.k_img = (const uint8_t *)k_img; a.v_img = (const uint8_t *)v_img;
  a.out = out; a.lse = lse; a.dout = dout; a.dqkv = dqkv;
  a.S = S; a.P = P; a.Pk = (P + 15) / 16 * 16; a.RT = (P + 127) / 128;
  const DropCfg d = drop_cfg(drop_p, seed);
  a.thr2 = d.thr2; a.dscale = d.dscale; a.salt = d.salt;
  const size_t smem = tat_bwd_smem(a.RT);
  const cudaStream_t st = (cudaStream_t)stream;
  int rc;
  if (d.live) {
    if ((rc = allow_smem(tc_attn_train_bwd_kernel<true>, smem))) return rc;
    tc_attn_train_bwd_kernel<true><<<S * 4, TAT_THREADS, smem, st>>>(a);
  } else {
    if ((rc = allow_smem(tc_attn_train_bwd_kernel<false>, smem))) return rc;
    tc_attn_train_bwd_kernel<false><<<S * 4, TAT_THREADS, smem, st>>>(a);
  }
  return check_launch("tc_attn_train_bwd_kernel");
}

extern "C" int step_tc_attn_train_keep_mask(int S, int P, float drop_p, unsigned long long seed, unsigned char *mask, void *stream) {
  STEP_REQUIRE(mask, "tc_attn_train_keep_mask: null pointer");
  TAT_CHECK_SHAPE("tc_attn_train_keep_mask");
  const DropCfg d = drop_cfg(drop_p, seed);
  const long long n = (long long)S * 4 * P * P;
  if (!d.live) {
    const cudaError_t e = cudaMemsetAsync(mask, 1, (size_t)n, (cudaStream_t)stream);
    return e == cudaSuccess ? STEP_OK : fail_msg((int)e, cudaGetErrorString(e));
  }
  tc_attn_keep_mask_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(S, P, d.thr2, d.salt, mask);
  return check_launch("tc_attn_keep_mask_kernel");
}
