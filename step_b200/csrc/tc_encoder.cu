// TSFormer encoder on the 5th-generation tensor cores: tcgen05.mma with TMEM accumulators, operands
// staged by 1-D TMA bulk copies of UMMA-canonical "tile images", warp-specialised (TMA producer /
// single-thread MMA issuer / epilogue or softmax warps) and mbarrier-pipelined.  bf16 operands, fp32
// accumulation, fp32 LayerNorm / softmax statistics.
//
// Reference semantics are those of csrc/ts_encoder.cu (same citations); this file is the
// "bf16 precision" implementation of SURVEY.md section 8 rows T1-T4.
//
// Inter-kernel activation format ("tile image", see tc_common.cuh): a [T, K] activation is stored as
// [T/128 tiles][K/8 chunks][128 rows][8] bf16.  Producers write it with perfectly coalesced 16-byte
// stores (lane = row), consumers fetch a whole 128 x 96 K-slice (24 KB) with ONE cp.async.bulk.
#include "common.cuh"
#include "tc_common.cuh"

namespace stepk {
using namespace tc;

constexpr int TCL_THREADS = 320;                 // warp 0: TMA, warp 1: MMA, warps 2-5 / 6-9: two epilogue groups
constexpr int TCL_STAGES = 4;
constexpr uint32_t SLICE_BYTES = 12 * 2048;      // 128 rows x 96 K, bf16
constexpr int HD = 24;                           // head dim

enum { TCM_F32 = 0, TCM_RELU_IMG = 1, TCM_RESLN = 2, TCM_QKV = 3 };

// Dropout masks of the tensor-core path: one counter hash (hash32 in tc_common.cuh) seeds each group of 8 consecutive
// elements, a 32-bit LCG step per element (one IMAD) walks the group, and the full 32-bit state is compared with the
// threshold (keep probability exactly 1 - thr16 / 65536).  ~4 integer ops per element instead of ~50 for
// Philox4x32-10, which matters because TSFormer draws 3.0 G attention-probability masks per step; still counter-based,
// so a mask is a pure function of (seed, site, element index).
__device__ __forceinline__ void drop8(float *v, uint64_t idx8, uint32_t thr16, float scale, uint64_t key) {
  const uint32_t salt = (uint32_t)key ^ ((uint32_t)(key >> 32) * 0x9E3779B9u) ^ ((uint32_t)(idx8 >> 32) * 0x85EBCA6Bu);
  uint32_t st = hash32((uint32_t)idx8 ^ salt);
  const uint32_t thr = thr16 << 16;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    st = st * 2891336453u + 1013904223u;          // full-period LCG mod 2^32 (L'Ecuyer multiplier); high bits decide
    v[i] = (st >= thr) ? v[i] * scale : 0.f;
  }
}
// One block of NC score columns of a row: p = 2^(s - m) (0 for columns >= `valid`), row sums, dropout, bf16 K-major image.
// `dst` points at this row's 16-byte slot of the block's first 8-column chunk; chunks at or beyond `chunks` are not stored.
template <int NC, bool DROP, bool PRED>
__device__ __forceinline__ void softmax_cols(float (&t)[NC], float negm, int valid, int chunks, float &l0, float &l1, float &l2,
                                             float &l3, uint32_t st, uint32_t cadd, uint32_t thr2, uint4 *dst) {
#pragma unroll
  for (int c = 0; c < NC; c += 4) {
    tc::fadd2(t[c], t[c + 1], negm, negm);
    tc::fadd2(t[c + 2], t[c + 3], negm, negm);
    t[c] = fast_exp2(t[c]); t[c + 1] = fast_exp2(t[c + 1]); t[c + 2] = fast_exp2(t[c + 2]); t[c + 3] = fast_exp2(t[c + 3]);
    if (PRED) {
      if (c >= valid) t[c] = 0.f;
      if (c + 1 >= valid) t[c + 1] = 0.f;
      if (c + 2 >= valid) t[c + 2] = 0.f;
      if (c + 3 >= valid) t[c + 3] = 0.f;
    }
    tc::fadd2(l0, l1, t[c], t[c + 1]);
    tc::fadd2(l2, l3, t[c + 2], t[c + 3]);
  }
#pragma unroll
  for (int cc = 0; cc < NC / 8; ++cc) {
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      w[j] = tc::pack_bf16(t[cc * 8 + 2 * j], t[cc * 8 + 2 * j + 1]);
      if (DROP) {
        st = st * 2891336453u + cadd;             // full-period LCG mod 2^32 (odd addend, one IMAD); both halves decide
        w[j] &= keep_mask_bf16x2(st, thr2);
      }
    }
    if (!PRED || cc < chunks) dst[(size_t)cc * 128] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// ===========================================================================
// weight packing: fp32 W [Nout][K] -> bf16 image [K/8][Nout][8]
// ===========================================================================
__global__ void tc_pack_weight_kernel(const float *__restrict__ w, int Nout, int K, uint4 *__restrict__ img) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;   // one 16-byte unit
  if (idx >= Nout * (K / 8)) return;
  const int c = idx / Nout, n = idx % Nout;
  float v[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = w[(size_t)n * K + c * 8 + i];
  img[idx] = pack8_bf16(v);
}

// row-major fp32 [T][K] <-> tile image (test / debug helpers)
__global__ void tc_rows_to_image_kernel(const float *__restrict__ x, long long T, int K, uint4 *__restrict__ img) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int KC = K / 8;
  const long long MT = (T + 127) / 128;
  if (idx >= MT * KC * 128) return;
  const int r = (int)(idx % 128);
  const int c = (int)((idx / 128) % KC);
  const long long mt = idx / (128LL * KC);
  const long long t = mt * 128 + r;
  float v[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = (t < T) ? x[t * K + c * 8 + i] : 0.f;
  img[idx] = pack8_bf16(v);
}
__global__ void tc_image_to_rows_kernel(const uint4 *__restrict__ img, long long T, int K, float *__restrict__ x) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int KC = K / 8;
  const long long MT = (T + 127) / 128;
  if (idx >= MT * KC * 128) return;
  const int r = (int)(idx % 128);
  const int c = (int)((idx / 128) % KC);
  const long long mt = idx / (128LL * KC);
  const long long t = mt * 128 + r;
  if (t >= T) return;
  float v[8];
  unpack8_bf16(img[idx], v);
#pragma unroll
  for (int i = 0; i < 8; ++i) x[t * K + c * 8 + i] = v[i];
}

// fp32 hidden states [B,N,P,96] -> sequence-major bf16 image [B][P*12][R][8] (Gram operand); used when the
// hidden states were assembled by an all-gather of node shards
__global__ void tc_hidden_to_seq_image_kernel(const float *__restrict__ h, int B, int N, int P, int R, uint4 *__restrict__ img) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;    // (b, kc, n) with n fastest
  const long long KC = (long long)P * 12;
  if (idx >= (long long)B * KC * N) return;
  const int n = (int)(idx % N);
  const long long kc = (idx / N) % KC;
  const long long b = idx / ((long long)N * KC);
  const int p = (int)(kc / 12), cc = (int)(kc % 12);
  const float *src = h + (((size_t)b * N + n) * P + p) * 96 + cc * 8;
  float v[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) v[j] = src[j];
  img[((size_t)b * KC + kc) * R + n] = pack8_bf16(v);
}

// ===========================================================================
// patch embedding -> X tile image.  block = (32 patches, 16 nodes, b) = 512 tokens; the series tile is staged
// through smem (coalesced node-major reads); thread = (feature chunk c, token lane): the 8 x 12 weights of its
// chunk live in registers and the thread walks over the block's tokens, so the inner loop is 12 broadcast-free
// LDS + 96 FMA + one coalesced 16-byte image store per token.
// ===========================================================================
__global__ void __launch_bounds__(256) tc_embed_kernel(const float *__restrict__ series, long long sB, long long sT,
                                                       long long sN, int N, int P, const float *__restrict__ w,
                                                       const float *__restrict__ bias, const float *__restrict__ pos,
                                                       uint4 *__restrict__ img, uint32_t thr16, float dscale, uint64_t key) {
  __shared__ float sv[16][32 * 13 + 3];   // [node][patch][13]: 12 time steps + 1 pad word (conflict-free strided reads)
  const int b = blockIdx.z, n0 = blockIdx.y * 16, p0 = blockIdx.x * 32, tid = threadIdx.x;
  const int np = min(32, P - p0);
  for (int i = tid; i < 16 * np * 12; i += 256) {
    const int nn = i & 15, tt = i >> 4;
    const int n = n0 + nn;
    sv[nn][(tt / 12) * 13 + tt % 12] = (n < N) ? series[b * sB + (long long)(p0 * 12 + tt) * sT + n * sN] : 0.f;
  }
  const int c = tid / 21, lane = tid % 21;          // 12 chunks x 21 token lanes (252 of 256 threads): a warp stores consecutive image rows
  float wr[8][12], br[8];
  if (c < 12) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      br[j] = bias[c * 8 + j];
#pragma unroll
      for (int t = 0; t < 12; ++t) wr[j][t] = w[(c * 8 + j) * 12 + t];
    }
  }
  __syncthreads();
  if (c >= 12) return;
  const float scale = sqrtf(96.f);
  for (int tk = lane; tk < 16 * np; tk += 21) {
    const int nn = tk / np, pp = tk - nn * np;      // consecutive lanes -> consecutive patches of one node: consecutive image rows
    const int n = n0 + nn;
    if (n >= N) break;
    const int p = p0 + pp;
    float x[12];
#pragma unroll
    for (int t = 0; t < 12; ++t) x[t] = sv[nn][pp * 13 + t];
    const float4 pa = *reinterpret_cast<const float4 *>(pos + (size_t)p * 96 + c * 8);
    const float4 pb = *reinterpret_cast<const float4 *>(pos + (size_t)p * 96 + c * 8 + 4);
    float v[8] = {pa.x, pa.y, pa.z, pa.w, pb.x, pb.y, pb.z, pb.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float acc = br[j] + v[j];
#pragma unroll
      for (int t = 0; t < 12; ++t) acc = fmaf(wr[j][t], x[t], acc);
      v[j] = acc;
    }
    const long long token = ((long long)(b * N + n)) * P + p;
    if (thr16) drop8(v, (uint64_t)token * 12 + c, thr16, dscale, key);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] *= scale;
    img[((token >> 7) * 12 + c) * 128 + (token & 127)] = pack8_bf16(v);
  }
}

// ===========================================================================
// token GEMM on tcgen05:  out = epilogue( A[T,K] W^T + b )
// ===========================================================================
struct TcLinearArgs {
  const uint8_t *A;        // tile image [MT][K/8][128][8]
  const uint8_t *W;        // weight image [K/8][Nout][8]
  const float *bias;       // [Nout]
  int MT, K, Nout, mode;
  long long T;             // valid rows
  const uint8_t *res;      // residual tile image [MT][12][128][8] (TCM_RESLN)
  const float *ln_w, *ln_b, *ln2_w, *ln2_b;
  uint8_t *out_img;        // TCM_RELU_IMG: [MT][Nout/8][128][8]; TCM_RESLN: [MT][12][128][8] (may be null)
  float *out_f32;          // TCM_F32: [T][Nout]; TCM_RESLN: [T][96] (may be null)
  uint8_t *seq_img;        // TCM_RESLN: per-sample K-major image [B][P*12 chunks][seq_rows][8] of the output (Gram operand)
  int seq_nodes, seq_rows; // nodes per sample, padded rows per chunk
  uint8_t *q_img, *k_img, *v_img;  // TCM_QKV
  float *bound;            // TCM_QKV: [nseq*4] max_j |k_j| (zeroed by the host), then [nseq*4][P] |q_i|; may be null
  long long nseq;
  int P, Pk, RT;
  float qscale;
  uint32_t thr16; float dscale; uint64_t key;
};

__device__ __forceinline__ void layer_norm96(float *v, const float *w, const float *b) {
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
  for (int c = 0; c < 96; c += 4) { s0 += v[c]; s1 += v[c + 1]; s2 += v[c + 2]; s3 += v[c + 3]; }
  const float mean = ((s0 + s1) + (s2 + s3)) * (1.f / 96.f);
  float q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f;
#pragma unroll
  for (int c = 0; c < 96; c += 4) {
    const float d0 = v[c] - mean, d1 = v[c + 1] - mean, d2 = v[c + 2] - mean, d3 = v[c + 3] - mean;
    q0 = fmaf(d0, d0, q0); q1 = fmaf(d1, d1, q1); q2 = fmaf(d2, d2, q2); q3 = fmaf(d3, d3, q3);
  }
  const float rstd = rsqrtf(((q0 + q1) + (q2 + q3)) * (1.f / 96.f) + 1e-5f);
#pragma unroll
  for (int c = 0; c < 96; ++c) v[c] = (v[c] - mean) * rstd * w[c] + b[c];
}

// MODE: epilogue (compile-time so that each variant gets its own register allocation);
// FINAL: last encoder layer (second LayerNorm, fp32 row-major hidden states, optional Gram operand image)
template <int MODE, bool FINAL>
__global__ void __launch_bounds__(TCL_THREADS, 1) tc_linear_kernel(TcLinearArgs a) {
  constexpr int mode = MODE;
  extern __shared__ __align__(1024) uint8_t smem[];
  const int KS = a.K / 96, NB = a.Nout / 96;
  const uint32_t wbytes = (uint32_t)a.K * a.Nout * 2;
  uint8_t *sW = smem;
  uint8_t *sA = smem + wbytes;
  uint64_t *bars = reinterpret_cast<uint64_t *>(sA + TCL_STAGES * SLICE_BYTES);
  uint64_t *full = bars, *empty = bars + TCL_STAGES, *tfull = bars + 2 * TCL_STAGES, *tempty = tfull + 4, *wbar = tempty + 4;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(wbar + 1);
  float *sBias = reinterpret_cast<float *>(bars + 32);     // [Nout] bias, then 4 x [96] LayerNorm vectors
  float *sLn = sBias + 384;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < a.Nout; i += blockDim.x) sBias[i] = a.bias[i];
  if (mode == TCM_RESLN) {
    for (int i = threadIdx.x; i < 96; i += blockDim.x) {
      sLn[i] = a.ln_w[i]; sLn[96 + i] = a.ln_b[i];
      sLn[192 + i] = a.ln2_w ? a.ln2_w[i] : 1.f; sLn[288 + i] = a.ln2_b ? a.ln2_b[i] : 0.f;
    }
  }

  if (threadIdx.x == 0) {
    for (int i = 0; i < TCL_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 4; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 4); }
    mbar_init(wbar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      mbar_expect_tx(wbar, wbytes);
      tma_bulk_g2s(sW, a.W, wbytes, wbar);
      uint32_t n = 0;
      for (int mt = blockIdx.x; mt < a.MT; mt += gridDim.x) {
        for (int ks = 0; ks < KS; ++ks, ++n) {
          const uint32_t s = n % TCL_STAGES, ph = (n / TCL_STAGES) & 1;
          mbar_wait(&empty[s], ph ^ 1);
          mbar_expect_tx(&full[s], SLICE_BYTES);
          tma_bulk_g2s(sA + s * SLICE_BYTES, a.A + ((size_t)mt * KS + ks) * SLICE_BYTES, SLICE_BYTES, &full[s]);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ MMA issuer (one thread) ------------------------------
    if (lane == 0) {
      mbar_wait(wbar, 0);
      const uint32_t idesc = umma_idesc_bf16(128, 96, 0, 0);
      const uint32_t sA_addr = smem_u32(sA), sW_addr = smem_u32(sW);
      const uint32_t w_lbo = (uint32_t)a.Nout * 16;
      uint32_t n = 0, it = 0;
      for (int mt = blockIdx.x; mt < a.MT; mt += gridDim.x, ++it) {
        for (int ks = 0; ks < KS; ++ks, ++n) {
          const uint32_t s = n % TCL_STAGES, ph = (n / TCL_STAGES) & 1;
          mbar_wait(&full[s], ph);
          tc_fence_after();
          for (int nb = 0; nb < NB; ++nb) {
            const uint32_t jj = it * NB + nb, slot = jj & 3, use = jj >> 2;
            if (ks == 0) {
              mbar_wait(&tempty[slot], (use & 1) ^ 1);
              tc_fence_after();
            }
#pragma unroll
            for (int kk = 0; kk < 6; ++kk) {
              const uint64_t adesc = umma_desc(sA_addr + s * SLICE_BYTES + kk * 2 * 2048, 2048, 128);
              const uint32_t cidx = ks * 12 + kk * 2;
              const uint64_t bdesc = umma_desc(sW_addr + cidx * w_lbo + nb * 96 * 16, w_lbo, 128);
              umma_bf16(tmem + slot * 96, adesc, bdesc, idesc, (ks | kk) != 0 ? 1u : 0u);
            }
          }
          umma_commit(&empty[s]);
          if (ks == KS - 1) {
            for (int nb = 0; nb < NB; ++nb) umma_commit(&tfull[(it * NB + nb) & 3]);
          }
        }
      }
    }
  } else {
    // ------------------------------ epilogue warps ------------------------------
    // two groups of four warps take alternate [128 x 96] sub-tiles (accumulator slots 0,2 / 1,3), so that one
    // group's TMEM loads / LayerNorm / stores overlap the other's
    const int q = warp & 3;                 // TMEM lane quadrant this warp may access
    const int grp = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    uint32_t it = 0;
    for (int mt = blockIdx.x; mt < a.MT; mt += gridDim.x, ++it) {
      const long long token = (long long)mt * 128 + row;
      const bool valid = token < a.T;
      for (int nb = 0; nb < NB; ++nb) {
        const uint32_t jj = it * NB + nb, slot = jj & 3, use = jj >> 2;
        if ((int)(jj & 1) != grp) continue;
        mbar_wait(&tfull[slot], use & 1);
        tc_fence_after();
        float v[96];
        {
          const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + slot * 96;
          float t0[32];
          tmem_ld32(taddr, t0);
#pragma unroll
          for (int c = 0; c < 32; ++c) v[c] = t0[c];
          tmem_ld32(taddr + 32, t0);
#pragma unroll
          for (int c = 0; c < 32; ++c) v[32 + c] = t0[c];
          tmem_ld32(taddr + 64, t0);
#pragma unroll
          for (int c = 0; c < 32; ++c) v[64 + c] = t0[c];
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[slot]);

        {
          const float4 *bias4 = reinterpret_cast<const float4 *>(sBias + nb * 96);
#pragma unroll
          for (int c4 = 0; c4 < 24; ++c4) {
            const float4 bb = bias4[c4];
            v[4 * c4] += bb.x; v[4 * c4 + 1] += bb.y; v[4 * c4 + 2] += bb.z; v[4 * c4 + 3] += bb.w;
          }
        }

        if (mode == TCM_F32) {
          if (valid) {
            float *o = a.out_f32 + token * a.Nout + nb * 96;
#pragma unroll
            for (int c = 0; c < 96; c += 4) *reinterpret_cast<float4 *>(o + c) = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
          }
        } else if (mode == TCM_RELU_IMG) {
          uint4 *o = reinterpret_cast<uint4 *>(a.out_img) + ((size_t)mt * (a.Nout / 8) + nb * 12) * 128 + row;
#pragma unroll
          for (int cc = 0; cc < 12; ++cc) {
            float x[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) x[j] = fmaxf(v[cc * 8 + j], 0.f);
            if (a.thr16) drop8(x, ((uint64_t)token * a.Nout + nb * 96) / 8 + cc, a.thr16, a.dscale, a.key);
            o[cc * 128] = pack8_bf16(x);
          }
        } else if (mode == TCM_RESLN) {
          const uint4 *res = reinterpret_cast<const uint4 *>(a.res) + ((size_t)mt * 12) * 128 + row;
#pragma unroll
          for (int cc = 0; cc < 12; ++cc) {
            if (a.thr16) drop8(&v[cc * 8], (uint64_t)token * 12 + cc, a.thr16, a.dscale, a.key);
            float r8[8];
            unpack8_bf16(res[cc * 128], r8);
#pragma unroll
            for (int j = 0; j < 8; ++j) v[cc * 8 + j] += r8[j];
          }
          layer_norm96(v, sLn, sLn + 96);
          if (FINAL && a.ln2_w != nullptr) layer_norm96(v, sLn + 192, sLn + 288);
          if (!FINAL || a.out_img != nullptr) {
            uint4 *o = reinterpret_cast<uint4 *>(a.out_img) + ((size_t)mt * 12) * 128 + row;
#pragma unroll
            for (int cc = 0; cc < 12; ++cc) o[cc * 128] = pack8_bf16(&v[cc * 8]);
          }
          if (FINAL && a.out_f32 != nullptr && valid) {
            float *o = a.out_f32 + token * 96;
#pragma unroll
            for (int c = 0; c < 96; c += 4) *reinterpret_cast<float4 *>(o + c) = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
          }
          if (FINAL && a.seq_img != nullptr && valid) {
            // row = node, K index = (patch, feature): the operand layout of the cosine-similarity Gram GEMM
            const long long sq = token / a.P;
            const int pp = (int)(token - sq * a.P);
            const long long bb = sq / a.seq_nodes;
            const int nn = (int)(sq - bb * a.seq_nodes);
            uint4 *o = reinterpret_cast<uint4 *>(a.seq_img) + ((size_t)bb * a.P * 12 + (size_t)pp * 12) * a.seq_rows + nn;
#pragma unroll
            for (int cc = 0; cc < 12; ++cc) o[(size_t)cc * a.seq_rows] = pack8_bf16(&v[cc * 8]);
          }
        } else {  // TCM_QKV: nb 0 -> Q (pre-scaled into the log2 softmax domain), 1 -> K, 2 -> V
          if (valid) {
            const long long s = token / a.P;
            const int p = (int)(token - s * a.P);
            if (nb == 0) {
              const int rt = p >> 7;
#pragma unroll
              for (int h = 0; h < 4; ++h) {
                const int r = (p & 127) + q_tail_offset(a.P, rt, h);
                uint4 *o = reinterpret_cast<uint4 *>(a.q_img) + (((size_t)s * 4 + h) * a.RT + rt) * 3 * 128 + r;
                float n2 = 0.f;
#pragma unroll
                for (int cc = 0; cc < 3; ++cc) {
                  float x[8];
#pragma unroll
                  for (int j = 0; j < 8; ++j) { x[j] = v[h * HD + cc * 8 + j] * a.qscale; n2 = fmaf(x[j], x[j], n2); }
                  o[cc * 128] = pack8_bf16(x);
                }
                // |q_i| for the attention kernel's row-maximum bound (the 1 % margin there covers the bf16 rounding)
                if (a.bound != nullptr) a.bound[(size_t)a.nseq * 4 + ((size_t)s * 4 + h) * a.P + p] = sqrtf(n2);
              }
            } else {
              uint8_t *base = (nb == 1) ? a.k_img : a.v_img;
#pragma unroll
              for (int h = 0; h < 4; ++h) {
                uint4 *o = reinterpret_cast<uint4 *>(base) + ((size_t)s * 4 + h) * 3 * a.Pk + p;
#pragma unroll
                for (int cc = 0; cc < 3; ++cc) o[(size_t)cc * a.Pk] = pack8_bf16(&v[h * HD + cc * 8]);
              }
            }
          }
          if (nb == 1 && a.bound != nullptr) {
            // max_j |k_j| per (sequence, head): non-negative floats order like their bit patterns -> integer atomicMax.
            // A warp holds 32 consecutive tokens; when they share one sequence a shuffle reduction leaves 4 atomics.
            const long long s = valid ? token / a.P : -1;
            const long long s0 = __shfl_sync(0xffffffffu, s, 0);
            const bool same = __all_sync(0xffffffffu, s == s0);
#pragma unroll
            for (int h = 0; h < 4; ++h) {
              float n2 = 0.f;
#pragma unroll
              for (int c = 0; c < HD; ++c) n2 = fmaf(v[h * HD + c], v[h * HD + c], n2);
              float kn = valid ? sqrtf(n2) : 0.f;
              uint32_t *dst = reinterpret_cast<uint32_t *>(a.bound);
              if (same) {
                kn = warp_max(kn);
                if (lane == 0 && s0 >= 0) atomicMax(dst + s0 * 4 + h, __float_as_uint(kn));
              } else if (valid) {
                atomicMax(dst + s * 4 + h, __float_as_uint(kn));
              }
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// ===========================================================================
// attention on tcgen05.  Persistent CTA (one per SM) streaming (sequence, head, row-tile) iterations:
//   S = Q K^T   (M=128, N=Pk, K=32: head dim 24 padded with a shared zero chunk in smem)
//   P = softmax rows (fp32 statistics read from TMEM, exp2 domain), written as a bf16 K-major image in smem
//   O = P V     (M=128, N=32, K=Pk; V is the MN-major B operand)
// Warp roles: warp 0 TMA producer, warp 1 MMA issuer, warps 2-5 and 6-9 two softmax groups that take
// alternate iterations with private S/O accumulators in TMEM and private P images (ping-pong): while one
// group exponentiates, the tensor core computes the other group's S and P.V.
// ===========================================================================
struct TcAttnArgs {
  const uint8_t *q_img, *k_img, *v_img;
  uint8_t *o_img;
  const float *bound;      // [S*4] max_j |k_j| (as uint bits) then [S*4][P] |q_i| of the bf16 operands; null -> exact row maxima
  int S, P, Pk, RT;
  uint32_t thr16; float dscale; uint64_t key;
};

constexpr int TCA_THREADS = 320;
constexpr int TCA_QBUF = 4, TCA_KVBUF = 3;
constexpr int TCA_KSPLIT = 176, TCA_KVBUF_SPLIT = 2, TCA_XROW = 27;   // key-split mode (P > 176)

// PF > 0: sequence length known at compile time (168 for every 2016-step STEP config) -> unrolled column loops
// without bounds predicates; DROP: attention-probability dropout compiled in or out.
//
// SPLIT (176 < P <= 352, e.g. the 4032-step PEMS03/04/08 histories with P = 336): one S accumulator no longer fits
// next to its ping-pong twin in the 512 TMEM columns, so the two softmax groups share every (sequence, head,
// row tile) iteration instead of alternating: group 0 owns keys [0, 176), group 1 keys [176, P).  Each computes
// a local max / sum and a partial O = P_g V_g in its private TMEM region; the halves are merged flash-decoding
// style through a small shared-memory exchange (O = (O0 2^(m0-m) + O1 2^(m1-m)) / (l0 2^(m0-m) + l1 2^(m1-m))).
template <int PF, bool DROP, bool SPLIT>
__global__ void __launch_bounds__(TCA_THREADS, 1) tc_attn_kernel(TcAttnArgs a) {
  static_assert(PF == 0 || PF == 168 || PF == 336, "compile-time sequence lengths: 168 (alternating groups) or 336 (key split)");
  extern __shared__ __align__(1024) uint8_t smem[];
  const int P = PF > 0 ? PF : a.P, Pk = PF > 0 ? (PF + 15) / 16 * 16 : a.Pk, RT = PF > 0 ? (PF + 127) / 128 : a.RT;
  constexpr int KVBUFS = SPLIT ? TCA_KVBUF_SPLIT : TCA_KVBUF;
  const uint32_t KVB = 3u * Pk * 16;          // bytes of one K (or V) image
  const uint32_t PB = SPLIT ? (uint32_t)(TCA_KSPLIT / 8) * 2048 : (uint32_t)(Pk / 8) * 2048;
  uint8_t *sQ = smem;                          // TCA_QBUF x 6144
  uint8_t *sK = sQ + TCA_QBUF * 6144;          // KVBUFS x KVB
  uint8_t *sV = sK + KVBUFS * KVB;             // KVBUFS x KVB
  uint8_t *sZ = sV + KVBUFS * KVB;             // zero chunk: max(128, Pk) rows x 16 B
  const uint32_t zrows = Pk > 128 ? Pk : 128;
  uint8_t *sP = sZ + zrows * 16;               // 2 x [cols/8][128][16 B]
  float *xch = reinterpret_cast<float *>(sP + 2 * PB);   // SPLIT: 2 x [128 rows][TCA_XROW] merge exchange
  uint64_t *bars = reinterpret_cast<uint64_t *>(sP + 2 * PB + (SPLIT ? 2 * 128 * TCA_XROW * 4 : 0));
  uint64_t *q_full = bars, *q_empty = bars + 4, *kv_full = bars + 8, *kv_empty = bars + 11;
  uint64_t *s_full = bars + 14, *s_empty = bars + 16, *p_ready = bars + 18, *o_full = bars + 20, *o_empty = bars + 22;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 24);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < TCA_QBUF; ++i) { mbar_init(&q_full[i], 1); mbar_init(&q_empty[i], 1); }
    for (int i = 0; i < KVBUFS; ++i) { mbar_init(&kv_full[i], 1); mbar_init(&kv_empty[i], 1); }
    for (int g = 0; g < 2; ++g) {
      mbar_init(&s_full[g], 1); mbar_init(&s_empty[g], 4); mbar_init(&p_ready[g], 4);
      mbar_init(&o_full[g], 1); mbar_init(&o_empty[g], 4);
    }
    fence_barrier_init();
  }
  for (uint32_t i = threadIdx.x; i < zrows * 4; i += blockDim.x) reinterpret_cast<uint32_t *>(sZ)[i] = 0u;
  fence_proxy_async();
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int my_seqs = (a.S - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int per_seq = 4 * RT;
  const int NIT = my_seqs * per_seq;

  if (warp == 0) {
    if (lane == 0) {
      for (int i = 0; i < NIT; ++i) {
        const int seq = blockIdx.x + (i / per_seq) * gridDim.x, w = i % per_seq, h = w / RT, rt = w % RT;
        if (rt == 0) {
          const int hi = i / RT, kvb = hi % KVBUFS;
          mbar_wait(&kv_empty[kvb], ((hi / KVBUFS) & 1) ^ 1);
          mbar_expect_tx(&kv_full[kvb], 2 * KVB);
          tma_bulk_g2s(sK + kvb * KVB, a.k_img + ((size_t)seq * 4 + h) * KVB, KVB, &kv_full[kvb]);
          tma_bulk_g2s(sV + kvb * KVB, a.v_img + ((size_t)seq * 4 + h) * KVB, KVB, &kv_full[kvb]);
        }
        const int qb = i & 3;
        mbar_wait(&q_empty[qb], ((i >> 2) & 1) ^ 1);
        mbar_expect_tx(&q_full[qb], 6144);
        tma_bulk_g2s(sQ + qb * 6144, a.q_img + (((size_t)seq * 4 + h) * RT + rt) * 6144, 6144, &q_full[qb]);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc_o = umma_idesc_bf16(128, 32, 0, 1);
      const uint32_t zaddr = smem_u32(sZ);
      if (SPLIT) {
        const int pkg[2] = {TCA_KSPLIT, Pk - TCA_KSPLIT};
        const uint32_t idesc_sg[2] = {umma_idesc_bf16(128, TCA_KSPLIT, 0, 0), umma_idesc_bf16(128, Pk - TCA_KSPLIT, 0, 0)};
        for (int j = 0; j <= NIT; ++j) {
          if (j < NIT) {
            const int i = j, rt = (i % per_seq) % RT, hi = i / RT, kvb = hi % KVBUFS, qb = i & 3;
            if (rt == 0) mbar_wait(&kv_full[kvb], (hi / KVBUFS) & 1);
            mbar_wait(&q_full[qb], (i >> 2) & 1);
            mbar_wait(&s_empty[0], (i & 1) ^ 1);
            mbar_wait(&s_empty[1], (i & 1) ^ 1);
            tc_fence_after();
            const uint32_t qa = smem_u32(sQ + qb * 6144);
#pragma unroll
            for (int g = 0; g < 2; ++g) {
              const uint32_t ka = smem_u32(sK + kvb * KVB) + g * TCA_KSPLIT * 16, ts = tmem + g * 256;
              umma_bf16(ts, umma_desc(qa, 2048, 128), umma_desc(ka, Pk * 16, 128), idesc_sg[g], 0u);
              umma_bf16(ts, umma_desc(qa + 2 * 2048, zaddr - (qa + 2 * 2048), 128),
                        umma_desc(ka + 2 * Pk * 16, zaddr - (ka + 2 * Pk * 16), 128), idesc_sg[g], 1u);
              umma_commit(&s_full[g]);
            }
            umma_commit(&q_empty[qb]);
          }
          if (j >= 1) {
            const int i = j - 1, rt = (i % per_seq) % RT, hi = i / RT, kvb = hi % KVBUFS;
#pragma unroll
            for (int g = 0; g < 2; ++g) {
              mbar_wait(&p_ready[g], i & 1);
              mbar_wait(&o_empty[g], (i & 1) ^ 1);
              tc_fence_after();
              const uint32_t pa = smem_u32(sP + g * PB), va = smem_u32(sV + kvb * KVB) + g * TCA_KSPLIT * 16;
              const uint32_t to = tmem + g * 256 + 192;
              for (int kk = 0; kk < pkg[g] / 16; ++kk)
                umma_bf16(to, umma_desc(pa + kk * 2 * 2048, 2048, 128), umma_desc(va + kk * 256, 128, Pk * 16), idesc_o,
                          kk != 0 ? 1u : 0u);
              umma_commit(&o_full[g]);
            }
            if (rt == RT - 1) umma_commit(&kv_empty[kvb]);
          }
        }
      } else {
      const uint32_t idesc_s = umma_idesc_bf16(128, Pk, 0, 0);
      for (int j = 0; j <= NIT; ++j) {
        if (j < NIT) {
          const int i = j, g = i & 1, u = i >> 1, rt = (i % per_seq) % RT, hi = i / RT, kvb = hi % TCA_KVBUF, qb = i & 3;
          if (rt == 0) mbar_wait(&kv_full[kvb], (hi / TCA_KVBUF) & 1);
          mbar_wait(&q_full[qb], (i >> 2) & 1);
          mbar_wait(&s_empty[g], (u & 1) ^ 1);
          tc_fence_after();
          const uint32_t qa = smem_u32(sQ + qb * 6144), ka = smem_u32(sK + kvb * KVB), ts = tmem + g * 256;
          // k-step 0: head dims 0..15 (chunks 0,1); k-step 1: dims 16..23 + the shared zero chunk
          umma_bf16(ts, umma_desc(qa, 2048, 128), umma_desc(ka, Pk * 16, 128), idesc_s, 0u);
          umma_bf16(ts, umma_desc(qa + 2 * 2048, zaddr - (qa + 2 * 2048), 128),
                    umma_desc(ka + 2 * Pk * 16, zaddr - (ka + 2 * Pk * 16), 128), idesc_s, 1u);
          umma_commit(&s_full[g]);
          umma_commit(&q_empty[qb]);
        }
        if (j >= 1) {
          const int i = j - 1, g = i & 1, u = i >> 1, rt = (i % per_seq) % RT, hi = i / RT, kvb = hi % TCA_KVBUF;
          mbar_wait(&p_ready[g], u & 1);
          mbar_wait(&o_empty[g], (u & 1) ^ 1);
          tc_fence_after();
          const uint32_t pa = smem_u32(sP + g * PB), va = smem_u32(sV + kvb * KVB), to = tmem + g * 256 + 192;
          for (int kk = 0; kk < Pk / 16; ++kk)
            umma_bf16(to, umma_desc(pa + kk * 2 * 2048, 2048, 128), umma_desc(va + kk * 256, 128, Pk * 16), idesc_o,
                      kk != 0 ? 1u : 0u);
          umma_commit(&o_full[g]);
          if (rt == RT - 1) umma_commit(&kv_empty[kvb]);
        }
      }
      }
    }
  } else {
    const int q = warp & 3, g = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    const uint32_t TM_S = tmem + g * 256, TM_O = tmem + g * 256 + 192;
    uint8_t *myP = sP + g * PB;
    // columns this group exponentiates: all Pk (alternating iterations) or its key block (SPLIT, every iteration)
    const int Pl = SPLIT ? (g == 0 ? TCA_KSPLIT : P - TCA_KSPLIT) : P;
    const int Pkl = SPLIT ? (g == 0 ? TCA_KSPLIT : Pk - TCA_KSPLIT) : Pk;
    const uint32_t thr2 = DROP ? drop_thr_bf16x2(a.thr16) : 0u;
    const uint32_t salt_lo = (uint32_t)a.key ^ ((uint32_t)(a.key >> 32) * 0x9E3779B9u);
    const uint32_t cadd = (salt_lo * 0x85EBCA6Bu) | 1u;
    const uint32_t *kmax = reinterpret_cast<const uint32_t *>(a.bound);
    const float *qnorm = a.bound != nullptr ? a.bound + (size_t)a.S * 4 : nullptr;
    // operand norms of iteration `it` (loaded one iteration ahead: the global-memory latency stays off the critical path)
    auto load_bound = [&](int it, float &qn, float &km) {
      qn = 0.f; km = 0.f;
      if (qnorm == nullptr || it >= NIT) return;
      const int seq = blockIdx.x + (it / per_seq) * gridDim.x, w = it % per_seq, h = w / RT, rt = w % RT;
      const int lrow = row - q_tail_offset(P, rt, h);
      if (lrow >= 0 && lrow < min(128, P - rt * 128)) qn = __ldg(qnorm + ((size_t)seq * 4 + h) * P + rt * 128 + lrow);
      km = __uint_as_float(__ldg(kmax + (size_t)seq * 4 + h));
    };
    float qn_next, km_next;
    load_bound(SPLIT ? 0 : g, qn_next, km_next);
    for (int i = SPLIT ? 0 : g; i < NIT; i += SPLIT ? 1 : 2) {
      const int u = SPLIT ? i : i >> 1;
      const int seq = blockIdx.x + (i / per_seq) * gridDim.x, w = i % per_seq, h = w / RT, rt = w % RT;
      const int rows_valid = min(128, P - rt * 128);
      const int roff = q_tail_offset(P, rt, h);
      const int lrow = row - roff;                       // query index inside the row tile
      const bool warp_active = q * 32 + 32 > roff && q * 32 < roff + rows_valid;
      const bool row_valid = lrow >= 0 && lrow < rows_valid;
      const float qn = qn_next, km = km_next;
      load_bound(i + (SPLIT ? 1 : 2), qn_next, km_next);
      // Upper bound of the row maximum without reading the scores (Cauchy-Schwarz on the bf16 operands, written by the
      // QKV epilogue): s_ij <= |q_i| max_j |k_j|.  Softmax is shift invariant, so any m >= max works as long as
      // 2^(s - m) stays representable: with m_b <= 40 every s - m_b lies in [-80, 0].  Rows with a larger bound (never
      // seen with LayerNorm'd inputs, but weights are data) take the exact two-pass route, warp-uniformly.
      float mb = 0.f;
      bool bounded = false;
      if (qnorm != nullptr && warp_active) {
        mb = fmaf(qn * km, 1.01f, 1e-3f);
        bounded = !__any_sync(0xffffffffu, !(mb <= 40.f));
      }
      mbar_wait(&s_full[g], u & 1);
      tc_fence_after();
      // V rows of the padded keys must be finite zeros (P is 0 there, but 0 * NaN = NaN)
      if (rt == 0 && q == 2 && (!SPLIT || g == 1)) {
        const int npad = Pk - P, kvb = (i / RT) % KVBUFS;
        for (int jz = lane; jz < npad * 3; jz += 32) {
          const int gg = jz / npad, rr = P + jz % npad;
          *reinterpret_cast<uint4 *>(sV + kvb * KVB + ((size_t)gg * Pk + rr) * 16) = make_uint4(0, 0, 0, 0);
        }
      }
      float m = -INFINITY, l = 0.f;
      if (warp_active) {
        // Full 32-column blocks run unpredicated; only the tail block (columns [c_tail, P), then zero fill up to Pk)
        // carries per-element predicates.
        const int c_tail = (Pl / 32) * 32;
        const bool tail32 = c_tail + 32 <= Pkl;          // else the tail is one 16-column load (Pk is a multiple of 16)
        if (bounded) {
          m = mb;
        } else {
          // ---- pass 1 (exact route only): row maximum ----
          float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
          for (int c0 = 0; c0 < c_tail; c0 += 32) {
            float t[32];
            tmem_ld32(TM_S + lane_base + c0, t);
#pragma unroll
            for (int c = 0; c < 32; c += 4) {
              m0 = fmaxf(m0, t[c]); m1 = fmaxf(m1, t[c + 1]); m2 = fmaxf(m2, t[c + 2]); m3 = fmaxf(m3, t[c + 3]);
            }
          }
          if (c_tail < Pl) {
            float t[32];
            if (tail32) {
              tmem_ld32(TM_S + lane_base + c_tail, t);
            } else {
              float t16[16];
              tmem_ld16(TM_S + lane_base + c_tail, t16);
#pragma unroll
              for (int c = 0; c < 16; ++c) t[c] = t16[c];
#pragma unroll
              for (int c = 16; c < 32; ++c) t[c] = -INFINITY;
            }
#pragma unroll
            for (int c = 0; c < 32; ++c) if (c_tail + c < Pl) m0 = fmaxf(m0, t[c]);
          }
          m = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
        }
        // ---- p = 2^(s - m), row sum, (dropout), bf16 image: one pass over the scores ----
        const float negm = -m;
        const uint64_t rowid = ((uint64_t)seq * 4 + h) * P + (uint64_t)(rt * 128 + lrow);
        const uint32_t salt = salt_lo ^ ((uint32_t)(rowid >> 28) * 0x85EBCA6Bu);
        const uint32_t ctr = (uint32_t)rowid * 16u + (SPLIT ? (uint32_t)g * 6u : 0u);   // + 32-column block index
        uint4 *prow = reinterpret_cast<uint4 *>(myP) + row;
        float l0 = 0.f, l1 = 0.f, l2 = 0.f, l3 = 0.f;
        if (PF > 0) {
          // compile-time sequence length (168 / 336): five full blocks per group, the load of block k+1 in flight
          // while block k is exponentiated (two register buffers)
          constexpr int NBLK = 5;
          float ta[32], tb[32];
          tmem_ld32_issue(TM_S + lane_base, ta);
#pragma unroll
          for (int k = 0; k < NBLK; ++k) {
            if ((k & 1) == 0) {
              tmem_wait_ld32(ta);
              if (k + 1 < NBLK) tmem_ld32_issue(TM_S + lane_base + (k + 1) * 32, tb);
              softmax_cols<32, DROP, false>(ta, negm, 32, 4, l0, l1, l2, l3, DROP ? hash32((ctr + k) ^ salt) : 0u, cadd, thr2,
                                            prow + (size_t)(k * 4) * 128);
            } else {
              tmem_wait_ld32(tb);
              if (k + 1 < NBLK) tmem_ld32_issue(TM_S + lane_base + (k + 1) * 32, ta);
              softmax_cols<32, DROP, false>(tb, negm, 32, 4, l0, l1, l2, l3, DROP ? hash32((ctr + k) ^ salt) : 0u, cadd, thr2,
                                            prow + (size_t)(k * 4) * 128);
            }
          }
          if (NBLK * 32 < Pkl) {                          // 16-column tail: PF = 168 (8 valid), group 0 of PF = 336 (16 valid)
            float t16[16];
            tmem_ld16_issue(TM_S + lane_base + NBLK * 32, t16);
            tmem_wait_ld16(t16);
            softmax_cols<16, DROP, true>(t16, negm, Pl - NBLK * 32, (Pkl - NBLK * 32) / 8, l0, l1, l2, l3,
                                         DROP ? hash32((ctr + NBLK) ^ salt) : 0u, cadd, thr2, prow + (size_t)(NBLK * 4) * 128);
          }
        } else {
          for (int c0 = 0; c0 < c_tail; c0 += 32) {
            float t[32];
            tmem_ld32_issue(TM_S + lane_base + c0, t);
            tmem_wait_ld32(t);
            softmax_cols<32, DROP, false>(t, negm, 32, 4, l0, l1, l2, l3, DROP ? hash32((ctr + (c0 >> 5)) ^ salt) : 0u, cadd, thr2,
                                          prow + (size_t)(c0 >> 3) * 128);
          }
          if (c_tail < Pkl) {
            const uint32_t st = DROP ? hash32((ctr + (c_tail >> 5)) ^ salt) : 0u;
            if (tail32) {
              float t[32];
              tmem_ld32_issue(TM_S + lane_base + c_tail, t);
              tmem_wait_ld32(t);
              softmax_cols<32, DROP, true>(t, negm, Pl - c_tail, (Pkl - c_tail) / 8, l0, l1, l2, l3, st, cadd, thr2,
                                           prow + (size_t)(c_tail >> 3) * 128);
            } else {
              float t16[16];
              tmem_ld16_issue(TM_S + lane_base + c_tail, t16);
              tmem_wait_ld16(t16);
              softmax_cols<16, DROP, true>(t16, negm, Pl - c_tail, (Pkl - c_tail) / 8, l0, l1, l2, l3, st, cadd, thr2,
                                           prow + (size_t)(c_tail >> 3) * 128);
            }
          }
        }
        l = (l0 + l1) + (l2 + l3);
      }
      tc_fence_before();
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) { mbar_arrive(&s_empty[g]); mbar_arrive(&p_ready[g]); }
      // epilogue: O / l  -> O tile image (token-tile format of the following out-projection GEMM)
      mbar_wait(&o_full[g], u & 1);
      tc_fence_after();
      float o[32];
      if (warp_active) tmem_ld32(TM_O + lane_base, o);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&o_empty[g]);
      float f0 = 1.f;
      if (SPLIT) {
        // merge the two key blocks: group 1 publishes (m, l, O[24]); group 0 combines and writes the tile
        float *x = xch + ((size_t)(i & 1) * 128 + row) * TCA_XROW;
        if (g == 1 && warp_active) {
          x[0] = m; x[1] = l;
#pragma unroll
          for (int c = 0; c < HD; ++c) x[2 + c] = o[c];
        }
        asm volatile("bar.sync 2, 256;" ::: "memory");
        if (g == 0 && row_valid) {
          const float m1 = x[0], l1 = x[1], mm = fmaxf(m, m1);
          f0 = fast_exp2(m - mm);
          const float f1 = fast_exp2(m1 - mm);
          l = l * f0 + l1 * f1;
#pragma unroll
          for (int c = 0; c < HD; ++c) o[c] = o[c] * f0 + x[2 + c] * f1;
        }
      }
      if (row_valid && (!SPLIT || g == 0)) {
        const float inv = a.dscale / l;
        const long long token = (long long)seq * P + rt * 128 + lrow;
        const long long mt = token >> 7;
        const int r = (int)(token & 127);
        uint4 *dst = reinterpret_cast<uint4 *>(a.o_img) + ((size_t)mt * 12 + 3 * h) * 128 + r;
#pragma unroll
        for (int cc = 0; cc < 3; ++cc) {
          float x8[8];
#pragma unroll
          for (int jx = 0; jx < 8; ++jx) x8[jx] = o[cc * 8 + jx] * inv;
          dst[cc * 128] = pack8_bf16(x8);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// ===========================================================================
// Gram matrix of the hidden states on tcgen05: G[b] = X[b] X[b]^T, X[b] = [N nodes, K = P*96] read from the
// sequence-major bf16 image [B][K/8][R][8] the encoder's last epilogue emits.  One CTA per
// (sample, 128-row tile, 256-column block); the K dimension streams through a 4-stage TMA ring, both MMA
// operands are row ranges of the same image.  fp32 accumulation in TMEM over the whole K = 16128.
// ===========================================================================
constexpr int TG_KC = 8;          // chunks (64 K elements) per pipeline stage
constexpr int TG_STAGES = 4;

struct TcGramArgs {
  const uint8_t *img;
  float *gram;              // [B][N][N] raw dot products
  int N, R, KC;             // nodes, padded rows per chunk, chunks per sample (multiple of TG_KC)
  int tile_first, tile_step; // row tiles handled by this launch: tile_first + i * tile_step (a rank's share when sharded)
};

__global__ void __launch_bounds__(192, 1) tc_gram_kernel(TcGramArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int b = blockIdx.z, mt = a.tile_first + blockIdx.y * a.tile_step, nblk = blockIdx.x;
  const int col0 = nblk * 256;
  const int Rb = min(256, a.R - col0);                         // B rows staged per chunk
  const int Ncols = min(256, ((a.N - col0) + 15) / 16 * 16);   // MMA N
  const uint32_t a_stage = TG_KC * 2048, b_stage = (uint32_t)TG_KC * Rb * 16;
  uint8_t *sA = smem;
  uint8_t *sB = smem + TG_STAGES * a_stage;
  uint64_t *bars = reinterpret_cast<uint64_t *>(sB + TG_STAGES * b_stage);
  uint64_t *full = bars, *empty = bars + TG_STAGES, *done = bars + 2 * TG_STAGES;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(done + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < TG_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(done, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int nslices = a.KC / TG_KC;
  const uint8_t *base = a.img + (size_t)b * a.KC * a.R * 16;

  if (warp == 0) {
    if (lane == 0) {
      for (int i = 0; i < nslices; ++i) {
        const int s = i % TG_STAGES, ph = (i / TG_STAGES) & 1;
        mbar_wait(&empty[s], ph ^ 1);
        mbar_expect_tx(&full[s], a_stage + b_stage);
        for (int c = 0; c < TG_KC; ++c) {
          const uint8_t *chunk = base + ((size_t)(i * TG_KC + c) * a.R) * 16;
          tma_bulk_g2s(sA + s * a_stage + c * 2048, chunk + (size_t)mt * 128 * 16, 2048, &full[s]);
          tma_bulk_g2s(sB + s * b_stage + (size_t)c * Rb * 16, chunk + (size_t)col0 * 16, (uint32_t)Rb * 16, &full[s]);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_bf16(128, Ncols, 0, 0);
      for (int i = 0; i < nslices; ++i) {
        const int s = i % TG_STAGES, ph = (i / TG_STAGES) & 1;
        mbar_wait(&full[s], ph);
        tc_fence_after();
        const uint32_t aa = smem_u32(sA + s * a_stage), ba = smem_u32(sB + s * b_stage);
#pragma unroll
        for (int kk = 0; kk < TG_KC / 2; ++kk)
          umma_bf16(tmem, umma_desc(aa + kk * 2 * 2048, 2048, 128), umma_desc(ba + kk * 2 * Rb * 16, Rb * 16, 128), idesc,
                    (i | kk) != 0 ? 1u : 0u);
        umma_commit(&empty[s]);
      }
      umma_commit(done);
    }
  } else {
    const int q = warp & 3, row = mt * 128 + q * 32 + lane;
    mbar_wait(done, 0);
    tc_fence_after();
    float *out = a.gram + ((size_t)b * a.N + row) * a.N + col0;
    for (int c0 = 0; c0 < Ncols; c0 += 32) {
      float t[32];
      if (c0 + 32 <= Ncols) {
        tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + c0, t);
      } else {
        float t16[16];
        tmem_ld16(tmem + ((uint32_t)(q * 32) << 16) + c0, t16);
#pragma unroll
        for (int c = 0; c < 16; ++c) t[c] = t16[c];
      }
      if (row < a.N) {
#pragma unroll
        for (int c = 0; c < 32; ++c)
          if (c0 + c < Ncols && col0 + c0 + c < a.N) out[c0 + c] = t[c];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 256);
}

// sim = G / ((sqrt(G_ii) + 1e-7)(sqrt(G_jj) + 1e-7))   (similarity.py:8-14; the norms are the Gram diagonal)
__global__ void gram_normalize_kernel(const float *__restrict__ g, int N, float *__restrict__ sim) {
  const int b = blockIdx.y;
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (long long)N * N) return;
  const int i = (int)(e / N), j = (int)(e - (long long)i * N);
  const float *gb = g + (size_t)b * N * N;
  const float ni = sqrtf(fmaxf(gb[(size_t)i * N + i], 0.f)) + 1e-7f, nj = sqrtf(fmaxf(gb[(size_t)j * N + j], 0.f)) + 1e-7f;
  sim[(size_t)b * N * N + e] = gb[e] / (ni * nj);
}

// ===========================================================================
// Fused token block of one encoder layer (everything between two attentions is row-local):
//   Y  = LN1(X + drop(O Wo^T + bo))                         (out-projection, nn.TransformerEncoderLayer norm1)
//   H  = drop(relu(Y W1^T + b1)),  X' = LN2(Y + drop(H W2^T + b2))      (feed-forward, norm2)
//   Q,K,V of the NEXT layer = X' Wqkv'^T + b'  (written straight into the attention operand images), or, for the last
//   layer, encoder_norm(X') as fp32 hidden states + the Gram operand image.
// One CTA owns a tile of 128 tokens at a time; Y, H (one 96-column slab at a time) and X' never leave shared memory, so a
// layer moves O + X in and X' + QKV out (1.3 GB at METR-LA) instead of the 3.9 GB of the four separate token GEMMs.
// All weights are streamed from L2 as twelve 18 KB K-major slices [12 chunks][96 rows][8] in program order
// (Wo | W1_0 W2_0 ... W1_3 W2_3 | Wq Wk Wv) through a 3-slot TMA ring; accumulators: two 96-column TMEM slots.
// Warp roles: 0 TMA producer, 1 MMA issuer (+ TMEM alloc), 2-5 epilogue (thread = token row).  The per-tile dependency
// chain MMA -> epilogue -> MMA is serial inside a CTA; two CTAs are co-resident per SM (110 KB smem, 256 TMEM columns
// each) and fill each other's bubbles.
// ===========================================================================
constexpr int TLK_THREADS = 192;
constexpr uint32_t TLK_SLICE = 12 * 96 * 16;           // 18432 B: one [96 x 96] weight slice
constexpr int TLK_RING = 3;

struct TcLayerArgs {
  const uint8_t *O, *X;            // attention output / layer input (residual) tile images [MT][12][128][8]
  const uint8_t *W;                // 12 (9 for the last layer) slices in program order
  const float *bo, *b1, *b2, *bqkv;
  const float *ln1w, *ln1b, *ln2w, *ln2b, *fnw, *fnb;
  uint8_t *Xout;                   // next layer's input image (nullptr for the last layer)
  uint8_t *q_img, *k_img, *v_img;  // next layer's attention operands
  float *bound;                    // next layer's row-maximum bound workspace (max |k| slots zeroed by the host); may be null
  long long nseq;
  float *hidden;                   // last layer: fp32 [T][96]
  uint8_t *seq_img;                // last layer: Gram operand image (may be null)
  int seq_nodes, seq_rows;
  int MT, P, Pk, RT, last;
  long long T;
  float qscale;
  uint32_t thr16; float dscale; uint64_t key_o, key_h, key_f;
};

__global__ void __launch_bounds__(TLK_THREADS, 2) tc_layer_kernel(TcLayerArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t *sRing = smem;                                   // TLK_RING x 18432
  uint8_t *sOH = sRing + TLK_RING * TLK_SLICE;             // O tile, later the H slab (same 24 KB)
  uint8_t *sY = sOH + SLICE_BYTES;                         // Y, later X'
  float *sPar = reinterpret_cast<float *>(sY + SLICE_BYTES);   // bo[96] b1[384] b2[96] bqkv[288] ln1w ln1b ln2w ln2b fnw fnb
  uint64_t *bars = reinterpret_cast<uint64_t *>(sPar + 96 + 384 + 96 + 288 + 6 * 96);
  uint64_t *ring_full = bars, *ring_empty = bars + 3, *o_full = bars + 6, *oh_free = bars + 7, *acc_full = bars + 8,
           *acc_empty = bars + 10, *y_ready = bars + 12, *h_ready = bars + 13, *h_free = bars + 14, *x_ready = bars + 15;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 16);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float *sBo = sPar, *sB1 = sPar + 96, *sB2 = sB1 + 384, *sBq = sB2 + 96, *sLn = sBq + 288;
  for (int i = threadIdx.x; i < 96; i += blockDim.x) {
    sBo[i] = a.bo[i]; sB2[i] = a.b2[i];
    sLn[i] = a.ln1w[i]; sLn[96 + i] = a.ln1b[i]; sLn[192 + i] = a.ln2w[i]; sLn[288 + i] = a.ln2b[i];
    sLn[384 + i] = a.fnw ? a.fnw[i] : 1.f; sLn[480 + i] = a.fnb ? a.fnb[i] : 0.f;
  }
  for (int i = threadIdx.x; i < 384; i += blockDim.x) sB1[i] = a.b1[i];
  if (!a.last)
    for (int i = threadIdx.x; i < 288; i += blockDim.x) sBq[i] = a.bqkv[i];
  if (threadIdx.x == 0) {
    for (int i = 0; i < TLK_RING; ++i) { mbar_init(&ring_full[i], 1); mbar_init(&ring_empty[i], 1); }
    mbar_init(o_full, 1); mbar_init(oh_free, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 4); }
    mbar_init(y_ready, 4); mbar_init(h_ready, 4); mbar_init(h_free, 1); mbar_init(x_ready, 4);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int NS = a.last ? 9 : 12;                          // weight slices per tile

  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      uint32_t n = 0, it = 0;
      for (int mt = blockIdx.x; mt < a.MT; mt += gridDim.x, ++it) {
        mbar_wait(oh_free, (it & 1) ^ 1);                  // the previous tile's last FFN2 has read the H slab
        mbar_expect_tx(o_full, SLICE_BYTES);
        tma_bulk_g2s(sOH, a.O + (size_t)mt * SLICE_BYTES, SLICE_BYTES, o_full);
        for (int s = 0; s < NS; ++s, ++n) {
          const uint32_t slot = n % TLK_RING;
          mbar_wait(&ring_empty[slot], ((n / TLK_RING) & 1) ^ 1);
          mbar_expect_tx(&ring_full[slot], TLK_SLICE);
          tma_bulk_g2s(sRing + slot * TLK_SLICE, a.W + (size_t)s * TLK_SLICE, TLK_SLICE, &ring_full[slot]);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ MMA issuer (one thread) ------------------------------
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_bf16(128, 96, 0, 0);
      const uint32_t oh = smem_u32(sOH), yy = smem_u32(sY), ring = smem_u32(sRing);
      uint32_t n = 0, it = 0, u0 = 0, u1 = 0, hcnt = 0;   // ring slices, tiles, uses of acc slot 0 / 1, H slabs
      // one [128 x 96] x [96 x 96]^T product: 6 k-steps of 16
      auto gemm96 = [&](uint32_t a_addr, uint32_t acc_col, bool accumulate) {
        const uint32_t slot = n % TLK_RING;
        mbar_wait(&ring_full[slot], (n / TLK_RING) & 1);
        tc_fence_after();
        const uint32_t w = ring + slot * TLK_SLICE;
#pragma unroll
        for (int kk = 0; kk < 6; ++kk)
          umma_bf16(tmem + acc_col, umma_desc(a_addr + kk * 2 * 2048, 2048, 128), umma_desc(w + kk * 2 * 1536, 1536, 128), idesc,
                    (accumulate || kk != 0) ? 1u : 0u);
        umma_commit(&ring_empty[slot]);
        ++n;
      };
      for (int mt = blockIdx.x; mt < a.MT; mt += gridDim.x, ++it) {
        // out-projection -> acc 0
        mbar_wait(o_full, it & 1);
        mbar_wait(&acc_empty[0], (u0 & 1) ^ 1);
        tc_fence_after();
        gemm96(oh, 0, false);
        umma_commit(&acc_full[0]); ++u0;
        // feed-forward: FFN1 slab j -> acc 1, FFN2 K-slab j accumulates into acc 0
        mbar_wait(y_ready, it & 1);
        tc_fence_after();
        for (int j = 0; j < 4; ++j, ++hcnt) {
          mbar_wait(&acc_empty[1], (u1 & 1) ^ 1);
          tc_fence_after();
          gemm96(yy, 128, false);
          umma_commit(&acc_full[1]); ++u1;
          mbar_wait(h_ready, hcnt & 1);
          if (j == 0) mbar_wait(&acc_empty[0], (u0 & 1) ^ 1);
          tc_fence_after();
          gemm96(oh, 0, j != 0);
          umma_commit(h_free);
        }
        umma_commit(&acc_full[0]); ++u0;
        umma_commit(oh_free);
        // QKV of the next layer from X' (in the Y buffer): Q -> acc 1, K -> acc 0, V -> acc 1
        if (!a.last) {
          mbar_wait(x_ready, it & 1);
          tc_fence_after();
          for (int q = 0; q < 3; ++q) {
            const int s = (q == 1) ? 0 : 1;
            uint32_t &u = s ? u1 : u0;
            mbar_wait(&acc_empty[s], (u & 1) ^ 1);
            tc_fence_after();
            gemm96(yy, s * 128, false);
            umma_commit(&acc_full[s]); ++u;
          }
        }
      }
    }
  } else {
    // ------------------------------ epilogue warps: thread = token row ------------------------------
    const int q = warp & 3, row = q * 32 + lane;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    uint32_t it = 0, u0 = 0, u1 = 0, hcnt = 0;
    auto load_acc = [&](int s, uint32_t &u, float (&v)[96]) {
      mbar_wait(&acc_full[s], u & 1);
      ++u;
      tc_fence_after();
      const uint32_t taddr = tmem + lane_base + s * 128;
      float t0[32];
      tmem_ld32(taddr, t0);
#pragma unroll
      for (int c = 0; c < 32; ++c) v[c] = t0[c];
      tmem_ld32(taddr + 32, t0);
#pragma unroll
      for (int c = 0; c < 32; ++c) v[32 + c] = t0[c];
      tmem_ld32(taddr + 64, t0);
#pragma unroll
      for (int c = 0; c < 32; ++c) v[64 + c] = t0[c];
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[s]);
    };
    for (int mt = blockIdx.x; mt < a.MT; mt += gridDim.x, ++it) {
      const long long token = (long long)mt * 128 + row;
      const bool valid = token < a.T;
      float v[96];
      // ---- E1: Y = LN1(X + drop(acc + bo)) -> sY ----
      load_acc(0, u0, v);
      {
        const uint4 *res = reinterpret_cast<const uint4 *>(a.X) + ((size_t)mt * 12) * 128 + row;
#pragma unroll
        for (int cc = 0; cc < 12; ++cc) {
#pragma unroll
          for (int j = 0; j < 8; ++j) v[cc * 8 + j] += sBo[cc * 8 + j];
          if (a.thr16) drop8(&v[cc * 8], (uint64_t)token * 12 + cc, a.thr16, a.dscale, a.key_o);
          float r8[8];
          unpack8_bf16(res[cc * 128], r8);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[cc * 8 + j] += r8[j];
        }
        layer_norm96(v, sLn, sLn + 96);
        uint4 *o = reinterpret_cast<uint4 *>(sY) + row;
#pragma unroll
        for (int cc = 0; cc < 12; ++cc) o[cc * 128] = pack8_bf16(&v[cc * 8]);
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(y_ready);
      }
      // ---- E2: H slab j = drop(relu(acc + b1[96j..])) -> sOH ----
      for (int j = 0; j < 4; ++j, ++hcnt) {
        load_acc(1, u1, v);
        mbar_wait(h_free, (hcnt & 1) ^ 1);                  // FFN2 of the previous slab has consumed the buffer
        uint4 *o = reinterpret_cast<uint4 *>(sOH) + row;
#pragma unroll
        for (int cc = 0; cc < 12; ++cc) {
          float x[8];
#pragma unroll
          for (int jx = 0; jx < 8; ++jx) x[jx] = fmaxf(v[cc * 8 + jx] + sB1[j * 96 + cc * 8 + jx], 0.f);
          if (a.thr16) drop8(x, ((uint64_t)token * 384 + j * 96) / 8 + cc, a.thr16, a.dscale, a.key_h);
          o[cc * 128] = pack8_bf16(x);
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(h_ready);
      }
      // ---- E3: X' = LN2(Y + drop(acc + b2)) ----
      load_acc(0, u0, v);
      {
        const uint4 *yres = reinterpret_cast<const uint4 *>(sY) + row;
#pragma unroll
        for (int cc = 0; cc < 12; ++cc) {
#pragma unroll
          for (int j = 0; j < 8; ++j) v[cc * 8 + j] += sB2[cc * 8 + j];
          if (a.thr16) drop8(&v[cc * 8], (uint64_t)token * 12 + cc, a.thr16, a.dscale, a.key_f);
          float r8[8];
          unpack8_bf16(yres[cc * 128], r8);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[cc * 8 + j] += r8[j];
        }
        layer_norm96(v, sLn + 192, sLn + 288);
        if (a.last) {
          if (a.fnw != nullptr) layer_norm96(v, sLn + 384, sLn + 480);
          if (valid) {
            float *o = a.hidden + token * 96;
#pragma unroll
            for (int c = 0; c < 96; c += 4) *reinterpret_cast<float4 *>(o + c) = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
            if (a.seq_img != nullptr) {
              const long long sq = token / a.P;
              const int pp = (int)(token - sq * a.P);
              const long long bb = sq / a.seq_nodes;
              const int nn = (int)(sq - bb * a.seq_nodes);
              uint4 *o2 = reinterpret_cast<uint4 *>(a.seq_img) + ((size_t)bb * a.P * 12 + (size_t)pp * 12) * a.seq_rows + nn;
#pragma unroll
              for (int cc = 0; cc < 12; ++cc) o2[(size_t)cc * a.seq_rows] = pack8_bf16(&v[cc * 8]);
            }
          }
        } else {
          uint4 *o = reinterpret_cast<uint4 *>(sY) + row;
          uint4 *og = reinterpret_cast<uint4 *>(a.Xout) + ((size_t)mt * 12) * 128 + row;
#pragma unroll
          for (int cc = 0; cc < 12; ++cc) {
            const uint4 pk = pack8_bf16(&v[cc * 8]);
            o[cc * 128] = pk;
            og[cc * 128] = pk;
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(x_ready);
        }
      }
      // ---- E4: Q, K, V of the next layer ----
      if (!a.last) {
        const long long s = valid ? token / a.P : 0;
        const int p = valid ? (int)(token - s * a.P) : 0;
        for (int qq = 0; qq < 3; ++qq) {
          if (qq == 1) load_acc(0, u0, v);
          else load_acc(1, u1, v);
#pragma unroll
          for (int c = 0; c < 96; ++c) v[c] += sBq[qq * 96 + c];
          if (!valid) continue;
          if (qq == 0) {
            const int rt = p >> 7;
#pragma unroll
            for (int h = 0; h < 4; ++h) {
              const int r = (p & 127) + q_tail_offset(a.P, rt, h);
              uint4 *o = reinterpret_cast<uint4 *>(a.q_img) + (((size_t)s * 4 + h) * a.RT + rt) * 3 * 128 + r;
              float n2 = 0.f;
#pragma unroll
              for (int cc = 0; cc < 3; ++cc) {
                float x[8];
#pragma unroll
                for (int jx = 0; jx < 8; ++jx) { x[jx] = v[h * HD + cc * 8 + jx] * a.qscale; n2 = fmaf(x[jx], x[jx], n2); }
                o[cc * 128] = pack8_bf16(x);
              }
              if (a.bound != nullptr) a.bound[(size_t)a.nseq * 4 + ((size_t)s * 4 + h) * a.P + p] = sqrtf(n2);
            }
          } else {
            uint8_t *base = (qq == 1) ? a.k_img : a.v_img;
#pragma unroll
            for (int h = 0; h < 4; ++h) {
              uint4 *o = reinterpret_cast<uint4 *>(base) + ((size_t)s * 4 + h) * 3 * a.Pk + p;
#pragma unroll
              for (int cc = 0; cc < 3; ++cc) o[(size_t)cc * a.Pk] = pack8_bf16(&v[h * HD + cc * 8]);
              if (qq == 1 && a.bound != nullptr) {      // max_j |k_j| of the next layer (see the TCM_QKV epilogue)
                float n2 = 0.f;
#pragma unroll
                for (int c = 0; c < HD; ++c) n2 = fmaf(v[h * HD + c], v[h * HD + c], n2);
                atomicMax(reinterpret_cast<uint32_t *>(a.bound) + s * 4 + h, __float_as_uint(sqrtf(n2)));
              }
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 256);
}

// ===========================================================================
// Fused feed-forward block of one encoder layer (transformer_layers.py:10-11 -> nn.TransformerEncoderLayer:
// linear1 -> ReLU -> dropout -> linear2 -> dropout2 -> + residual -> norm2 [-> encoder_norm]) per 128-token tile:
//   H  = drop(relu(X1 W1^T + b1))         four [128 x 96] accumulators in TMEM slots 0..3, K = 96
//   Y  = H W2^T                           one  [128 x 96] accumulator in slot 4, K = 4 x 96: the bf16 H slice of
//                                         sub-tile nb goes through ONE 24 KB shared-memory buffer, never to HBM
//   X2 = LN2(X1 + drop(Y + b2))           residual read from the X1 tile that is still in shared memory
// Both weight images stay resident (2 x 72 KB); persistent CTA, one per SM.  Same MMAs in the same K order, same
// dropout counters and the same epilogue arithmetic as tc_linear_kernel<TCM_RELU_IMG> followed by
// tc_linear_kernel<TCM_RESLN>: results are bit-identical, the 768 B/token H round trip through HBM is gone.
// Warp roles: warp 0 TMA producer (X1 tiles, 2 stages), warp 1 MMA issuer, warps 2-5 / 6-9 two H groups (group g takes
// sub-tiles g and g + 2 of every tile and hands its bf16 slice to the MMA issuer), warps 10-13 the residual + LayerNorm
// epilogue of every tile - the H pipeline never waits for a LayerNorm.
// ===========================================================================
struct TcFfnArgs {
  const uint8_t *A;              // X1 tile image [MT][12][128][8]
  const uint8_t *W1, *W2;        // lin1 image [12][384][8], lin2 image [48][96][8]
  const float *b1, *b2, *ln_w, *ln_b, *ln2_w, *ln2_b;
  int MT; long long T;
  uint8_t *out_img;              // X2 tile image (may be null when out_f32 is given)
  float *out_f32;                // last layer: fp32 [T][96] after the final LayerNorm
  uint8_t *seq_img; int seq_nodes, seq_rows, P;
  uint32_t thr16; float dscale; uint64_t key_h, key_f;
  volatile int *dbg;             // STEP_FFN_DEBUG builds only: host-mapped progress slots [grid][16]
};
constexpr uint32_t TFF_W_BYTES = 96 * 384 * 2;
constexpr int TFF_THREADS = 448;   // warp 0 TMA, warp 1 MMA, warps 2-5 / 6-9 the two H groups, warps 10-13 the LayerNorm epilogue

#ifdef STEP_FFN_DEBUG
// debug build: every wait site records (site, tile) in a host-mapped buffer slot per warp before blocking and clears it after
#define FFN_WAIT(bar, par, site)                                                                      \
  do {                                                                                                \
    if (a.dbg && (threadIdx.x & 31) == 0) { a.dbg[blockIdx.x * 16 + (threadIdx.x >> 5)] = (site); __threadfence_system(); } \
    mbar_wait(bar, par);                                                                              \
    if (a.dbg && (threadIdx.x & 31) == 0) { a.dbg[blockIdx.x * 16 + (threadIdx.x >> 5)] = 100 + (site); }  \
  } while (0)
#else
#define FFN_WAIT(bar, par, site) mbar_wait(bar, par)
#endif
template <bool FINAL>
__global__ void __launch_bounds__(TFF_THREADS, 1) tc_ffn_kernel(TcFfnArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t *sW1 = smem;
  uint8_t *sW2 = sW1 + TFF_W_BYTES;
  uint8_t *sA = sW2 + TFF_W_BYTES;                    // 2 stages
  uint8_t *sH = sA + 2 * SLICE_BYTES;
  uint64_t *bars = reinterpret_cast<uint64_t *>(sH + SLICE_BYTES);
  // h_ready / h_free exist once per H group: a group that alternates with the other one on a shared barrier could wait
  // for a phase two completions ahead, which a parity wait cannot tell from one already completed
  uint64_t *full = bars, *empty = bars + 2, *tfull1 = bars + 4, *tempty1 = bars + 8, *h_ready = bars + 12, *h_free = bars + 14;
  uint64_t *acc2_full = bars + 16, *acc2_empty = bars + 18, *wbar = bars + 19;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 20);
  float *sB1 = reinterpret_cast<float *>(bars + 22);   // b1[384], b2[96], ln_w, ln_b, ln2_w, ln2_b
  float *sB2 = sB1 + 384, *sLn = sB2 + 96;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < 384; i += blockDim.x) sB1[i] = a.b1[i];
  for (int i = threadIdx.x; i < 96; i += blockDim.x) {
    sB2[i] = a.b2[i];
    sLn[i] = a.ln_w[i]; sLn[96 + i] = a.ln_b[i];
    sLn[192 + i] = a.ln2_w ? a.ln2_w[i] : 1.f; sLn[288 + i] = a.ln2_b ? a.ln2_b[i] : 0.f;
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 4); }
    for (int i = 0; i < 4; ++i) { mbar_init(&tfull1[i], 1); mbar_init(&tempty1[i], 4); }
    for (int i = 0; i < 2; ++i) { mbar_init(&h_ready[i], 4); mbar_init(&h_free[i], 1); }
    mbar_init(acc2_full, 1);
    mbar_init(acc2_empty, 4); mbar_init(wbar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int ntiles = (a.MT - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(wbar, 2 * TFF_W_BYTES);
      tma_bulk_g2s(sW1, a.W1, TFF_W_BYTES, wbar);
      tma_bulk_g2s(sW2, a.W2, TFF_W_BYTES, wbar);
      for (int it = 0; it < ntiles; ++it) {
        const int mt = blockIdx.x + it * gridDim.x, s = it & 1;
        FFN_WAIT(&empty[s], ((it >> 1) & 1) ^ 1, 1);
        mbar_expect_tx(&full[s], SLICE_BYTES);
        tma_bulk_g2s(sA + s * SLICE_BYTES, a.A + (size_t)mt * SLICE_BYTES, SLICE_BYTES, &full[s]);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      FFN_WAIT(wbar, 0, 2);
      const uint32_t idesc = umma_idesc_bf16(128, 96, 0, 0);
      const uint32_t sA_addr = smem_u32(sA), sW1_addr = smem_u32(sW1), sW2_addr = smem_u32(sW2), sH_addr = smem_u32(sH);
      auto mma1 = [&](int it, int nb) {            // H sub-tile nb of tile it: [128 x 96] x W1 rows [96 nb, 96 nb + 96)
        const uint32_t abase = sA_addr + (it & 1) * SLICE_BYTES;
#pragma unroll
        for (int kk = 0; kk < 6; ++kk)
          umma_bf16(tmem + nb * 96, umma_desc(abase + kk * 2 * 2048, 2048, 128),
                    umma_desc(sW1_addr + (uint32_t)(kk * 2) * 6144 + nb * 96 * 16, 6144, 128), idesc, kk != 0 ? 1u : 0u);
        umma_commit(&tfull1[nb]);
      };
      if (ntiles > 0) {
        FFN_WAIT(&full[0], 0, 3);
        tc_fence_after();
        for (int nb = 0; nb < 4; ++nb) mma1(0, nb);
      }
      for (int it = 0; it < ntiles; ++it) {
        for (int nb = 0; nb < 4; ++nb) {
          const uint32_t k = (uint32_t)it * 2 + (nb >> 1);        // this is the k-th slice of epilogue group nb & 1
          if (nb == 0) FFN_WAIT(acc2_empty, (it & 1) ^ 1, 4);
          FFN_WAIT(&h_ready[nb & 1], k & 1, 5);
          tc_fence_after();
#pragma unroll
          for (int kk = 0; kk < 6; ++kk)
            umma_bf16(tmem + 384, umma_desc(sH_addr + kk * 2 * 2048, 2048, 128),
                      umma_desc(sW2_addr + (uint32_t)(nb * 12 + kk * 2) * 1536, 1536, 128), idesc, (nb | kk) != 0 ? 1u : 0u);
          umma_commit(&h_free[(nb & 1) ^ 1]);                      // the H buffer passes to the other group
          if (nb == 3) umma_commit(acc2_full);
          if (it + 1 < ntiles) {
            if (nb == 0) FFN_WAIT(&full[(it + 1) & 1], ((it + 1) >> 1) & 1, 6);
            FFN_WAIT(&tempty1[nb], ((it + 1) & 1) ^ 1, 7);
            tc_fence_after();
            mma1(it + 1, nb);
          }
        }
      }
    }
  } else {
    const int q = warp & 3, grp = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    auto load_acc = [&](uint32_t col, float *v) {
      float t0[32];
      tmem_ld32(tmem + lane_base + col, t0);
#pragma unroll
      for (int c = 0; c < 32; ++c) v[c] = t0[c];
      tmem_ld32(tmem + lane_base + col + 32, t0);
#pragma unroll
      for (int c = 0; c < 32; ++c) v[32 + c] = t0[c];
      tmem_ld32(tmem + lane_base + col + 64, t0);
#pragma unroll
      for (int c = 0; c < 32; ++c) v[64 + c] = t0[c];
    };
    for (int it = 0; it < ntiles; ++it) {
      const int mt = blockIdx.x + it * gridDim.x;
      const long long token = (long long)mt * 128 + row;
      const bool valid = token < a.T;
      // ---- E1 (warps 2-5 / 6-9): H sub-tiles of this group ----
      for (int nb = grp; nb < 4 && grp < 2; nb += 2) {
        const uint32_t k = (uint32_t)it * 2 + (nb >> 1);
        FFN_WAIT(&tfull1[nb], it & 1, 8);
        tc_fence_after();
        float v[96];
        load_acc(nb * 96, v);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty1[nb]);
        const float4 *bias4 = reinterpret_cast<const float4 *>(sB1 + nb * 96);
#pragma unroll
        for (int c4 = 0; c4 < 24; ++c4) {
          const float4 bb = bias4[c4];
          v[4 * c4] += bb.x; v[4 * c4 + 1] += bb.y; v[4 * c4 + 2] += bb.z; v[4 * c4 + 3] += bb.w;
        }
        uint4 pk[12];
#pragma unroll
        for (int cc = 0; cc < 12; ++cc) {
          float x[8];
#pragma unroll
          for (int jx = 0; jx < 8; ++jx) x[jx] = fmaxf(v[cc * 8 + jx], 0.f);
          if (a.thr16) drop8(x, ((uint64_t)token * 384 + nb * 96) / 8 + cc, a.thr16, a.dscale, a.key_h);
          pk[cc] = pack8_bf16(x);
        }
        // the previous slice (the other group's) has been consumed by its MMAs: group 0's k-th turn follows the (k-1)-th
        // hand-over to it (none before its first), group 1's k-th turn the k-th
        FFN_WAIT(&h_free[grp], grp == 0 ? ((k & 1) ^ 1) : (k & 1), 9);
        uint4 *o = reinterpret_cast<uint4 *>(sH) + row;
#pragma unroll
        for (int cc = 0; cc < 12; ++cc) o[cc * 128] = pk[cc];
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&h_ready[grp]);
      }
      // ---- E2 (warps 10-13): residual + LayerNorm epilogue of every tile ----
      if (grp != 2) continue;
      const int s = it & 1;
      FFN_WAIT(acc2_full, it & 1, 10);
      FFN_WAIT(&full[s], (it >> 1) & 1, 11);            // X1 tile (TMA-written) visible to this thread: residual operand
      tc_fence_after();
      float v[96];
      load_acc(384, v);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc2_empty);
      {
        const float4 *bias4 = reinterpret_cast<const float4 *>(sB2);
#pragma unroll
        for (int c4 = 0; c4 < 24; ++c4) {
          const float4 bb = bias4[c4];
          v[4 * c4] += bb.x; v[4 * c4 + 1] += bb.y; v[4 * c4 + 2] += bb.z; v[4 * c4 + 3] += bb.w;
        }
      }
      const uint4 *res = reinterpret_cast<const uint4 *>(sA + s * SLICE_BYTES) + row;
#pragma unroll
      for (int cc = 0; cc < 12; ++cc) {
        if (a.thr16) drop8(&v[cc * 8], (uint64_t)token * 12 + cc, a.thr16, a.dscale, a.key_f);
        float r8[8];
        unpack8_bf16(res[cc * 128], r8);
#pragma unroll
        for (int jx = 0; jx < 8; ++jx) v[cc * 8 + jx] += r8[jx];
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[s]);
      layer_norm96(v, sLn, sLn + 96);
      if (FINAL && a.ln2_w != nullptr) layer_norm96(v, sLn + 192, sLn + 288);
      if (!FINAL || a.out_img != nullptr) {
        uint4 *o = reinterpret_cast<uint4 *>(a.out_img) + ((size_t)mt * 12) * 128 + row;
#pragma unroll
        for (int cc = 0; cc < 12; ++cc) o[cc * 128] = pack8_bf16(&v[cc * 8]);
      }
      if (FINAL && a.out_f32 != nullptr && valid) {
        float *o = a.out_f32 + token * 96;
#pragma unroll
        for (int c = 0; c < 96; c += 4) *reinterpret_cast<float4 *>(o + c) = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
      }
      if (FINAL && a.seq_img != nullptr && valid) {
        const long long sq = token / a.P;
        const int pp = (int)(token - sq * a.P);
        const long long bb = sq / a.seq_nodes;
        const int nn = (int)(sq - bb * a.seq_nodes);
        uint4 *o = reinterpret_cast<uint4 *>(a.seq_img) + ((size_t)bb * a.P * 12 + (size_t)pp * 12) * a.seq_rows + nn;
#pragma unroll
        for (int cc = 0; cc < 12; ++cc) o[(size_t)cc * a.seq_rows] = pack8_bf16(&v[cc * 8]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

static size_t tff_smem_bytes() { return 2 * (size_t)TFF_W_BYTES + 3 * (size_t)SLICE_BYTES + 22 * 8 + (384 + 96 + 4 * 96) * 4 + 16; }

// ---------------------------------------------------------------------------
static size_t tcl_smem_bytes(int K, int Nout) {
  return (size_t)K * Nout * 2 + TCL_STAGES * SLICE_BYTES + 32 * 8 + (384 + 4 * 96) * 4 + 16;
}
static size_t tca_smem_bytes(int Pk) {
  const size_t zrows = Pk > 128 ? Pk : 128;
  if (Pk > TCA_KSPLIT)
    return TCA_QBUF * 6144 + 2 * TCA_KVBUF_SPLIT * (size_t)(3 * Pk * 16) + zrows * 16 + 2 * (size_t)(TCA_KSPLIT / 8) * 2048 +
           2 * 128 * TCA_XROW * 4 + 32 * 8 + 16;
  return TCA_QBUF * 6144 + 2 * TCA_KVBUF * (size_t)(3 * Pk * 16) + zrows * 16 + 2 * (size_t)(Pk / 8) * 2048 + 32 * 8 + 16;
}

static int tc_linear_launch(const TcLinearArgs &a, cudaStream_t st) {
  if (!((a.K == 96 || a.K == 384) && a.Nout % 96 == 0 && a.Nout >= 96 && a.Nout <= 384))
    return fail(STEP_EUNSUPPORTED, "tc_linear: unsupported shape K=%lld Nout=%lld", a.K, a.Nout);
  const size_t smem = tcl_smem_bytes(a.K, a.Nout);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int grid = a.MT < sms ? a.MT : sms;
  const bool fin = (a.mode == TCM_RESLN) && (a.ln2_w != nullptr || a.out_f32 != nullptr || a.seq_img != nullptr);
  int rc;
#define TCL_LAUNCH(M, F)                                                        \
  do {                                                                          \
    if ((rc = allow_smem(tc_linear_kernel<M, F>, 227 * 1024))) return rc;       \
    tc_linear_kernel<M, F><<<grid, TCL_THREADS, smem, st>>>(a);                 \
  } while (0)
  switch (a.mode) {
    case TCM_F32: TCL_LAUNCH(TCM_F32, false); break;
    case TCM_RELU_IMG: TCL_LAUNCH(TCM_RELU_IMG, false); break;
    case TCM_QKV: TCL_LAUNCH(TCM_QKV, false); break;
    default:
      if (fin) TCL_LAUNCH(TCM_RESLN, true);
      else TCL_LAUNCH(TCM_RESLN, false);
  }
#undef TCL_LAUNCH
  return check_launch("tc_linear_kernel");
}

static size_t tlk_smem_bytes() { return TLK_RING * (size_t)TLK_SLICE + 2 * (size_t)SLICE_BYTES + (96 + 384 + 96 + 288 + 6 * 96) * 4 + 17 * 8 + 16; }

static int tc_layer_launch(const TcLayerArgs &a, cudaStream_t st) {
  int dev = 0, sms = 148, rc;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const size_t smem = tlk_smem_bytes();
  if ((rc = allow_smem(tc_layer_kernel, smem))) return rc;
  const int grid = a.MT < 2 * sms ? a.MT : 2 * sms;
  tc_layer_kernel<<<grid, TLK_THREADS, smem, st>>>(a);
  return check_launch("tc_layer_kernel");
}

static int tc_ffn_launch(const TcFfnArgs &a, cudaStream_t st) {
  int dev = 0, sms = 148, rc;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const size_t smem = tff_smem_bytes();
  const int grid = a.MT < sms ? a.MT : sms;
  const bool fin = a.ln2_w != nullptr || a.out_f32 != nullptr || a.seq_img != nullptr;
  if (fin) {
    if ((rc = allow_smem(tc_ffn_kernel<true>, smem))) return rc;
    tc_ffn_kernel<true><<<grid, TFF_THREADS, smem, st>>>(a);
  } else {
    if ((rc = allow_smem(tc_ffn_kernel<false>, smem))) return rc;
    tc_ffn_kernel<false><<<grid, TFF_THREADS, smem, st>>>(a);
  }
  return check_launch("tc_ffn_kernel");
}

// STEP_B200_FFN_FUSED=1 selects the one-launch feed-forward kernel.  Default off: measured 0.51 ms per layer against
// 0.42 ms for the two HBM-bound tc_linear launches (profiles/r02_fused_ffn.md) - the per-row epilogue chains, not the
// 768 B/token H round trip, set its pace.
static bool tc_use_fused_ffn() {
  const char *e = getenv("STEP_B200_FFN_FUSED");
  return e && e[0] == '1';
}

}  // namespace stepk

using namespace stepk;

extern "C" int step_tc_pack_weight(const float *w, int Nout, int K, void *img, void *stream) {
  STEP_REQUIRE(w && img && Nout > 0 && K > 0 && K % 8 == 0, "tc_pack_weight: bad argument");
  const int units = Nout * (K / 8);
  tc_pack_weight_kernel<<<(units + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w, Nout, K, reinterpret_cast<uint4 *>(img));
  return check_launch("tc_pack_weight_kernel");
}

extern "C" int step_tc_rows_to_image(const float *x, long long T, int K, void *img, void *stream) {
  STEP_REQUIRE(x && img && T > 0 && K % 8 == 0, "tc_rows_to_image: bad argument");
  const long long units = ((T + 127) / 128) * (K / 8) * 128;
  tc_rows_to_image_kernel<<<(unsigned)((units + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, T, K, reinterpret_cast<uint4 *>(img));
  return check_launch("tc_rows_to_image_kernel");
}

extern "C" int step_tc_image_to_rows(const void *img, long long T, int K, float *x, void *stream) {
  STEP_REQUIRE(x && img && T > 0 && K % 8 == 0, "tc_image_to_rows: bad argument");
  const long long units = ((T + 127) / 128) * (K / 8) * 128;
  tc_image_to_rows_kernel<<<(unsigned)((units + 255) / 256), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const uint4 *>(img), T, K, x);
  return check_launch("tc_image_to_rows_kernel");
}

extern "C" int step_tc_linear(const void *a_img, const void *w_img, const float *bias, long long T, int K, int Nout, int mode,
                              const void *res_img, const float *ln_w, const float *ln_b, void *out_img, float *out_f32,
                              void *stream) {
  STEP_REQUIRE(a_img && w_img && bias && T > 0, "tc_linear: bad argument");
  STEP_REQUIRE(mode == TCM_F32 || mode == TCM_RELU_IMG || mode == TCM_RESLN, "tc_linear: bad mode");
  if (mode == TCM_RESLN) STEP_REQUIRE(res_img && ln_w && ln_b && Nout == 96, "tc_linear: residual+LN needs its operands");
  TcLinearArgs a{};
  a.A = (const uint8_t *)a_img; a.W = (const uint8_t *)w_img; a.bias = bias;
  a.MT = (int)((T + 127) / 128); a.K = K; a.Nout = Nout; a.mode = mode; a.T = T;
  a.res = (const uint8_t *)res_img; a.ln_w = ln_w; a.ln_b = ln_b;
  a.out_img = (uint8_t *)out_img; a.out_f32 = out_f32;
  a.dscale = 1.f;
  return tc_linear_launch(a, (cudaStream_t)stream);
}

extern "C" int step_tc_embed_fwd(const float *series, long long sB, long long sT, long long sN, int B, int N, int P,
                                 const float *patch_w, const float *patch_b, const float *pos, void *x_img, float drop_p,
                                 unsigned long long seed, void *stream) {
  STEP_REQUIRE(series && patch_w && patch_b && pos && x_img && B > 0 && N > 0 && P > 0, "tc_embed: bad argument");
  STEP_REQUIRE(drop_p >= 0.f && drop_p < 1.f, "tc_embed: drop_p must be in [0, 1)");
  uint32_t thr16 = 0; float dscale = 1.f;
  if (drop_p > 0.f) { thr16 = (uint32_t)(drop_p * 65536.0f); dscale = 1.f / (1.f - drop_p); }
  tc_embed_kernel<<<dim3((P + 31) / 32, (N + 15) / 16, B), 256, 0, (cudaStream_t)stream>>>(
      series, sB, sT, sN, N, P, patch_w, patch_b, pos, reinterpret_cast<uint4 *>(x_img), thr16, dscale, rng_key(seed, 1));
  return check_launch("tc_embed_kernel");
}

extern "C" int step_tc_linear_drop(const void *a_img, const void *w_img, const float *bias, long long T, int K, int Nout, int mode,
                                   const void *res_img, const float *ln_w, const float *ln_b, void *out_img, float *out_f32,
                                   float drop_p, unsigned long long seed, void *stream) {
  STEP_REQUIRE(a_img && w_img && bias && T > 0, "tc_linear_drop: bad argument");
  STEP_REQUIRE(mode == TCM_RELU_IMG || mode == TCM_RESLN, "tc_linear_drop: dropout sites exist in modes 1 and 2 only");
  STEP_REQUIRE(drop_p >= 0.f && drop_p < 1.f, "tc_linear_drop: drop_p must be in [0, 1)");
  if (mode == TCM_RESLN) STEP_REQUIRE(res_img && ln_w && ln_b && Nout == 96, "tc_linear_drop: residual+LN needs its operands");
  TcLinearArgs a{};
  a.A = (const uint8_t *)a_img; a.W = (const uint8_t *)w_img; a.bias = bias;
  a.MT = (int)((T + 127) / 128); a.K = K; a.Nout = Nout; a.mode = mode; a.T = T;
  a.res = (const uint8_t *)res_img; a.ln_w = ln_w; a.ln_b = ln_b;
  a.out_img = (uint8_t *)out_img; a.out_f32 = out_f32;
  a.dscale = 1.f;
  if (drop_p > 0.f) { a.thr16 = (uint32_t)(drop_p * 65536.0f); a.dscale = 1.f / (1.f - drop_p); a.key = rng_key(seed, 0); }
  return tc_linear_launch(a, (cudaStream_t)stream);
}

extern "C" size_t step_tc_attn_image_bytes(int S, int P, int which) {
  const int Pk = (P + 15) / 16 * 16, RT = (P + 127) / 128;
  if (which == 0) return (size_t)S * 4 * RT * 6144;
  if (which == 2) return (size_t)S * 4 * (P + 1) * sizeof(float);   // row-maximum bound workspace
  return (size_t)S * 4 * 3 * Pk * 16;
}

// memset of the max |k| slots + the TCM_QKV arguments shared by the public entry point and the encoder driver
static int tc_qkv_bound_reset(float *bound, long long S, cudaStream_t st) {
  if (bound == nullptr) return STEP_OK;
  cudaError_t e = cudaMemsetAsync(bound, 0, (size_t)S * 4 * sizeof(float), st);
  return e == cudaSuccess ? STEP_OK : fail_msg((int)e, cudaGetErrorString(e));
}

extern "C" int step_tc_qkv(const void *x_img, const void *w_img, const float *bias, int S, int P, void *q_img, void *k_img,
                           void *v_img, float *bound, void *stream) {
  STEP_REQUIRE(x_img && w_img && bias && q_img && k_img && v_img && S > 0 && P > 0, "tc_qkv: bad argument");
  int rc0 = tc_qkv_bound_reset(bound, S, (cudaStream_t)stream);
  if (rc0) return rc0;
  TcLinearArgs a{};
  a.bound = bound; a.nseq = S;
  const long long T = (long long)S * P;
  a.A = (const uint8_t *)x_img; a.W = (const uint8_t *)w_img; a.bias = bias;
  a.MT = (int)((T + 127) / 128); a.K = 96; a.Nout = 288; a.mode = TCM_QKV; a.T = T;
  a.q_img = (uint8_t *)q_img; a.k_img = (uint8_t *)k_img; a.v_img = (uint8_t *)v_img;
  a.P = P; a.Pk = (P + 15) / 16 * 16; a.RT = (P + 127) / 128;
  a.qscale = 0.20412414523193154f * 1.4426950408889634f;
  a.dscale = 1.f;
  return tc_linear_launch(a, (cudaStream_t)stream);
}

static int tc_attn_launch(const void *q_img, const void *k_img, const void *v_img, void *o_img, const float *bound, int S, int P,
                          float drop_p, uint64_t seed, uint32_t site, cudaStream_t st) {
  TcAttnArgs a{};
  a.bound = bound;
  a.q_img = (const uint8_t *)q_img; a.k_img = (const uint8_t *)k_img; a.v_img = (const uint8_t *)v_img; a.o_img = (uint8_t *)o_img;
  a.S = S; a.P = P; a.Pk = (P + 15) / 16 * 16; a.RT = (P + 127) / 128;
  if (a.Pk > 2 * TCA_KSPLIT) return fail(STEP_EUNSUPPORTED, "tc_attention: P=%lld > 352 is served by the fp32 path", P);
  if (drop_p > 0.f) { a.thr16 = (uint32_t)(drop_p * 65536.0f); a.dscale = 1.f / (1.f - drop_p); }
  else { a.thr16 = 0; a.dscale = 1.f; }
  a.key = rng_key(seed, site);
  int dev = 0, sms = 148, rc;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int grid = S < sms ? S : sms;
  const size_t smem = tca_smem_bytes(a.Pk);
#define TCA_LAUNCH(PF, DR, SP)                                                   \
  do {                                                                           \
    if ((rc = allow_smem(tc_attn_kernel<PF, DR, SP>, 227 * 1024))) return rc;    \
    tc_attn_kernel<PF, DR, SP><<<grid, TCA_THREADS, smem, st>>>(a);              \
  } while (0)
  if (P == 168) { if (a.thr16) TCA_LAUNCH(168, true, false); else TCA_LAUNCH(168, false, false); }
  else if (P == 336) { if (a.thr16) TCA_LAUNCH(336, true, true); else TCA_LAUNCH(336, false, true); }
  else if (a.Pk > TCA_KSPLIT) { if (a.thr16) TCA_LAUNCH(0, true, true); else TCA_LAUNCH(0, false, true); }
  else { if (a.thr16) TCA_LAUNCH(0, true, false); else TCA_LAUNCH(0, false, false); }
#undef TCA_LAUNCH
  return check_launch("tc_attn_kernel");
}

extern "C" int step_tc_attention(const void *q_img, const void *k_img, const void *v_img, void *o_img, const float *bound, int S,
                                 int P, float drop_p, unsigned long long seed, void *stream) {
  STEP_REQUIRE(q_img && k_img && v_img && o_img && S > 0 && P > 0, "tc_attention: bad argument");
  return tc_attn_launch(q_img, k_img, v_img, o_img, bound, S, P, drop_p, seed, 0, (cudaStream_t)stream);
}

// host-only: the packed bf16x2 threshold pattern the attention kernel compares its random halves with (see drop_thr_bf16x2)
extern "C" unsigned int step_tc_attn_drop_threshold(float drop_p) {
  if (!(drop_p > 0.f) || !(drop_p < 1.f)) return 0u;
  return drop_thr_bf16x2((uint32_t)(drop_p * 65536.0f));
}

extern "C" size_t step_tc_seq_image_bytes(int B, int N, int P) {
  const size_t R = (size_t)(N + 127) / 128 * 128;
  return (size_t)B * P * 12 * R * 16;
}

extern "C" int step_tc_hidden_to_seq_image(const float *hidden, int B, int N, int P, void *seq_img, void *stream) {
  STEP_REQUIRE(hidden && seq_img && B > 0 && N > 0 && P > 0, "tc_hidden_to_seq_image: bad argument");
  const long long units = (long long)B * P * 12 * N;
  tc_hidden_to_seq_image_kernel<<<(unsigned)((units + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      hidden, B, N, P, (N + 127) / 128 * 128, reinterpret_cast<uint4 *>(seq_img));
  return check_launch("tc_hidden_to_seq_image_kernel");
}

static int tc_gram_raw_launch(const void *seq_img, int B, int N, int P, int tile_first, int tile_step, float *gram, cudaStream_t st) {
  if ((P * 12) % TG_KC != 0) return fail(STEP_EUNSUPPORTED, "tc_cosine_gram: P*12 = %lld must be a multiple of 8", (long long)P * 12);
  TcGramArgs a{};
  a.img = (const uint8_t *)seq_img; a.gram = gram; a.N = N; a.R = (N + 127) / 128 * 128; a.KC = P * 12;
  a.tile_first = tile_first; a.tile_step = tile_step;
  const int tiles = a.R / 128;
  const int mine = tile_first < tiles ? (tiles - tile_first + tile_step - 1) / tile_step : 0;
  if (mine == 0) return STEP_OK;
  const int nblk = (N + 255) / 256;
  const int Rb = a.R < 256 ? a.R : 256;
  const size_t smem = TG_STAGES * (size_t)(TG_KC * 2048 + TG_KC * Rb * 16) + 16 * 8 + 16;
  int rc = allow_smem(tc_gram_kernel, 227 * 1024);
  if (rc) return rc;
  tc_gram_kernel<<<dim3(nblk, mine, B), 192, smem, st>>>(a);
  return check_launch("tc_gram_kernel");
}

extern "C" int step_tc_gram_rows(const void *seq_img, int B, int N, int P, int tile_first, int tile_step, float *gram, void *stream) {
  STEP_REQUIRE(seq_img && gram && B > 0 && N > 0 && P > 0 && tile_first >= 0 && tile_step >= 1, "tc_gram_rows: bad argument");
  return tc_gram_raw_launch(seq_img, B, N, P, tile_first, tile_step, gram, (cudaStream_t)stream);
}

extern "C" int step_gram_normalize(const float *gram, int B, int N, float *sim, void *stream) {
  STEP_REQUIRE(gram && sim && B > 0 && N > 0, "gram_normalize: bad argument");
  const long long per = (long long)N * N;
  gram_normalize_kernel<<<dim3((unsigned)((per + 255) / 256), B), 256, 0, (cudaStream_t)stream>>>(gram, N, sim);
  return check_launch("gram_normalize_kernel");
}

extern "C" int step_tc_cosine_gram(const void *seq_img, int B, int N, int P, float *gram_scratch, float *sim, void *stream) {
  STEP_REQUIRE(seq_img && gram_scratch && sim && B > 0 && N > 0 && P > 0, "tc_cosine_gram: bad argument");
  int rc = tc_gram_raw_launch(seq_img, B, N, P, 0, 1, gram_scratch, (cudaStream_t)stream);
  if (rc) return rc;
  return step_gram_normalize(gram_scratch, B, N, sim, stream);
}

// packed weight images of one encoder layer
extern "C" size_t step_ts_encoder_bf16_workspace_bytes(int B, int N, int P) {
  const long long S = (long long)B * N, T = S * P, MT = (T + 127) / 128;
  const int Pk = (P + 15) / 16 * 16, RT = (P + 127) / 128;
  size_t b = 0;
  b += 4 * (size_t)MT * SLICE_BYTES;                // X, X1, X2, O images
  b += (size_t)MT * 4 * SLICE_BYTES;                // H image (K = 384)
  b += (size_t)S * 4 * RT * 6144;                   // Q
  b += 2 * (size_t)S * 4 * 3 * Pk * 16;             // K, V
  b += (size_t)S * 4 * (P + 1) * sizeof(float) + 1024;   // row-maximum bound: max |k| per (sequence, head), |q| per query
  return b + 4096;
}

extern "C" int step_ts_encoder_fwd_bf16(const float *series, long long sB, long long sT, long long sN, int B, int N, int P,
                                        const float *patch_w, const float *patch_b, const float *pos,
                                        const step_ts_layer_weights *L, const step_ts_layer_images *I, int n_layers,
                                        const float *fnw, const float *fnb, float *hidden, void *seq_img, void *workspace,
                                        size_t workspace_bytes, float drop_p, unsigned long long seed, void *stream) {
  STEP_REQUIRE(series && patch_w && patch_b && pos && L && I && fnw && fnb && hidden && workspace, "ts_encoder_bf16: null pointer");
  STEP_REQUIRE(n_layers >= 1 && B > 0 && N > 0 && P > 0, "ts_encoder_bf16: bad shape");
  if (workspace_bytes < step_ts_encoder_bf16_workspace_bytes(B, N, P))
    return fail(STEP_EWORKSPACE, "ts_encoder_bf16: workspace too small (%lld bytes needed)",
                (long long)step_ts_encoder_bf16_workspace_bytes(B, N, P));
  cudaStream_t st = (cudaStream_t)stream;
  const long long S = (long long)B * N, T = S * P, MT = (T + 127) / 128;
  const int Pk = (P + 15) / 16 * 16, RT = (P + 127) / 128;
  uint8_t *ws = reinterpret_cast<uint8_t *>(((uintptr_t)workspace + 1023) & ~(uintptr_t)1023);
  uint8_t *X = ws; ws += (size_t)MT * SLICE_BYTES;
  uint8_t *X1 = ws; ws += (size_t)MT * SLICE_BYTES;
  uint8_t *X2 = ws; ws += (size_t)MT * SLICE_BYTES;
  uint8_t *O = ws; ws += (size_t)MT * SLICE_BYTES;
  uint8_t *H = ws; ws += (size_t)MT * 4 * SLICE_BYTES;
  uint8_t *Q = ws; ws += (size_t)S * 4 * RT * 6144;
  uint8_t *Kimg = ws; ws += (size_t)S * 4 * 3 * Pk * 16;
  uint8_t *Vimg = ws; ws += (size_t)S * 4 * 3 * Pk * 16;
  float *bound = reinterpret_cast<float *>(((uintptr_t)ws + 1023) & ~(uintptr_t)1023);
  uint32_t thr16 = 0; float dscale = 1.f;
  if (drop_p > 0.f) { thr16 = (uint32_t)(drop_p * 65536.0f); dscale = 1.f / (1.f - drop_p); }

  tc_embed_kernel<<<dim3((P + 31) / 32, (N + 15) / 16, B), 256, 0, st>>>(series, sB, sT, sN, N, P, patch_w, patch_b, pos,
                                                                        reinterpret_cast<uint4 *>(X), thr16, dscale,
                                                                        rng_key(seed, 1));
  STEP_LAUNCH_CHECK("tc_embed_kernel");
  uint8_t *cur = X, *nxt = X2;
  int rc;
  bool fused = true;                      // one token-block kernel per layer (needs the per-layer slice buffers)
  for (int l = 0; l < n_layers; ++l) fused = fused && (I[l].fused != nullptr);
  if (fused) {
    // QKV of layer 0 from the embedded tokens, then per layer: attention + ONE fused token-block kernel that also emits
    // the next layer's Q/K/V (2 launches per layer)
    TcLinearArgs a{};
    a.A = cur; a.W = (const uint8_t *)I[0].in_proj; a.bias = L[0].in_proj_b; a.MT = (int)MT; a.K = 96; a.Nout = 288;
    a.mode = TCM_QKV; a.T = T; a.q_img = Q; a.k_img = Kimg; a.v_img = Vimg; a.P = P; a.Pk = Pk; a.RT = RT;
    a.qscale = 0.20412414523193154f * 1.4426950408889634f; a.dscale = 1.f;
    a.bound = bound; a.nseq = S;
    if ((rc = tc_qkv_bound_reset(bound, S, st))) return rc;
    if ((rc = tc_linear_launch(a, st))) return rc;
    for (int l = 0; l < n_layers; ++l) {
      const uint32_t site = 16u * (l + 1);
      const bool last = (l == n_layers - 1);
      if ((rc = tc_attn_launch(Q, Kimg, Vimg, O, bound, (int)S, P, drop_p, seed, site + 1, st))) return rc;
      if (!last && (rc = tc_qkv_bound_reset(bound, S, st))) return rc;
      TcLayerArgs t{};
      t.bound = bound; t.nseq = S;
      t.O = O; t.X = cur; t.W = (const uint8_t *)I[l].fused;
      t.bo = L[l].out_proj_b; t.b1 = L[l].lin1_b; t.b2 = L[l].lin2_b; t.bqkv = last ? nullptr : L[l + 1].in_proj_b;
      t.ln1w = L[l].norm1_w; t.ln1b = L[l].norm1_b; t.ln2w = L[l].norm2_w; t.ln2b = L[l].norm2_b;
      t.MT = (int)MT; t.P = P; t.Pk = Pk; t.RT = RT; t.T = T; t.last = last ? 1 : 0;
      t.qscale = 0.20412414523193154f * 1.4426950408889634f;
      t.thr16 = thr16; t.dscale = dscale;
      t.key_o = rng_key(seed, site + 2); t.key_h = rng_key(seed, site + 3); t.key_f = rng_key(seed, site + 4);
      if (last) {
        t.fnw = fnw; t.fnb = fnb; t.hidden = hidden; t.seq_img = (uint8_t *)seq_img; t.seq_nodes = N;
        t.seq_rows = (N + 127) / 128 * 128;
      } else {
        t.Xout = nxt; t.q_img = Q; t.k_img = Kimg; t.v_img = Vimg;
      }
      if ((rc = tc_layer_launch(t, st))) return rc;
      uint8_t *tmp = cur; cur = nxt; nxt = tmp;
    }
    return STEP_OK;
  }
  for (int l = 0; l < n_layers; ++l) {
    const uint32_t site = 16u * (l + 1);
    TcLinearArgs a{};
    // QKV projection -> attention operand images
    a.A = cur; a.W = (const uint8_t *)I[l].in_proj; a.bias = L[l].in_proj_b; a.MT = (int)MT; a.K = 96; a.Nout = 288;
    a.mode = TCM_QKV; a.T = T; a.q_img = Q; a.k_img = Kimg; a.v_img = Vimg; a.P = P; a.Pk = Pk; a.RT = RT;
    a.qscale = 0.20412414523193154f * 1.4426950408889634f; a.dscale = 1.f;
    a.bound = bound; a.nseq = S;
    if ((rc = tc_qkv_bound_reset(bound, S, st))) return rc;
    if ((rc = tc_linear_launch(a, st))) return rc;
    if ((rc = tc_attn_launch(Q, Kimg, Vimg, O, bound, (int)S, P, drop_p, seed, site + 1, st))) return rc;
    // X1 = LN1(cur + drop(O Wo^T + bo))
    a = TcLinearArgs{};
    a.A = O; a.W = (const uint8_t *)I[l].out_proj; a.bias = L[l].out_proj_b; a.MT = (int)MT; a.K = 96; a.Nout = 96;
    a.mode = TCM_RESLN; a.T = T; a.res = cur; a.ln_w = L[l].norm1_w; a.ln_b = L[l].norm1_b; a.out_img = X1;
    a.thr16 = thr16; a.dscale = dscale; a.key = rng_key(seed, site + 2);
    if ((rc = tc_linear_launch(a, st))) return rc;
    const bool last = (l == n_layers - 1);
    if (tc_use_fused_ffn()) {
      // X2 = LN2(X1 + drop(drop(relu(X1 W1^T + b1)) W2^T + b2)) in one launch: the hidden activations stay on chip
      TcFfnArgs f{};
      f.A = X1; f.W1 = (const uint8_t *)I[l].lin1; f.W2 = (const uint8_t *)I[l].lin2;
      f.b1 = L[l].lin1_b; f.b2 = L[l].lin2_b; f.ln_w = L[l].norm2_w; f.ln_b = L[l].norm2_b;
      f.MT = (int)MT; f.T = T; f.P = P;
      if (last) {
        f.ln2_w = fnw; f.ln2_b = fnb; f.out_f32 = hidden; f.out_img = nullptr;
        f.seq_img = (uint8_t *)seq_img; f.seq_nodes = N; f.seq_rows = (N + 127) / 128 * 128;
      } else {
        f.out_img = nxt;
      }
      f.thr16 = thr16; f.dscale = dscale; f.key_h = rng_key(seed, site + 3); f.key_f = rng_key(seed, site + 4);
#ifdef STEP_FFN_DEBUG
      { const char *e = getenv("STEP_FFN_DEBUG_PTR"); f.dbg = e ? (volatile int *)strtoull(e, nullptr, 0) : nullptr; }
#endif
      if ((rc = tc_ffn_launch(f, st))) return rc;
    } else {
    // H = drop(relu(X1 W1^T + b1))
    a = TcLinearArgs{};
    a.A = X1; a.W = (const uint8_t *)I[l].lin1; a.bias = L[l].lin1_b; a.MT = (int)MT; a.K = 96; a.Nout = 384;
    a.mode = TCM_RELU_IMG; a.T = T; a.out_img = H; a.thr16 = thr16; a.dscale = dscale; a.key = rng_key(seed, site + 3);
    if ((rc = tc_linear_launch(a, st))) return rc;
    // X2 = LN2(X1 + drop(H W2^T + b2)); last layer: + encoder_norm, fp32 row-major hidden
    a = TcLinearArgs{};
    a.A = H; a.W = (const uint8_t *)I[l].lin2; a.bias = L[l].lin2_b; a.MT = (int)MT; a.K = 384; a.Nout = 96;
    a.mode = TCM_RESLN; a.T = T; a.res = X1; a.ln_w = L[l].norm2_w; a.ln_b = L[l].norm2_b;
    if (last) {
      a.ln2_w = fnw; a.ln2_b = fnb; a.out_f32 = hidden; a.out_img = nullptr;
      a.seq_img = (uint8_t *)seq_img; a.seq_nodes = N; a.seq_rows = (N + 127) / 128 * 128; a.P = P;
    }
    else a.out_img = nxt;
    a.thr16 = thr16; a.dscale = dscale; a.key = rng_key(seed, site + 4);
    if ((rc = tc_linear_launch(a, st))) return rc;
    }
    uint8_t *t = cur; cur = nxt; nxt = t;
  }
  return STEP_OK;
}
