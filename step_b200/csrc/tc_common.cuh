// tcgen05 / TMEM / TMA-bulk / mbarrier PTX wrappers (sm_100a).  Hand-written: no CUTLASS.
//
// Operand layouts used everywhere in this library ("tile images"):
//   K-major, no swizzle (UMMA "interleave" canonical layout): a [R rows x K] bf16 operand is stored as
//   [K/8 chunks][R rows][8 elements]; one 16-byte unit = 8 consecutive K elements of one row, the 8 rows
//   of a core matrix are 128 contiguous bytes.  Descriptor: LBO = byte distance between consecutive
//   K chunks (= R*16), SBO = byte distance between consecutive 8-row groups (= 128).
//   MN-major, no swizzle (used for V in P.V): [MN/8 groups][K rows][8 elements]; LBO = distance between
//   8-row K groups (= 128), SBO = distance between MN groups (= Krows*16).
// Because an image of a 128-row tile is one contiguous block in global memory, a whole operand tile is
// fetched with a single 1-D TMA bulk copy (cp.async.bulk, SASS UBLKCP) that signals an mbarrier.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier -------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Bounded spin: a protocol bug traps (kernel error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done = 0;
  for (uint32_t it = 0; it < (1u << 28); ++it) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) return;
  }
  asm volatile("trap;");
}

// ---- TMA 1-D bulk copy global -> shared, completion on an mbarrier ------------------------------------
__device__ __forceinline__ void tma_bulk_g2s(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ---- TMEM ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t *smem_dst, uint32_t ncols) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // same warp that allocated
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 columns of 32-bit: thread i of the warp receives columns [col, col+32) of TMEM lane (base lane + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  tmem_wait_ld();
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  tmem_wait_ld();
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// issue-only variants (no wait): the destination registers are valid after the next tmem_wait_ld(); lets the load of
// block k+1 fly while block k is being processed
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, float (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]),
        "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15]), "=f"(v[16]),
        "=f"(v[17]), "=f"(v[18]), "=f"(v[19]), "=f"(v[20]), "=f"(v[21]), "=f"(v[22]), "=f"(v[23]), "=f"(v[24]),
        "=f"(v[25]), "=f"(v[26]), "=f"(v[27]), "=f"(v[28]), "=f"(v[29]), "=f"(v[30]), "=f"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, float (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]),
        "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15])
      : "r"(taddr)
      : "memory");
}

// wait for the loads issued above; the registers are threaded through the asm as in/out operands so that no
// arithmetic on them can be scheduled above the wait
__device__ __forceinline__ void tmem_wait_ld32(float (&v)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7]), "+f"(v[8]),
                 "+f"(v[9]), "+f"(v[10]), "+f"(v[11]), "+f"(v[12]), "+f"(v[13]), "+f"(v[14]), "+f"(v[15]), "+f"(v[16]),
                 "+f"(v[17]), "+f"(v[18]), "+f"(v[19]), "+f"(v[20]), "+f"(v[21]), "+f"(v[22]), "+f"(v[23]), "+f"(v[24]),
                 "+f"(v[25]), "+f"(v[26]), "+f"(v[27]), "+f"(v[28]), "+f"(v[29]), "+f"(v[30]), "+f"(v[31])
               :
               : "memory");
}
__device__ __forceinline__ void tmem_wait_ld16(float (&v)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7]), "+f"(v[8]),
                 "+f"(v[9]), "+f"(v[10]), "+f"(v[11]), "+f"(v[12]), "+f"(v[13]), "+f"(v[14]), "+f"(v[15])
               :
               : "memory");
}
// packed fp32 add (Blackwell FADD2, PTX add.rn.f32x2): (a0, a1) += (b0, b1) in one issue slot
__device__ __forceinline__ void fadd2(float &a0, float &a1, float b0, float b1) {
  asm("{\n\t.reg .b64 ra, rb;\n\t"
      "mov.b64 ra, {%0, %1};\n\tmov.b64 rb, {%2, %3};\n\t"
      "add.rn.f32x2 ra, ra, rb;\n\tmov.b64 {%0, %1}, ra;\n\t}"
      : "+f"(a0), "+f"(a1)
      : "f"(b0), "f"(b1));
}

// 64 columns in one instruction (fewer load round trips for reduction-only passes)
__device__ __forceinline__ void tmem_ld64(uint32_t taddr, float (&v)[64]) {
  uint32_t r[64];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32,%33,%34,%35,%36,%37,%38,%39,%40,%41,%42,%43,%44,%45,%46,%47,%48,%49,%50,%51,%52,%53,%54,%55,%56,%57,%58,%59,%60,%61,%62,%63}, [%64];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]), "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47]), "=r"(r[48]), "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]), "=r"(r[55]), "=r"(r[56]), "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
      : "r"(taddr)
      : "memory");
  tmem_wait_ld();
#pragma unroll
  for (int i = 0; i < 64; ++i) v[i] = __uint_as_float(r[i]);
}
// two loads (32 + 16 columns) in flight under one wait
__device__ __forceinline__ void tmem_ld32_16(uint32_t taddr32, uint32_t taddr16, float (&v)[32], float (&w)[16]) {
  uint32_t r[32], q[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr32)
      : "memory");
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(q[0]), "=r"(q[1]), "=r"(q[2]), "=r"(q[3]), "=r"(q[4]), "=r"(q[5]), "=r"(q[6]), "=r"(q[7]), "=r"(q[8]),
        "=r"(q[9]), "=r"(q[10]), "=r"(q[11]), "=r"(q[12]), "=r"(q[13]), "=r"(q[14]), "=r"(q[15])
      : "r"(taddr16)
      : "memory");
  tmem_wait_ld();
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
#pragma unroll
  for (int i = 0; i < 16; ++i) w[i] = __uint_as_float(q[i]);
}

// ---- UMMA descriptors -----------------------------------------------------------------------------------
// shared-memory matrix descriptor, SWIZZLE_NONE (bit layout: cute/arch/mma_sm100_desc.hpp SmemDescriptor):
//   [0,14) start address >> 4, [16,30) leading byte offset >> 4, [32,46) stride byte offset >> 4,
//   [46,48) version = 1, [49,52) base offset = 0, [52] lbo mode = 0, [61,64) layout type = 0.
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}
// instruction descriptor for kind::f16 with bf16 inputs, fp32 accumulation (InstrDescriptor bit layout):
//   [4,6) c_format = 1 (F32), [7,10) a_format = 1 (BF16), [10,13) b_format = 1 (BF16), [15] a_major, [16] b_major
//   (0 = K-major, 1 = MN-major), [17,23) N >> 3, [24,29) M >> 4.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread on behalf of the CTA
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier when every tcgen05 operation issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---- 256-bit streaming load (sm_100: LDG.E.256): 8 consecutive floats, 32-byte aligned, read-only path, no L1 allocation ----
struct f8 { float v[8]; };
__device__ __forceinline__ f8 ld256_nc(const float *p) {
  f8 r;
  asm volatile("ld.global.nc.L1::no_allocate.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]), "=f"(r.v[7])
               : "l"(p));
  return r;
}

// ---- bf16 packing -------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t *>(&v);
}
__device__ __forceinline__ uint4 pack8_bf16(const float *v) {
  return make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
}
__device__ __forceinline__ void unpack8_bf16(uint4 u, float *v) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = __uint_as_float(w[i] << 16);
    v[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
  }
}

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ---- counter hash of the tensor-core dropout sites (lowbias32-style finaliser: 2 multiplies + 2 xor-shifts) -------------
__device__ __forceinline__ uint32_t hash32(uint32_t x) {
  x *= 0x9E3779B1u; x ^= x >> 16; x *= 0x85EBCA77u; x ^= x >> 15;
  return x;
}

// ---- attention-probability dropout: two keep decisions per 32-bit random word -------------------------------------
// Each half of the word is compared AS A bf16 NUMBER with a threshold (one HSET2.BF16 for two elements, result 0xFFFF /
// 0x0000 per half, applied to the packed bf16 probabilities with one AND).  As numbers the 65536 patterns order as
// -inf = 0xFF80 < ... < 0x8001 < -0 = +0 < 0x0001 < ... < +inf, and the 254 NaN patterns fail every comparison, so
// "dropped" = NaNs + the (D - 254) most negative patterns for D = p * 65536 dropped patterns out of 65536: the keep
// probability is exactly 1 - D / 65536 for p >= 254 / 65536 (smaller p are served as 254 / 65536).
__host__ __device__ inline uint32_t drop_thr_bf16x2(uint32_t thr16) {
  const uint32_t need = thr16 > 254u ? thr16 - 254u : 0u;
  uint32_t t;
  if (need <= 32640u) t = 0xFF80u - need;
  else { t = need - 32641u; if (t > 0x7F80u) t = 0x7F80u; }
  return t | (t << 16);
}
__device__ __forceinline__ uint32_t keep_mask_bf16x2(uint32_t r, uint32_t thr2) {
  uint32_t m;
  asm("set.ge.u32.bf16x2 %0, %1, %2;" : "=r"(m) : "r"(r), "r"(thr2));
  return m;
}

// Placement of a (head, row tile) of the attention Q image in the 128 TMEM lanes: a last tile of <= 64 queries sits at
// lanes 64.. for odd heads, so that the partial tiles of consecutive heads are exponentiated by warps of different SM
// sub-partitions.
__host__ __device__ __forceinline__ int q_tail_offset(int P, int rt, int h) {
  return ((P - rt * 128) <= 64 && (h & 1)) ? 64 : 0;
}

}  // namespace tc
