// Fused attention on tcgen05/TMEM, head_dim 128 or 256 -- second schedule ("tc2").
//
// Same operator and building blocks as attention_tc.cu; different occupancy plan.  Instead of one CTA carrying
// two ping-pong Q tiles, each CTA carries ONE 128-row Q tile with K/V tiles of 64 keys, a DOUBLE-BUFFERED score
// accumulator, and only 256 TMEM columns / 96 KB smem / <= 128 registers, so TWO CTAs are resident per SM:
//   TMEM: S[0] (64 cols) | S[1] (64 cols) | O (128 cols); P[b] (bf16) aliases the first 32 columns of S[b].
//   The MMA warp issues S(j+2) right after PV(j), i.e. scores run two tiles ahead of the softmax, so the softmax
//   warpgroup never waits for its own MMAs; the other resident CTA fills the tensor pipe in the meantime.
// head_dim 256 (r2: the GDINO bi-attention, 4 heads x 256 -- modeling_ov_grounding_dino_mask_dn.py:893-1006): the same
// schedule with Q = 4 x 16 KB column chunks, K/V tiles of 64 keys x 512 B, O = 256 TMEM columns (S[0] | S[1] | O in a
// 512-column allocation), 193 KB smem => one CTA per SM.  KM = true adds an arbitrary key mask [batch, Tk] (1 = attend:
// the text / vision padding masks of the bi-attention); n_splits > 1 lets several CTAs share one query tile along the key
// axis (80 text queries over 21760 pixels) and write unnormalised partials in attention.cu's split-KV workspace layout.
#include "common.cuh"
#include "tc_common.cuh"

namespace {

constexpr int BQ = 128, BKV = 64, STG = 2;
constexpr int THREADS = 256;
template <int D> struct Cfg {
  static constexpr int NCH = D / 64;                         // 64-column (128-byte, one swizzle atom wide) chunks
  static constexpr int Q_BYTES = BQ * D * 2, Q_CHUNK = BQ * 128;
  static constexpr int KV_BYTES = BKV * D * 2, KV_CHUNK = BKV * 128;
  static constexpr int SMEM = Q_BYTES + 2 * STG * KV_BYTES + 1024 + 256;
  static constexpr int TMEM_COLS = D == 128 ? 256 : 512;     // S[0] | S[1] | O (power of two)
  static constexpr int CTAS = D == 128 ? 2 : 1;
};

struct Args {
  __nv_bfloat16* o;
  long long o_bs, o_ts;
  const int* seqlens;
  int Tq, Tk, heads, kv_heads, causal;
  float scale_log2;
  const unsigned char* key_mask;   // [batch, Tk], 1 = attend (KM instantiations only)
  int km_vec;                      // mask rows can be read as 16-byte vectors
  int n_splits;                    // CTAs per query tile along the key axis
  float* ws;                       // [batch*heads*n_splits*Tq][D + 2] fp32: unnormalised O, m (log2 domain), l
};

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ uint64_t desc_sw128(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((addr & 0x3FFFF) >> 4);
  d |= (uint64_t)(lbo_bytes >> 4) << 16;
  d |= (uint64_t)(sbo_bytes >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));    // low half = a
  return r;
}
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// p = exp2(s*scale - m) for 32 keys of this thread's row; packs bf16 P and stores it to TMEM (16 columns)
__device__ __forceinline__ void exp_half(const uint32_t (&r)[32], uint32_t taddr, float scale_log2, float m_use,
                                         float& rs0, float& rs1, float& rs2, float& rs3) {
  uint32_t pk[16];
#pragma unroll
  for (int k = 0; k < 32; k += 4) {
    const float p0 = ex2(fmaf(__uint_as_float(r[k]), scale_log2, -m_use));
    const float p1 = ex2(fmaf(__uint_as_float(r[k + 1]), scale_log2, -m_use));
    const float p2 = ex2(fmaf(__uint_as_float(r[k + 2]), scale_log2, -m_use));
    const float p3 = ex2(fmaf(__uint_as_float(r[k + 3]), scale_log2, -m_use));
    rs0 += p0; rs1 += p1; rs2 += p2; rs3 += p3;
    pk[k >> 1] = pack2(p0, p1);
    pk[(k >> 1) + 1] = pack2(p2, p3);
  }
  tmem_st_32x16(taddr, pk);
}

template <int D, bool KM>
__global__ void __launch_bounds__(THREADS, Cfg<D>::CTAS)
attn_fwd_tc2_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
                    const __grid_constant__ CUtensorMap tm_v, const Args a) {
  constexpr int NCH = Cfg<D>::NCH, Q_BYTES = Cfg<D>::Q_BYTES, Q_CHUNK = Cfg<D>::Q_CHUNK;
  constexpr int KV_BYTES = Cfg<D>::KV_BYTES, KV_CHUNK = Cfg<D>::KV_CHUNK, TMEM_COLS = Cfg<D>::TMEM_COLS;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - tc::smem_u32(smem_raw));
  const uint32_t sQ = base, sK = sQ + Q_BYTES, sV = sK + STG * KV_BYTES, bar = sV + STG * KV_BYTES;
  const uint32_t q_full = bar;
  auto k_full = [&](int s) { return bar + 8 * (1 + s); };
  auto v_full = [&](int s) { return bar + 8 * (3 + s); };
  auto k_empty = [&](int s) { return bar + 8 * (5 + s); };
  auto v_empty = [&](int s) { return bar + 8 * (7 + s); };
  auto s_full = [&](int b) { return bar + 8 * (9 + b); };
  auto p_ready = [&](int b) { return bar + 8 * (11 + b); };
  const uint32_t o_full = bar + 8 * 13;
  const uint32_t tmem_slot = bar + 8 * 14;
  // committed once, after the last PV: the epilogue cannot wait on o_full's parity, because when the softmax finishes
  // its last tile only PV(n-3) is known to have landed and o_full may still be two phases behind
  const uint32_t o_done = bar + 8 * 15;
  uint32_t* tmem_slot_gen = reinterpret_cast<uint32_t*>(gen + (tmem_slot - base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int split = blockIdx.x % a.n_splits;
  const int q0 = (blockIdx.x / a.n_splits) * BQ, head = blockIdx.y, b = blockIdx.z;
  const int kvh = head / (a.heads / a.kv_heads);
  const int len = a.seqlens ? min(a.seqlens[b], a.Tk) : a.Tk;
  const int coff = a.Tk - a.Tq;
  int k_end = len;
  if (a.causal) k_end = min(k_end, q0 + BQ + coff);
  const int n_all = k_end > 0 ? (k_end + BKV - 1) / BKV : 0;
  const int per_split = (n_all + a.n_splits - 1) / a.n_splits;
  const int t0 = split * per_split;                        // this CTA's key tiles: [t0, t0 + n)
  const int n = max(0, min(n_all - t0, per_split));

  if (warp == 0 && lane == 0) { tc::tma_prefetch_desc(&tm_q); tc::tma_prefetch_desc(&tm_k); tc::tma_prefetch_desc(&tm_v); }
  if (warp == 1 && lane == 0) {
    tc::mbar_init(q_full, 1);
    for (int s = 0; s < STG; ++s) {
      tc::mbar_init(k_full(s), 1); tc::mbar_init(v_full(s), 1); tc::mbar_init(k_empty(s), 1); tc::mbar_init(v_empty(s), 1);
      tc::mbar_init(s_full(s), 1); tc::mbar_init(p_ready(s), 128);
    }
    tc::mbar_init(o_full, 1);
    tc::mbar_init(o_done, 1);
    tc::mbar_fence_init();
  }
  if (warp == 2) tc::tmem_alloc<1>(tmem_slot, TMEM_COLS);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = *tmem_slot_gen;
  const uint32_t tO = tmem + 128;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (tc::elect_one() && n > 0) {
      tc::mbar_arrive_expect_tx(q_full, Q_BYTES);
      for (int h = 0; h < NCH; ++h) tma_load_3d(sQ + h * Q_CHUNK, &tm_q, q_full, head * D + h * 64, q0, b);
      for (int j = 0; j < n; ++j) {
        const int s = j % STG;
        const uint32_t ph = ((j / STG) & 1) ^ 1;
        tc::mbar_wait(k_empty(s), ph);
        tc::mbar_arrive_expect_tx(k_full(s), KV_BYTES);
        for (int h = 0; h < NCH; ++h) tma_load_3d(sK + s * KV_BYTES + h * KV_CHUNK, &tm_k, k_full(s), kvh * D + h * 64, (t0 + j) * BKV, b);
        tc::mbar_wait(v_empty(s), ph);
        tc::mbar_arrive_expect_tx(v_full(s), KV_BYTES);
        for (int h = 0; h < NCH; ++h) tma_load_3d(sV + s * KV_BYTES + h * KV_CHUNK, &tm_v, v_full(s), kvh * D + h * 64, (t0 + j) * BKV, b);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc_s = tc::umma_idesc_bf16_f32(BQ, BKV);
    constexpr uint32_t idesc_pv = tc::umma_idesc_bf16_f32(BQ, D) | (1u << 16);   // B (= V) MN-major
    auto issue_s = [&](int j) {           // S[j%2] = Q K_j^T
      const int s = j % STG;
      const uint32_t ka = sK + s * KV_BYTES;
#pragma unroll
      for (int kk = 0; kk < D / 16; ++kk)
        tc::umma_f16<1>(tmem + s * 64, desc_sw128(sQ + (kk >> 2) * Q_CHUNK + (kk & 3) * 32, 16, 1024),
                        desc_sw128(ka + (kk >> 2) * KV_CHUNK + (kk & 3) * 32, 16, 1024), idesc_s, kk != 0);
      tc::umma_commit<1>(s_full(s));
      tc::umma_commit<1>(k_empty(s));
    };
    auto issue_pv = [&](int j) {          // O (+)= P[j%2] V_j
      const int s = j % STG;
      const uint32_t va = sV + s * KV_BYTES;
#pragma unroll
      for (int kk = 0; kk < BKV / 16; ++kk)
        umma_ts(tO, tmem + s * 64 + kk * 8, desc_sw128(va + kk * 2048, KV_CHUNK, 1024), idesc_pv, (j | kk) != 0);
      tc::umma_commit<1>(o_full);
      tc::umma_commit<1>(v_empty(s));
    };
    if (n > 0) {
      tc::mbar_wait(q_full, 0);
      for (int t = 0; t < 2 && t < n; ++t) {
        tc::mbar_wait(k_full(t), 0);
        tc::tc_fence_after();
        if (tc::elect_one()) issue_s(t);
        __syncwarp();
      }
      for (int j = 0; j < n; ++j) {
        const int s = j % STG;
        const uint32_t ph = (j / STG) & 1;
        tc::mbar_wait(v_full(s), ph);
        tc::mbar_wait(p_ready(s), ph);
        tc::tc_fence_after();
        if (tc::elect_one()) issue_pv(j);
        __syncwarp();
        if (j + 2 < n) {
          tc::mbar_wait(k_full(s), ((j + 2) / STG) & 1);
          tc::tc_fence_after();
          if (tc::elect_one()) issue_s(j + 2);
          __syncwarp();
        }
      }
      if (tc::elect_one()) tc::umma_commit<1>(o_done);
      __syncwarp();
    }
  } else if (warp >= 4) {
    // ===================== softmax warpgroup: one thread per query row =====================
    const int quarter = warp & 3;
    const int row = q0 + quarter * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
    constexpr float RESCALE_THRESHOLD = 8.f;
    float m = -INFINITY, l = 0.f;
    for (int j = 0; j < n; ++j) {
      const int s = j % STG;
      const uint32_t tS = tmem + lane_addr + s * 64;
      tc::mbar_wait(s_full(s), (j / STG) & 1);
      tc::tc_fence_after();
      uint32_t ra[32], rb[32];                       // two 32-key halves (separate arrays stay in registers)
      tc::tmem_ld_32x32(tS, ra);
      tc::tmem_ld_32x32(tS + 32, rb);
      tc::tmem_ld_wait();
      const int n0 = (t0 + j) * BKV;
      if constexpr (KM) {
        // arbitrary key mask: the 64 mask bytes of this tile are the same for every row (broadcast loads)
        const unsigned char* km = a.key_mask + (size_t)b * a.Tk + n0;
        if (a.km_vec && n0 + BKV <= a.Tk) {
          const uint4* kp = reinterpret_cast<const uint4*>(km);
#pragma unroll
          for (int h = 0; h < 4; ++h) {
            const uint4 w = __ldg(kp + h);
            const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const bool keep = (ww[i >> 2] >> ((i & 3) * 8)) & 0xffu;
              if (!keep) { if (h < 2) ra[h * 16 + i] = 0xff800000u; else rb[(h - 2) * 16 + i] = 0xff800000u; }
            }
          }
        } else {
#pragma unroll
          for (int k = 0; k < 32; ++k) {
            if (n0 + k < a.Tk && !__ldg(km + k)) ra[k] = 0xff800000u;
            if (n0 + 32 + k < a.Tk && !__ldg(km + 32 + k)) rb[k] = 0xff800000u;
          }
        }
      }
      const bool need_mask = (n0 + BKV > len) || (a.causal && (n0 + BKV - 1 > q0 + coff));
      if (need_mask) {
        const int lim = (a.causal ? min(len, row + coff + 1) : len) - n0;
#pragma unroll
        for (int k = 0; k < 32; ++k) {
          if (k >= lim) ra[k] = 0xff800000u;
          if (k + 32 >= lim) rb[k] = 0xff800000u;
        }
      }
      float mx = -INFINITY;
#pragma unroll
      for (int k = 0; k < 32; k += 2) {
        mx = fmaxf(mx, fmaxf(__uint_as_float(ra[k]), __uint_as_float(ra[k + 1])));
        mx = fmaxf(mx, fmaxf(__uint_as_float(rb[k]), __uint_as_float(rb[k + 1])));
      }
      const float m_tile = mx * a.scale_log2;
      const bool grow = m_tile > m + RESCALE_THRESHOLD;
      if (j == 0) {
        m = m_tile;
      } else if (__any_sync(0xffffffffu, grow)) {
        const float m_new = grow ? m_tile : m;
        const float corr = (m == -INFINITY) ? 0.f : ex2(m - m_new);
        l *= corr;
        m = m_new;
        tc::mbar_wait(o_full, (j - 1) & 1);
        tc::tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < D; c += 16) {              // rare path: small chunks keep the score registers live
          uint32_t o[16];
          tmem_ld_32x16(tO + lane_addr + c, o);
          tc::tmem_ld_wait();
#pragma unroll
          for (int k = 0; k < 16; ++k) o[k] = __float_as_uint(__uint_as_float(o[k]) * corr);
          tmem_st_32x16(tO + lane_addr + c, o);
        }
      }
      const float m_use = (m == -INFINITY) ? 0.f : m;
      float rs0 = 0.f, rs1 = 0.f, rs2 = 0.f, rs3 = 0.f;
      exp_half(ra, tS, a.scale_log2, m_use, rs0, rs1, rs2, rs3);
      exp_half(rb, tS + 16, a.scale_log2, m_use, rs0, rs1, rs2, rs3);
      tmem_st_wait();
      tc::tc_fence_before();
      tc::mbar_arrive(p_ready(s));
      l += (rs0 + rs1) + (rs2 + rs3);
    }
    // epilogue: O / l -> bf16, 32 columns at a time
    if (n > 0) {
      tc::mbar_wait(o_done, 0);
      tc::tc_fence_after();
    }
    if (a.n_splits > 1) {
      // partial of this key range: unnormalised O, the running max actually used (log2 domain) and the sum
      float* wp = a.ws + ((((size_t)b * a.heads + head) * a.n_splits + split) * a.Tq + row) * (D + 2);
#pragma unroll 1
      for (int c = 0; c < D; c += 32) {
        uint32_t o[32];
        if (n > 0) { tc::tmem_ld_32x32(tO + lane_addr + c, o); tc::tmem_ld_wait(); }
        else {
#pragma unroll
          for (int k = 0; k < 32; ++k) o[k] = 0u;
        }
        if (row < a.Tq) {
#pragma unroll
          for (int k = 0; k < 32; k += 2) *reinterpret_cast<uint2*>(wp + c + k) = make_uint2(o[k], o[k + 1]);
        }
      }
      if (row < a.Tq) { wp[D] = n > 0 ? m : -INFINITY; wp[D + 1] = l; }
    } else {
    const float inv = l > 0.f ? 1.f / l : 0.f;
    __nv_bfloat16* op = a.o + b * a.o_bs + (long long)row * a.o_ts + head * D;
#pragma unroll
    for (int c = 0; c < D; c += 32) {
      uint32_t o[32];
      if (n > 0) { tc::tmem_ld_32x32(tO + lane_addr + c, o); tc::tmem_ld_wait(); }
      else {
#pragma unroll
        for (int k = 0; k < 32; ++k) o[k] = 0u;
      }
      if (row < a.Tq) {
#pragma unroll
        for (int k = 0; k < 32; k += 8) {
          uint4 u;
          __nv_bfloat162 h0 = __floats2bfloat162_rn(__uint_as_float(o[k]) * inv, __uint_as_float(o[k + 1]) * inv);
          __nv_bfloat162 h1 = __floats2bfloat162_rn(__uint_as_float(o[k + 2]) * inv, __uint_as_float(o[k + 3]) * inv);
          __nv_bfloat162 h2 = __floats2bfloat162_rn(__uint_as_float(o[k + 4]) * inv, __uint_as_float(o[k + 5]) * inv);
          __nv_bfloat162 h3 = __floats2bfloat162_rn(__uint_as_float(o[k + 6]) * inv, __uint_as_float(o[k + 7]) * inv);
          u.x = *reinterpret_cast<uint32_t*>(&h0); u.y = *reinterpret_cast<uint32_t*>(&h1);
          u.z = *reinterpret_cast<uint32_t*>(&h2); u.w = *reinterpret_cast<uint32_t*>(&h3);
          *reinterpret_cast<uint4*>(op + c + k) = u;
        }
      }
    }
    }
  }

  tc::tc_fence_before();
  __syncthreads();
  if (warp == 2) tc::tmem_dealloc<1>(tmem, TMEM_COLS);
}

int make_tmap(CUtensorMap* m, const void* base, uint64_t cols, uint64_t tokens, uint64_t batch, uint64_t token_pitch,
              uint64_t batch_pitch, uint32_t box_rows) {
  PFN_cuTensorMapEncodeTiled_v12000 enc = vllm_tma_encoder();
  if (!enc) return -100;
  cuuint64_t dims[3] = {cols, tokens, batch};
  cuuint64_t strides[2] = {token_pitch * 2, batch_pitch * 2};
  cuuint32_t box[3] = {64, box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  if (batch == 1) strides[1] = token_pitch * 2 * (tokens > 0 ? tokens : 1);
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : -101;
}

}  // namespace

template <int D, bool KM>
static int launch_tc2(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const Args& a, int batch,
                      cudaStream_t st) {
  auto kern = attn_fwd_tc2_kernel<D, KM>;
  static bool set = false;
  if (!set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<D>::SMEM);
    if (e != cudaSuccess) return (int)e;
    set = true;
  }
  dim3 grid((unsigned)(((a.Tq + BQ - 1) / BQ) * a.n_splits), a.heads, batch);
  kern<<<grid, THREADS, Cfg<D>::SMEM, st>>>(tq, tk, tv, a);
  VLLM_CHECK_LAUNCH();
  return VLLM_OK;
}

// head_dim 128 / 256; key_mask optional ([batch, Tk] bytes, 1 = attend); n_splits > 1: partials go to `ws`
// ([batch*heads*n_splits*Tq][head_dim + 2] fp32) and the caller merges them (attention.cu splitkv_combine_kernel).
int vllm_attention_tc2(const void* q, const void* k, const void* v, void* o, int batch, int Tq, int Tk, int heads,
                       int kv_heads, int head_dim, long long q_bs, long long q_ts, long long k_bs, long long k_ts,
                       long long v_bs, long long v_ts, long long o_bs, long long o_ts, const int* seqlens,
                       const unsigned char* key_mask, int causal, float scale, int n_splits, float* ws, cudaStream_t st) {
  if (head_dim != 128 && head_dim != 256) return VLLM_EUNSUPPORTED;
  if (n_splits < 1 || (n_splits > 1 && (!ws || causal))) return VLLM_EINVAL;
  const uint64_t D = (uint64_t)head_dim;
  CUtensorMap tq, tk, tv;
  if (make_tmap(&tq, q, (uint64_t)heads * D, Tq, batch, q_ts, q_bs, BQ)) return VLLM_EUNSUPPORTED;
  if (make_tmap(&tk, k, (uint64_t)kv_heads * D, Tk, batch, k_ts, k_bs, BKV)) return VLLM_EUNSUPPORTED;
  if (make_tmap(&tv, v, (uint64_t)kv_heads * D, Tk, batch, v_ts, v_bs, BKV)) return VLLM_EUNSUPPORTED;
  Args a;
  a.o = (__nv_bfloat16*)o; a.o_bs = o_bs; a.o_ts = o_ts; a.seqlens = seqlens; a.Tq = Tq; a.Tk = Tk;
  a.heads = heads; a.kv_heads = kv_heads; a.causal = causal; a.scale_log2 = scale * 1.4426950408889634f;
  a.key_mask = key_mask; a.km_vec = (key_mask && Tk % 16 == 0 && vllm_aligned(key_mask, 16)) ? 1 : 0;
  a.n_splits = n_splits; a.ws = ws;
  if (head_dim == 128) return key_mask ? launch_tc2<128, true>(tq, tk, tv, a, batch, st) : launch_tc2<128, false>(tq, tk, tv, a, batch, st);
  return key_mask ? launch_tc2<256, true>(tq, tk, tv, a, batch, st) : launch_tc2<256, false>(tq, tk, tv, a, batch, st);
}

int vllm_attention_tc2_d128(const void* q, const void* k, const void* v, void* o, int batch, int Tq, int Tk, int heads,
                            int kv_heads, long long q_bs, long long q_ts, long long k_bs, long long k_ts, long long v_bs,
                            long long v_ts, long long o_bs, long long o_ts, const int* seqlens, int causal, float scale,
                            cudaStream_t st) {
  return vllm_attention_tc2(q, k, v, o, batch, Tq, Tk, heads, kv_heads, 128, q_bs, q_ts, k_bs, k_ts, v_bs, v_ts, o_bs, o_ts,
                            seqlens, nullptr, causal, scale, 1, nullptr, st);
}
