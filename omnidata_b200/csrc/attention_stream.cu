// tcgen05 / TMEM fused attention above 640 tokens (d = 64): out = softmax(q k^T * scale) v.
//
// The arithmetic is that of attention_tc_kernel (attention_tc.cu), which serves <= 640 tokens with all K and V
// blocks of an (image, head) resident in shared memory.  Here K and V blocks stream through a ring of
// kStStages shared-memory stages instead, so the sequence length is bounded by nothing but memory:
//   * exact two-pass softmax: pass 1 computes S = Q K_j^T for every key block j (row maximum), pass 2
//     re-computes S, writes P = exp2(s*c - m*c) as bf16 into the UMMA operand layout and sums the unrounded
//     P in fp32; O += P V_j accumulates in TMEM and is never rescaled.  K is read twice per query tile, V once.
//   * a work unit is one (image, head, 128-query tile), numbered with the query tile fastest: the CTAs that
//     run at the same time work on the same few (image, head) pairs, whose K and V then come from L2.  Every
//     unit does the same arithmetic in the same order whatever else is in the batch.
//   * the TMA producer loads ring stages in exactly the order the MMA issuer consumes them (st_sched), and the
//     issuer releases a stage with a tcgen05.commit once the MMAs reading it are done.
// Warp roles, barriers and the TMEM plan (S triple-buffered in columns [0,384), O in [384,448)) are those of
// attention_tc_kernel:
//   warp 0      TMA producer (Q tile; K / V ring)
//   warp 1      tcgen05.mma issuer
//   warps 2-9   softmax (two threads per query row, 64 of the 128 columns of an S block each) + epilogue
#include "common.cuh"
#include "host_util.h"
#include "../../include/omnidata_b200.h"

namespace odb {

constexpr int kStBlk = 128;                   // queries per tile == keys per block
constexpr int kStStages = 8;                  // K / V ring depth
constexpr int kStTileBytes = kStBlk * 128;    // 128 rows x 64 bf16
constexpr int kStThreads = 320;
constexpr int kStSoftmaxThreads = 256;

constexpr int kStOffRing = 0;
constexpr int kStOffQ = kStStages * kStTileBytes;
constexpr int kStOffP = kStOffQ + 2 * kStTileBytes;
constexpr int kStOffX = kStOffP + 2 * kStTileBytes;          // fp32 exchange [2 halves][128 rows] (max, then sum)
constexpr int kStOffBar = kStOffX + 2 * 128 * 4;
constexpr int kStSmemBytes = kStOffBar + 512 + 1024;
static_assert(kStSmemBytes <= 232448, "streaming attention smem plan exceeds 227 KiB");

struct AttnStreamParams {
  CUtensorMap qkv_map;   // dims {64 d, 3*heads, tokens, batch}; box {64, 1, 128, 1}
  bf16* out;
  int tokens, heads, batch;
  float scale_log2e;
  unsigned long long* trace;   // diagnostics: per CTA kTraceSlots stamps; per unit i < 15 at 8 + 8 i:
                               // first S seen, maxima exchanged, first P block handed over, last P block handed
                               // over, sums exchanged, O ready, tile stored
};
#define ODB_STRACE(i, k)                                                                           \
  do {                                                                                             \
    if (p.trace != nullptr && (i) < 15u && warp == 2 && lane == 0) {                               \
      unsigned long long t_;                                                                       \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                                       \
      p.trace[static_cast<long long>(blockIdx.x) * kTraceSlots + 8 + 8 * static_cast<int>(i) + (k)] = t_; \
    }                                                                                              \
  } while (0)

ODB_DEVINL float fast_exp2_st(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// The t-th of the 3n ring loads of a query tile over n key blocks, in the MMA issuer's order: the S blocks of
// pass 1 (K_0 .. K_{n-1}) and the first two of pass 2, then for every key block j the pass-2 S block two ahead
// (K_{j+2}) followed by the PV product of block j (V_j).  Returns the qkv slot (1 = K, 2 = V) and sets *blk.
ODB_DEVINL int st_sched(int t, int n, int* blk) {
  const int lead = n + 2 < 2 * n ? n + 2 : 2 * n;
  if (t < lead) {
    *blk = t < n ? t : t - n;
    return 1;
  }
  t -= lead;
  const int pairs = n > 2 ? n - 2 : 0;
  if (t < 2 * pairs) {
    *blk = (t & 1) ? t >> 1 : (t >> 1) + 2;
    return (t & 1) ? 2 : 1;
  }
  *blk = pairs + (t - 2 * pairs);
  return 2;
}

ODB_DEVINL constexpr uint32_t umma_idesc_bf16_bmn_st(int m, int n) {
  return umma_idesc_bf16(m, n) | (1u << 16);     // MN-major B operand
}

__global__ void __launch_bounds__(kStThreads, 1) attention_stream_kernel(const __grid_constant__ AttnStreamParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen_base = smem_raw + (sbase - smem_u32(smem_raw));
  const uint32_t bar0 = sbase + kStOffBar;
  auto st_full = [&](int i) { return bar0 + 8u * i; };                        // kStStages
  auto st_empty = [&](int i) { return bar0 + 64u + 8u * i; };                 // kStStages
  auto q_full = [&](int i) { return bar0 + 128u + 8u * i; };
  auto q_empty = [&](int i) { return bar0 + 144u + 8u * i; };
  auto s_full = [&](int i) { return bar0 + 160u + 8u * i; };                  // 3 buffers
  auto s_empty = [&](int i) { return bar0 + 184u + 8u * i; };                 // 3 buffers
  const uint32_t p_full = bar0 + 208, p_empty = bar0 + 216, o_full = bar0 + 224, o_empty = bar0 + 232;
  const uint32_t tmem_slot = bar0 + 240;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gen_base + kStOffBar + 240);
  constexpr uint32_t kOCol = 3 * kStBlk;                       // first TMEM column of O
  float* xmax = reinterpret_cast<float*>(gen_base + kStOffX);  // row maxima, later the row sums (as attention_tc)
  float* xsum = xmax;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nblk = (p.tokens + kStBlk - 1) / kStBlk;     // key blocks == query tiles
  const int units = p.batch * p.heads * nblk;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kStStages; ++i) { mbar_init(st_full(i), 1); mbar_init(st_empty(i), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(q_full(i), 1); mbar_init(q_empty(i), 1); }
    for (int i = 0; i < 3; ++i) { mbar_init(s_full(i), 1); mbar_init(s_empty(i), 8); }
    mbar_init(p_full, kStSoftmaxThreads); mbar_init(p_empty, 1);
    mbar_init(o_full, 1); mbar_init(o_empty, 8);
    mbar_fence_init();
    tma_prefetch_desc(&p.qkv_map);
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  grid_dep_wait();
  grid_dep_launch();

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      uint32_t u_iter = 0, ring = 0;
      for (int unit = blockIdx.x; unit < units; unit += gridDim.x, ++u_iter) {
        const int bh = unit / nblk, qt = unit - bh * nblk;
        const int b = bh / p.heads, h = bh - b * p.heads;
        const int qb = u_iter & 1u;
        mbar_wait(q_empty(qb), ((u_iter >> 1) & 1u) ^ 1u);
        mbar_expect_tx(q_full(qb), kStTileBytes);
        tma_load_4d(sbase + kStOffQ + qb * kStTileBytes, &p.qkv_map, q_full(qb), 0, h, qt * kStBlk, b);
        for (int t = 0; t < 3 * nblk; ++t, ++ring) {
          int j;
          const int slot = st_sched(t, nblk, &j);
          const uint32_t st = ring % kStStages;
          mbar_wait(st_empty(st), ((ring / kStStages) & 1u) ^ 1u);
          mbar_expect_tx(st_full(st), kStTileBytes);
          tma_load_4d(sbase + kStOffRing + st * kStTileBytes, &p.qkv_map, st_full(st), 0, slot * p.heads + h,
                      j * kStBlk, b);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc_s = umma_idesc_bf16(kStBlk, kStBlk);
      constexpr uint32_t idesc_pv = umma_idesc_bf16_bmn_st(kStBlk, 64);
      uint32_t u_iter = 0, ring = 0, sb_iter = 0, p_iter = 0;
      // takes the next ring stage, which must hold what st_sched says it holds
      auto stage_in = [&]() {
        const uint32_t st = ring % kStStages;
        mbar_wait(st_full(st), (ring / kStStages) & 1u);
        return st;
      };
      auto stage_out = [&](uint32_t st) {
        umma_commit(st_empty(st));
        ++ring;
      };
      for (int unit = blockIdx.x; unit < units; unit += gridDim.x, ++u_iter) {
        const int qb = u_iter & 1u;
        mbar_wait(q_full(qb), (u_iter >> 1) & 1u);
        tc_fence_after();
        auto issue_s = [&]() {
          const uint32_t sbuf = sb_iter % 3u;
          const uint32_t st = stage_in();
          mbar_wait(s_empty(sbuf), ((sb_iter / 3u) & 1u) ^ 1u);
          tc_fence_after();
          const uint64_t adesc = umma_desc_sw128(sbase + kStOffQ + qb * kStTileBytes);
          const uint64_t bdesc = umma_desc_sw128(sbase + kStOffRing + st * kStTileBytes);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_ss(tmem_base + sbuf * kStBlk, adesc + 2u * k, bdesc + 2u * k, idesc_s, k != 0 ? 1u : 0u);
          umma_commit(s_full(sbuf));
          stage_out(st);
          ++sb_iter;
        };
        // S blocks in issue order: pass 1 then pass 2, up to two blocks ahead of the PV products
        int next_s = 0;
        auto pump = [&](int upto) {
          const int lim = upto < 2 * nblk ? upto : 2 * nblk;
          for (; next_s < lim; ++next_s) issue_s();
        };
        pump(nblk + 2);
        for (int j = 0; j < nblk; ++j) {
          pump(nblk + j + 3);
          const uint32_t st = stage_in();                       // V_j
          mbar_wait(p_full, p_iter & 1u);
          tc_fence_after();
          if (j == 0) {                                         // the epilogue has drained the previous O
            mbar_wait(o_empty, (u_iter & 1u) ^ 1u);
            tc_fence_after();
          }
#pragma unroll
          for (int kk = 0; kk < 8; ++kk) {
            // A = P (K-major, two 64-key k-blocks), B = V_j rows kk*16.. (MN-major: +16 rows = 2048 B)
            const uint64_t adesc = umma_desc_sw128(sbase + kStOffP + (kk >> 2) * kStTileBytes) + 2u * (kk & 3);
            const uint64_t bdesc = umma_desc_sw128(sbase + kStOffRing + st * kStTileBytes + kk * 2048);
            umma_bf16_ss(tmem_base + kOCol, adesc, bdesc, idesc_pv, (j | kk) != 0 ? 1u : 0u);
          }
          umma_commit(p_empty);
          stage_out(st);
          ++p_iter;
        }
        umma_commit(o_full);
        umma_commit(q_empty(qb));
      }
    }
  } else {
    // ------------------------------------------------------------------ softmax + epilogue
    const int quad = warp & 3;
    const int half = (warp - 2) >> 2;
    const int row = quad * 32 + lane;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    const float c = p.scale_log2e;
    uint32_t u_iter = 0, sb_iter = 0, p_iter = 0;
    for (int unit = blockIdx.x; unit < units; unit += gridDim.x, ++u_iter) {
      const int bh = unit / nblk, qt = unit - bh * nblk;
      const int b = bh / p.heads, h = bh - b * p.heads;
      // ---- pass 1: row maximum over all valid keys
      float mx = -INFINITY;
      for (int j = 0; j < nblk; ++j, ++sb_iter) {
        const uint32_t sbuf = sb_iter % 3u;
        mbar_wait(s_full(sbuf), (sb_iter / 3u) & 1u);
        tc_fence_after();
        if (j == 0) ODB_STRACE(u_iter, 0);
        uint32_t r[64];
        tmem_ld_32x32(t_lane + sbuf * kStBlk + half * 64, r);
        tmem_ld_32x32(t_lane + sbuf * kStBlk + half * 64 + 32, r + 32);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(s_empty(sbuf));
        const int key0 = j * kStBlk + half * 64;
        if (key0 + 64 <= p.tokens) {
#pragma unroll
          for (int i = 0; i < 64; ++i) mx = fmaxf(mx, __uint_as_float(r[i]));
        } else {
#pragma unroll
          for (int i = 0; i < 64; ++i)
            if (key0 + i < p.tokens) mx = fmaxf(mx, __uint_as_float(r[i]));
        }
      }
      xmax[half * 128 + row] = mx;
      named_bar_sync(1, kStSoftmaxThreads);
      const float m = fmaxf(xmax[row], xmax[128 + row]);
      const float mc = m * c;
      ODB_STRACE(u_iter, 1);
      // ---- pass 2: P = exp2(s*c - m*c) -> bf16 operand tile in smem, fp32 row sum
      float l = 0.f;
      for (int j = 0; j < nblk; ++j, ++sb_iter, ++p_iter) {
        const uint32_t sbuf = sb_iter % 3u;
        mbar_wait(s_full(sbuf), (sb_iter / 3u) & 1u);
        tc_fence_after();
        uint32_t r[64];
        tmem_ld_32x32(t_lane + sbuf * kStBlk + half * 64, r);
        tmem_ld_32x32(t_lane + sbuf * kStBlk + half * 64 + 32, r + 32);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(s_empty(sbuf));
        const int key0 = j * kStBlk + half * 64;
        uint32_t packed[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float p0 = fast_exp2_st(fmaf(__uint_as_float(r[2 * i]), c, -mc));
          float p1 = fast_exp2_st(fmaf(__uint_as_float(r[2 * i + 1]), c, -mc));
          if (key0 + 2 * i >= p.tokens) p0 = 0.f;
          if (key0 + 2 * i + 1 >= p.tokens) p1 = 0.f;
          l += p0 + p1;
          packed[i] = pack_bf16x2(p0, p1);
        }
        mbar_wait(p_empty, (p_iter & 1u) ^ 1u);     // PV of the previous block has consumed P
        const uint32_t prow = sbase + kStOffP + half * kStTileBytes + static_cast<uint32_t>(row) * 128u;
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          const uint32_t addr = prow + (static_cast<uint32_t>(jj ^ (row & 7)) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(packed[4 * jj]),
                       "r"(packed[4 * jj + 1]), "r"(packed[4 * jj + 2]), "r"(packed[4 * jj + 3])
                       : "memory");
        }
        fence_proxy_async_smem();
        mbar_arrive(p_full);
        if (j == 0) ODB_STRACE(u_iter, 2);
      }
      ODB_STRACE(u_iter, 3);
      xsum[half * 128 + row] = l;
      named_bar_sync(1, kStSoftmaxThreads);
      const float inv = 1.0f / (xsum[row] + xsum[128 + row]);
      ODB_STRACE(u_iter, 4);
      // ---- epilogue: O / l -> bf16 -> global (each thread: 32 of the 64 head dims of its row)
      mbar_wait(o_full, u_iter & 1u);
      tc_fence_after();
      ODB_STRACE(u_iter, 5);
      uint32_t o[32];
      tmem_ld_32x32(t_lane + kOCol + half * 32, o);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_empty);
      const int qrow = qt * kStBlk + row;
      if (qrow < p.tokens) {
        bf16* dst = p.out + ((long long)b * p.tokens + qrow) * (p.heads * 64) + h * 64 + half * 32;
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          uint4 v;
          v.x = pack_bf16x2(__uint_as_float(o[8 * jj + 0]) * inv, __uint_as_float(o[8 * jj + 1]) * inv);
          v.y = pack_bf16x2(__uint_as_float(o[8 * jj + 2]) * inv, __uint_as_float(o[8 * jj + 3]) * inv);
          v.z = pack_bf16x2(__uint_as_float(o[8 * jj + 4]) * inv, __uint_as_float(o[8 * jj + 5]) * inv);
          v.w = pack_bf16x2(__uint_as_float(o[8 * jj + 6]) * inv, __uint_as_float(o[8 * jj + 7]) * inv);
          *reinterpret_cast<uint4*>(dst + jj * 8) = v;
        }
      }
      ODB_STRACE(u_iter, 6);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// called by odb_attention above 640 tokens (arguments checked there)
int attention_stream(const void* qkv, void* out, int b, int tokens, int heads, float scale, cudaStream_t stream) {
  const long long units = (long long)b * heads * ((tokens + kStBlk - 1) / kStBlk);
  if (units > 0x7fffffffLL) return fail(ODB_ERR_UNSUPPORTED, "attention: too many (image, head, query tile) units");
  AttnStreamParams p;
  memset(&p, 0, sizeof(p));
  {
    cuuint64_t dims[4] = {64, (cuuint64_t)(3 * heads), (cuuint64_t)tokens, (cuuint64_t)b};
    cuuint64_t strides[3] = {128, (cuuint64_t)(3 * heads) * 128, (cuuint64_t)tokens * (3 * heads) * 128};
    cuuint32_t box[4] = {64, 1, (cuuint32_t)kStBlk, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    int rc = encode_tiled(&p.qkv_map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(qkv), dims,
                          strides, box, estr, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  p.out = static_cast<bf16*>(out);
  p.tokens = tokens; p.heads = heads; p.batch = b;
  p.scale_log2e = scale * 1.4426950408889634f;
  p.trace = debug_trace();
  static bool configured[kMaxDevices] = {};
  const int dev_ = current_device();
  if (!configured[dev_]) {
    cudaError_t e = cudaFuncSetAttribute(attention_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         kStSmemBytes);
    if (e != cudaSuccess) return fail_cuda(e, "attention_stream: cudaFuncSetAttribute");
    configured[dev_] = true;
  }
  const int grid = units < num_sms() ? (int)units : num_sms();
  cudaError_t le = launch_pdl(attention_stream_kernel, dim3(grid), dim3(kStThreads), kStSmemBytes, stream, p);
  count_launch();
  if (le != cudaSuccess) return fail_cuda(le, "attention_stream: launch");
  return check_launch("attention_stream");
}

}  // namespace odb
