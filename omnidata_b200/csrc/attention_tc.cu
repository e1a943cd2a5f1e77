// tcgen05 / TMEM fused attention for the ViT-B/16 blocks of DPT-Hybrid (<= 640 tokens, d = 64):
//   out = softmax(q k^T * scale) v        (timm Attention.forward; block loop at M/vit.py:150-151)
//
// One persistent CTA per SM; a work unit is one (image, head).  K and V of the unit (5 blocks of
// 128 keys x 64 d each) are TMA-loaded once into shared memory and stay resident; the 128-query
// tiles of the unit stream through a double-buffered Q slot.
//   warp 0      TMA producer (K, V blocks; Q tiles)
//   warp 1      tcgen05.mma issuer:  S = Q K_j^T  (M=128, N=128, K=64, both operands K-major)
//                                    O += P_j V_j (M=128, N=64, K=128, V is the MN-major B operand)
//   warps 2-9   softmax: two threads per query row (each owns 64 of the 128 columns of an S block)
// Softmax is two-pass and exact: pass 1 reads the five S blocks from TMEM for the row maximum,
// pass 2 re-computes them (the tensor pipe is far from saturated), writes P = exp2(s*c - m*c) as
// bf16 straight into the K-major UMMA operand layout in shared memory and accumulates the fp32 row
// sum of the unrounded P.  O therefore never needs rescaling and lives in TMEM until the epilogue.
// TMEM: S triple-buffered in columns [0,384) (the MMA warp runs up to two S blocks ahead of the
// softmax warps, which hides the commit -> mbarrier -> tcgen05.ld hand-off latency), O in [384,448).
#include "common.cuh"
#include "host_util.h"
#include "../../include/omnidata_b200.h"

namespace odb {

constexpr int kTcBlk = 128;         // queries per tile == keys per block
constexpr int kTcMaxBlocks = 5;     // 640 keys
constexpr int kTcTileBytes = kTcBlk * 128;   // 128 rows x 64 bf16
constexpr int kTcThreads = 320;
constexpr int kTcSoftmaxThreads = 256;

constexpr int kTcOffK = 0;
constexpr int kTcOffV = kTcMaxBlocks * kTcTileBytes;
constexpr int kTcOffQ = 2 * kTcMaxBlocks * kTcTileBytes;
constexpr int kTcOffP = kTcOffQ + 2 * kTcTileBytes;
constexpr int kTcOffX = kTcOffP + 2 * kTcTileBytes;          // fp32 exchange [2 halves][128 rows] (max, then sum)
constexpr int kTcOffBar = kTcOffX + 2 * 128 * 4;
constexpr int kTcSmemBytes = kTcOffBar + 256 + 1024;
static_assert(kTcSmemBytes <= 232448, "attention smem plan exceeds 227 KiB");

struct AttnTcParams {
  CUtensorMap qkv_map;   // dims {64 d, 3*heads, tokens, batch}; box {64, 1, 128, 1}
  bf16* out;
  float* lse;            // optional [batch][heads][tokens]: log2 sum_j exp2(s_j c) per query row (training)
  int tokens, heads, batch;
  float scale_log2e;
  unsigned long long* trace;   // diagnostics: per CTA kTraceSlots stamps; per q tile i < 8 at 8 + 12 i:
                               // first S seen, maxima exchanged, P block 0..4 handed over, sums exchanged, O ready, tile stored
};
#define ODB_ATRACE(i, k)                                                                           \
  do {                                                                                             \
    if (p.trace != nullptr && (i) < 8u && warp == 2 && lane == 0) {                                \
      unsigned long long t_;                                                                       \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                                       \
      p.trace[static_cast<long long>(blockIdx.x) * kTraceSlots + 8 + 12 * static_cast<int>(i) + (k)] = t_; \
    }                                                                                              \
  } while (0)

ODB_DEVINL float fast_exp2_tc(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// instruction descriptor with an MN-major B operand (bit 16)
ODB_DEVINL constexpr uint32_t umma_idesc_bf16_bmn(int m, int n) {
  return umma_idesc_bf16(m, n) | (1u << 16);
}

__global__ void __launch_bounds__(kTcThreads, 1) attention_tc_kernel(const __grid_constant__ AttnTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen_base = smem_raw + (sbase - smem_u32(smem_raw));
  const uint32_t bar0 = sbase + kTcOffBar;
  const uint32_t kv_full = bar0, kv_empty = bar0 + 8;
  auto q_full = [&](int i) { return bar0 + 16u + 8u * i; };
  auto q_empty = [&](int i) { return bar0 + 32u + 8u * i; };
  auto s_full = [&](int i) { return bar0 + 48u + 8u * i; };    // 3 buffers
  auto s_empty = [&](int i) { return bar0 + 72u + 8u * i; };   // 3 buffers
  const uint32_t p_full = bar0 + 96, p_empty = bar0 + 104, o_full = bar0 + 112, o_empty = bar0 + 120;
  const uint32_t tmem_slot = bar0 + 128;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gen_base + kTcOffBar + 128);
  constexpr uint32_t kOCol = 3 * kTcBlk;                       // first TMEM column of O
  // K and V arrive block by block (own barrier each): the first S block of a unit starts after 16 KiB
  // instead of after the whole 160 KiB, the rest of the fetch hides behind pass 1
  auto k_full = [&](int j) { return bar0 + 136u + 8u * j; };
  auto v_full = [&](int j) { return bar0 + 176u + 8u * j; };
  // one exchange array serves the row maxima and later the row sums: a thread can only reach its
  // row-sum write after every thread has arrived on p_full for block 0, i.e. after it read the maxima
  float* xmax = reinterpret_cast<float*>(gen_base + kTcOffX);
  float* xsum = xmax;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nblk = (p.tokens + kTcBlk - 1) / kTcBlk;     // key blocks == query tiles
  const int units = p.batch * p.heads;

  if (threadIdx.x == 0) {
    mbar_init(kv_full, 1); mbar_init(kv_empty, 1);
    for (int j = 0; j < kTcMaxBlocks; ++j) { mbar_init(k_full(j), 1); mbar_init(v_full(j), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(q_full(i), 1); mbar_init(q_empty(i), 1); }
    for (int i = 0; i < 3; ++i) { mbar_init(s_full(i), 1); mbar_init(s_empty(i), 8); }
    mbar_init(p_full, kTcSoftmaxThreads); mbar_init(p_empty, 1);
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
      uint32_t u_iter = 0, qt_iter = 0;
      for (int unit = blockIdx.x; unit < units; unit += gridDim.x, ++u_iter) {
        const int b = unit / p.heads, h = unit % p.heads;
        mbar_wait(kv_empty, (u_iter & 1u) ^ 1u);
        for (int j = 0; j < nblk; ++j) {
          mbar_expect_tx(k_full(j), kTcTileBytes);
          tma_load_4d(sbase + kTcOffK + j * kTcTileBytes, &p.qkv_map, k_full(j), 0, p.heads + h, j * kTcBlk, b);
        }
        for (int j = 0; j < nblk; ++j) {
          mbar_expect_tx(v_full(j), kTcTileBytes);
          tma_load_4d(sbase + kTcOffV + j * kTcTileBytes, &p.qkv_map, v_full(j), 0, 2 * p.heads + h, j * kTcBlk, b);
        }
        for (int qt = 0; qt < nblk; ++qt, ++qt_iter) {
          const int qb = qt_iter & 1u;
          mbar_wait(q_empty(qb), ((qt_iter >> 1) & 1u) ^ 1u);
          mbar_expect_tx(q_full(qb), kTcTileBytes);
          tma_load_4d(sbase + kTcOffQ + qb * kTcTileBytes, &p.qkv_map, q_full(qb), 0, h, qt * kTcBlk, b);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc_s = umma_idesc_bf16(kTcBlk, kTcBlk);
      constexpr uint32_t idesc_pv = umma_idesc_bf16_bmn(kTcBlk, 64);
      uint32_t u_iter = 0, qt_iter = 0, sb_iter = 0, p_iter = 0;
      auto issue_s = [&](int j, int qb) {
        const uint32_t sbuf = sb_iter % 3u;
        mbar_wait(k_full(j), u_iter & 1u);                      // K block j of this unit has landed
        mbar_wait(s_empty(sbuf), ((sb_iter / 3u) & 1u) ^ 1u);
        tc_fence_after();
        const uint64_t adesc = umma_desc_sw128(sbase + kTcOffQ + qb * kTcTileBytes);
        const uint64_t bdesc = umma_desc_sw128(sbase + kTcOffK + j * kTcTileBytes);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16_ss(tmem_base + sbuf * kTcBlk, adesc + 2u * k, bdesc + 2u * k, idesc_s, k != 0 ? 1u : 0u);
        umma_commit(s_full(sbuf));
        ++sb_iter;
      };
      for (int unit = blockIdx.x; unit < units; unit += gridDim.x, ++u_iter) {
        for (int qt = 0; qt < nblk; ++qt, ++qt_iter) {
          const int qb = qt_iter & 1u;
          mbar_wait(q_full(qb), (qt_iter >> 1) & 1u);
          tc_fence_after();
          // S blocks of this tile in issue order: pass 1 (row maxima) then pass 2 (probabilities);
          // the issuer keeps up to two blocks ahead of what the softmax warps / the PV MMAs need
          int next_s = 0;
          auto pump = [&](int upto) {
            const int lim = upto < 2 * nblk ? upto : 2 * nblk;
            for (; next_s < lim; ++next_s) issue_s(next_s < nblk ? next_s : next_s - nblk, qb);
          };
          pump(nblk + 2);
          for (int j = 0; j < nblk; ++j) {
            pump(nblk + j + 3);
            mbar_wait(v_full(j), u_iter & 1u);                    // V block j of this unit has landed
            mbar_wait(p_full, p_iter & 1u);
            tc_fence_after();
            if (j == 0) {                                         // the epilogue has drained the previous O
              mbar_wait(o_empty, (qt_iter & 1u) ^ 1u);
              tc_fence_after();
            }
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) {
              // A = P (K-major, two 64-key k-blocks), B = V_j rows kk*16.. (MN-major: +16 rows = 2048 B)
              const uint64_t adesc =
                  umma_desc_sw128(sbase + kTcOffP + (kk >> 2) * kTcTileBytes) + 2u * (kk & 3);
              const uint64_t bdesc = umma_desc_sw128(sbase + kTcOffV + j * kTcTileBytes + kk * 2048);
              umma_bf16_ss(tmem_base + kOCol, adesc, bdesc, idesc_pv, (j | kk) != 0 ? 1u : 0u);
            }
            umma_commit(p_empty);
            ++p_iter;
          }
          umma_commit(o_full);
          umma_commit(q_empty(qb));
        }
        umma_commit(kv_empty);
      }
    }
  } else {
    // ------------------------------------------------------------------ softmax + epilogue
    const int quad = warp & 3;
    const int half = (warp - 2) >> 2;
    const int row = quad * 32 + lane;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    const float c = p.scale_log2e;
    uint32_t qt_iter = 0, sb_iter = 0, p_iter = 0;
    for (int unit = blockIdx.x; unit < units; unit += gridDim.x) {
      const int b = unit / p.heads, h = unit % p.heads;
      for (int qt = 0; qt < nblk; ++qt, ++qt_iter) {
        // ---- pass 1: row maximum over all valid keys
        float mx = -INFINITY;
        for (int j = 0; j < nblk; ++j, ++sb_iter) {
          const uint32_t sbuf = sb_iter % 3u;
          mbar_wait(s_full(sbuf), (sb_iter / 3u) & 1u);
          tc_fence_after();
          if (j == 0) ODB_ATRACE(qt_iter, 0);
          uint32_t r[64];
          tmem_ld_32x32(t_lane + sbuf * kTcBlk + half * 64, r);
          tmem_ld_32x32(t_lane + sbuf * kTcBlk + half * 64 + 32, r + 32);
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(s_empty(sbuf));
          const int key0 = j * kTcBlk + half * 64;
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
        named_bar_sync(1, kTcSoftmaxThreads);
        const float m = fmaxf(xmax[row], xmax[128 + row]);
        const float mc = m * c;
        ODB_ATRACE(qt_iter, 1);
        // ---- pass 2: P = exp2(s*c - m*c) -> bf16 operand tile in smem, fp32 row sum
        float l = 0.f;
        for (int j = 0; j < nblk; ++j, ++sb_iter, ++p_iter) {
          const uint32_t sbuf = sb_iter % 3u;
          mbar_wait(s_full(sbuf), (sb_iter / 3u) & 1u);
          tc_fence_after();
          uint32_t r[64];
          tmem_ld_32x32(t_lane + sbuf * kTcBlk + half * 64, r);
          tmem_ld_32x32(t_lane + sbuf * kTcBlk + half * 64 + 32, r + 32);
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(s_empty(sbuf));
          const int key0 = j * kTcBlk + half * 64;
          uint32_t packed[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            float p0 = fast_exp2_tc(fmaf(__uint_as_float(r[2 * i]), c, -mc));
            float p1 = fast_exp2_tc(fmaf(__uint_as_float(r[2 * i + 1]), c, -mc));
            if (key0 + 2 * i >= p.tokens) p0 = 0.f;
            if (key0 + 2 * i + 1 >= p.tokens) p1 = 0.f;
            l += p0 + p1;
            packed[i] = pack_bf16x2(p0, p1);
          }
          mbar_wait(p_empty, (p_iter & 1u) ^ 1u);     // PV of the previous block has consumed P
          const uint32_t prow = sbase + kTcOffP + half * kTcTileBytes + static_cast<uint32_t>(row) * 128u;
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) {
            const uint32_t addr = prow + (static_cast<uint32_t>(jj ^ (row & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(packed[4 * jj]),
                         "r"(packed[4 * jj + 1]), "r"(packed[4 * jj + 2]), "r"(packed[4 * jj + 3])
                         : "memory");
          }
          fence_proxy_async_smem();
          mbar_arrive(p_full);
          ODB_ATRACE(qt_iter, 2 + j);
        }
        xsum[half * 128 + row] = l;
        named_bar_sync(1, kTcSoftmaxThreads);
        const float lsum = xsum[row] + xsum[128 + row];
        const float inv = 1.0f / lsum;
        if (p.lse != nullptr && half == 0 && qt * kTcBlk + row < p.tokens)
          p.lse[((long long)b * p.heads + h) * p.tokens + qt * kTcBlk + row] = mc + log2f(lsum);
        ODB_ATRACE(qt_iter, 7);
        // ---- epilogue: O / l -> bf16 -> global (each thread: 32 of the 64 head dims of its row)
        mbar_wait(o_full, qt_iter & 1u);
        tc_fence_after();
        ODB_ATRACE(qt_iter, 8);
        uint32_t o[32];
        tmem_ld_32x32(t_lane + kOCol + half * 32, o);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(o_empty);
        const int qrow = qt * kTcBlk + row;
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
        ODB_ATRACE(qt_iter, 9);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace odb

namespace odb { int attention_stream(const void* qkv, void* out, int b, int tokens, int heads, float scale,
                                     cudaStream_t stream); }   // attention_stream.cu

using namespace odb;

extern "C" int odb_attention(const void* qkv, void* out, float* lse, int32_t b, int32_t tokens, int32_t heads,
                             float scale, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (!qkv || !out || b < 1 || heads < 1 || tokens < 1)
    return fail(ODB_ERR_INVALID, "attention: bad argument");
  if (reinterpret_cast<uintptr_t>(qkv) & 15u) return fail(ODB_ERR_INVALID, "attention: qkv must be 16-byte aligned");
  if (tokens > kTcBlk * kTcMaxBlocks) {
    // K and V no longer fit in shared memory: they stream through a ring of stages instead
    if (lse != nullptr) return fail(ODB_ERR_UNSUPPORTED, "attention: lse is only written up to 640 tokens");
    return attention_stream(qkv, out, b, tokens, heads, scale, stream);
  }
  AttnTcParams p;
  memset(&p, 0, sizeof(p));
  {
    cuuint64_t dims[4] = {64, (cuuint64_t)(3 * heads), (cuuint64_t)tokens, (cuuint64_t)b};
    cuuint64_t strides[3] = {128, (cuuint64_t)(3 * heads) * 128, (cuuint64_t)tokens * (3 * heads) * 128};
    cuuint32_t box[4] = {64, 1, (cuuint32_t)kTcBlk, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    int rc = encode_tiled(&p.qkv_map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(qkv), dims,
                          strides, box, estr, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  p.out = static_cast<bf16*>(out);
  p.lse = lse;
  p.tokens = tokens; p.heads = heads; p.batch = b;
  p.scale_log2e = scale * 1.4426950408889634f;
  p.trace = debug_trace();
  static bool configured[kMaxDevices] = {};
  const int dev_ = current_device();
  if (!configured[dev_]) {
    cudaError_t e = cudaFuncSetAttribute(attention_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         kTcSmemBytes);
    if (e != cudaSuccess) return fail_cuda(e, "attention: cudaFuncSetAttribute");
    configured[dev_] = true;
  }
  const int units = b * heads;
  const int grid = units < num_sms() ? units : num_sms();
  cudaError_t le = launch_pdl(attention_tc_kernel, dim3(grid), dim3(kTcThreads), kTcSmemBytes, stream, p);
  count_launch();
  if (le != cudaSuccess) return fail_cuda(le, "attention_tc: launch");
  return check_launch("attention_tc");
}
