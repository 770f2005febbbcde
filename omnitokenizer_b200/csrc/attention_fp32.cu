// Exact-fp32 attention cores (CUDA-core FFMA) for the three token topologies of the path:
//   spatial  : full attention over the N = h*w tokens of one frame          (attention.py:451)
//   window   : 8x8 windows of the (h,w) grid + relative position bias       (attention.py:275-286)
//   temporal : causal attention over the T' frames of one pixel             (attention.py:451, is_causal)
// All three read q/k/v straight out of the canonical X[B][T'][N][*] projections through an index
// map -- the reference's rearrange copies (omnitokenizer.py:891,902,907) never materialise.
#include "omt_common.cuh"

namespace omt {

constexpr int AQ = 64;    // queries per CTA
constexpr int AK = 64;    // keys per chunk
constexpr int AD = 64;    // head dim

// float offset of 16-byte chunk c of row r in a [64][64] tile, XOR-swizzled so that the 4x4
// register-blocked reads (rows 4*lane_x + jj, same chunk) hit 8 distinct bank groups.
__device__ __forceinline__ int sw(int r, int c) { return r * 64 + ((c ^ ((r >> 2) & 7)) << 2); }

struct AttnArgs {
  const float* q; int ldq;
  const float* k; int ldk;
  const float* v; int ldv;
  float* o; int ldo;
  uint16_t* o_hi; uint16_t* o_lo;   // optional fp16 hi / bf16 lo operand planes instead of o (ld = ldo)
  const float* bias;   // window: [heads][64][64]
  int N;               // tokens per frame
  int h, w, ws;        // window mode
  float scale;
};

template <bool WINDOW>
__device__ __forceinline__ long long token_row(const AttnArgs& a, int seq, int i) {
  if (!WINDOW) return (long long)seq * a.N + i;
  const int nwx = a.w / a.ws;
  const int nW = (a.h / a.ws) * nwx;
  const int frame = seq / nW, win = seq % nW;
  const int wy = win / nwx, wx = win % nwx;
  const int sy = i / a.ws, sx = i % a.ws;
  return (long long)frame * a.N + (wy * a.ws + sy) * a.w + wx * a.ws + sx;
}

template <bool WINDOW>
__global__ void __launch_bounds__(256, 2) attn_flash_kernel(const AttnArgs a) {
  pdl_sync();
  extern __shared__ __align__(16) float smem[];
  float* Qs = smem;                 // [64][64] swizzled, pre-scaled
  float* Ks = smem + 4096;          // [64][64] swizzled
  float* Vs = smem + 8192;          // [64][64] plain
  float* Ps = smem + 12288;         // [64][64] swizzled
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int qt = WINDOW ? 0 : blockIdx.x, head = blockIdx.y;
  const int seq = WINDOW ? blockIdx.x : blockIdx.z;   // window sequences can exceed gridDim.z
  const int seq_len = WINDOW ? 64 : a.N;
  const int lc = tid & 15, lr = tid >> 4;   // loader: chunk, row (+16*it)

  // Q tile
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int r = lr + it * 16;
    const long long row = token_row<WINDOW>(a, seq, qt * AQ + r);
    float4 v = *reinterpret_cast<const float4*>(a.q + row * a.ldq + head * AD + lc * 4);
    v.x *= a.scale; v.y *= a.scale; v.z *= a.scale; v.w *= a.scale;
    *reinterpret_cast<float4*>(Qs + sw(r, lc)) = v;
  }

  float o[4][4];
  float mrow[4], lrow[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    mrow[i] = -INFINITY; lrow[i] = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) o[i][j] = 0.f;
  }

  float4 pk[4], pv[4];
  auto prefetch = [&](int kc) {
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int r = lr + it * 16;
      const long long row = token_row<WINDOW>(a, seq, kc * AK + r);
      pk[it] = *reinterpret_cast<const float4*>(a.k + row * a.ldk + head * AD + lc * 4);
      pv[it] = *reinterpret_cast<const float4*>(a.v + row * a.ldv + head * AD + lc * 4);
    }
  };
  const int nkc = seq_len / AK;
  prefetch(0);
  for (int kc = 0; kc < nkc; ++kc) {
    __syncthreads();     // previous chunk's readers of Ks/Vs/Ps are done (and Qs is visible)
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int r = lr + it * 16;
      *reinterpret_cast<float4*>(Ks + sw(r, lc)) = pk[it];
      *reinterpret_cast<float4*>(Vs + r * 64 + lc * 4) = pv[it];
    }
    __syncthreads();
    if (kc + 1 < nkc) prefetch(kc + 1);

    // S = (scale * Q) K^T, 4x4 per thread
    float s[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) s[i][j] = 0.f;
#pragma unroll 4
    for (int c = 0; c < 16; ++c) {
      float4 qf[4], kf[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) qf[i] = *reinterpret_cast<const float4*>(Qs + sw(ty * 4 + i, c));
#pragma unroll
      for (int j = 0; j < 4; ++j) kf[j] = *reinterpret_cast<const float4*>(Ks + sw(tx * 4 + j, c));
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          s[i][j] = fmaf(qf[i].x, kf[j].x, s[i][j]);
          s[i][j] = fmaf(qf[i].y, kf[j].y, s[i][j]);
          s[i][j] = fmaf(qf[i].z, kf[j].z, s[i][j]);
          s[i][j] = fmaf(qf[i].w, kf[j].w, s[i][j]);
        }
    }
    if (WINDOW) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 b = *reinterpret_cast<const float4*>(a.bias + ((size_t)head * 64 + ty * 4 + i) * 64 + tx * 4);
        s[i][0] += b.x; s[i][1] += b.y; s[i][2] += b.z; s[i][3] += b.w;
      }
    }
    // online softmax; a row is shared by the 16 lanes with equal ty (a half warp)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float mx = fmaxf(fmaxf(s[i][0], s[i][1]), fmaxf(s[i][2], s[i][3]));
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
      const float mnew = fmaxf(mrow[i], mx);
      const float corr = expf(mrow[i] - mnew);
      float ps = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) { s[i][j] = expf(s[i][j] - mnew); ps += s[i][j]; }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) ps += __shfl_xor_sync(0xffffffffu, ps, off);
      lrow[i] = lrow[i] * corr + ps;
      mrow[i] = mnew;
#pragma unroll
      for (int j = 0; j < 4; ++j) o[i][j] *= corr;
      *reinterpret_cast<float4*>(Ps + sw(ty * 4 + i, tx)) = make_float4(s[i][0], s[i][1], s[i][2], s[i][3]);
    }
    __syncthreads();
    // O += P V
#pragma unroll 4
    for (int jc = 0; jc < 16; ++jc) {
      float4 pf[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) pf[i] = *reinterpret_cast<const float4*>(Ps + sw(ty * 4 + i, jc));
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        const float4 vf = *reinterpret_cast<const float4*>(Vs + (jc * 4 + jj) * 64 + tx * 4);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float p = (jj == 0) ? pf[i].x : (jj == 1) ? pf[i].y : (jj == 2) ? pf[i].z : pf[i].w;
          o[i][0] = fmaf(p, vf.x, o[i][0]);
          o[i][1] = fmaf(p, vf.y, o[i][1]);
          o[i][2] = fmaf(p, vf.z, o[i][2]);
          o[i][3] = fmaf(p, vf.w, o[i][3]);
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long row = token_row<WINDOW>(a, seq, qt * AQ + ty * 4 + i);
    const float inv = 1.0f / lrow[i];
    const float4 ov = make_float4(o[i][0] * inv, o[i][1] * inv, o[i][2] * inv, o[i][3] * inv);
    if (a.o_hi != nullptr) store_split4(a.o_hi, a.o_lo, (size_t)(row * a.ldo + head * AD + tx * 4), ov);
    else *reinterpret_cast<float4*>(a.o + row * a.ldo + head * AD + tx * 4) = ov;
  }
}

// Temporal attention: one warp per (b, n, head); lane l owns dims (2l, 2l+1); K/V of the
// whole (short) sequence stay in registers.
template <int T>
__global__ void __launch_bounds__(256) attn_temporal_kernel(const float* __restrict__ q, int ldq,
                                                            const float* __restrict__ k, int ldk,
                                                            const float* __restrict__ v, int ldv,
                                                            float* __restrict__ o, uint16_t* __restrict__ o_hi,
                                                            uint16_t* __restrict__ o_lo, int ldo, int B,
                                                            int N, int heads, float scale, int causal) {
  pdl_sync();
  const int lane = threadIdx.x & 31;
  const long long wid = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const long long total = (long long)B * N * heads;
  if (wid >= total) return;
  const int head = (int)(wid % heads);
  const long long bn = wid / heads;
  const int n = (int)(bn % N);
  const int b = (int)(bn / N);
  const size_t col = (size_t)head * 64 + 2 * lane;
  float2 kr[T], vr[T], qr[T];           // all 3 T loads of the sequence are in flight before the first use
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const size_t row = ((size_t)b * T + t) * N + n;
    kr[t] = *reinterpret_cast<const float2*>(k + row * ldk + col);
    vr[t] = *reinterpret_cast<const float2*>(v + row * ldv + col);
    qr[t] = *reinterpret_cast<const float2*>(q + row * ldq + col);
  }
#pragma unroll
  for (int i = 0; i < T; ++i) {
    const size_t row = ((size_t)b * T + i) * N + n;
    const float2 qv = qr[i];
    float s[T];
#pragma unroll
    for (int j = 0; j < T; ++j) s[j] = qv.x * kr[j].x + qv.y * kr[j].y;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1)
#pragma unroll
      for (int j = 0; j < T; ++j) s[j] += __shfl_xor_sync(0xffffffffu, s[j], off);
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < T; ++j) {
      s[j] *= scale;
      if (!causal || j <= i) mx = fmaxf(mx, s[j]);
    }
    float den = 0.f, ox = 0.f, oy = 0.f;
#pragma unroll
    for (int j = 0; j < T; ++j) {
      if (!causal || j <= i) {
        const float p = expf(s[j] - mx);
        den += p;
        ox = fmaf(p, vr[j].x, ox);
        oy = fmaf(p, vr[j].y, oy);
      }
    }
    const float2 ov = make_float2(ox / den, oy / den);
    if (o_hi != nullptr) store_split2(o_hi, o_lo, row * ldo + col, ov);
    else *reinterpret_cast<float2*>(o + row * ldo + col) = ov;
  }
}

template <int T>
static int launch_temporal(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv,
                           float* o, uint16_t* o_hi, uint16_t* o_lo, int ldo, int B, int N, int heads, float scale, int causal,
                           cudaStream_t st) {
  const long long warps = (long long)B * N * heads;
  const unsigned blocks = (unsigned)((warps + 7) / 8);
  OMT_CUDA(launch_k(attn_temporal_kernel<T>, dim3(blocks), dim3(256), 0, st, q, ldq, k, ldk, v, ldv, o, o_hi, o_lo, ldo, B, N, heads, scale, causal));
  OMT_LAUNCH_CHECK();
  return OMT_OK;
}

// Temporal attention for T' > 17: one warp per (b, n, head) and tile of 32 query frames, lane = query frame.  q and the
// O accumulator stay in registers; K / V stream through shared memory in chunks of TK frames (cp.async, double-buffered
// per warp, so no block barrier), and every lane reads the same k_j / v_j (a broadcast: no bank conflicts, no shuffles).
// Online softmax per lane with one max update and one O rescale per chunk.  The arithmetic of an output element depends
// on T', its frame and the causal flag only -- never on B, N or the grid -- so a batch shard reproduces the full batch.
constexpr int TQ = 32;    // query frames per warp (one per lane)
constexpr int TK = 16;    // key frames per chunk
constexpr int TW = 4;     // warps (consecutive b*N + n sequences of one head) per CTA
constexpr int T_WARP_FLOATS = 2 * 2 * TK * AD;          // [buffer][K | V][TK][64] per warp: 16 KiB
constexpr int T_SMEM = TW * T_WARP_FLOATS * 4;

__device__ __forceinline__ void cp_async16(float* dst, const float* src, bool ok) {    // zero-fill when !ok
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src),
               "r"(ok ? 16 : 0) : "memory");
}

__global__ void __launch_bounds__(TW * 32) attn_temporal_long_kernel(const float* __restrict__ q, int ldq,
                                                                      const float* __restrict__ k, int ldk,
                                                                      const float* __restrict__ v, int ldv,
                                                                      float* __restrict__ o, uint16_t* __restrict__ o_hi,
                                                                      uint16_t* __restrict__ o_lo, int ldo, int B, int T,
                                                                      int N, float scale, int causal) {
  pdl_sync();
  extern __shared__ __align__(16) float tsm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long seq = (long long)blockIdx.x * TW + warp;      // b * N + n
  if (seq >= (long long)B * N) return;                          // ragged B*N: warps never meet at a block barrier
  const int b = (int)(seq / N), n = (int)(seq % N);
  const size_t row0 = (size_t)b * T * N + n;                    // canonical row of frame t: row0 + t * N
  const size_t col = (size_t)blockIdx.y * AD;
  const int q0 = blockIdx.z * TQ, i = q0 + lane;
  const int kend = causal ? min(T, q0 + TQ) : T;                // a causal tile stops at its last query's key
  const int nch = (kend + TK - 1) / TK;
  float* const sm = tsm + warp * T_WARP_FLOATS;

  // chunk c -> buffer c & 1: TK rows of 256 bytes each for K and V, 16 consecutive lanes per row; frames >= kend read as 0
  auto load = [&](int c) {
    float* dst = sm + (c & 1) * (2 * TK * AD);
#pragma unroll
    for (int it = 0; it < TK * 16 / 32; ++it) {
      const int idx = it * 32 + lane, r = idx >> 4, sg = (idx & 15) * 4;
      const int t = c * TK + r;
      const size_t row = row0 + (size_t)(t < kend ? t : 0) * N;
      cp_async16(dst + r * AD + sg, k + row * ldk + col + sg, t < kend);
      cp_async16(dst + TK * AD + r * AD + sg, v + row * ldv + col + sg, t < kend);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  load(0);

  float qr[AD], acc[AD];
  {
    const float* qp = q + (row0 + (size_t)(i < T ? i : 0) * N) * ldq + col;
#pragma unroll
    for (int d = 0; d < AD; d += 4) {
      const float4 x = *reinterpret_cast<const float4*>(qp + d);
      qr[d] = x.x; qr[d + 1] = x.y; qr[d + 2] = x.z; qr[d + 3] = x.w;
      acc[d] = acc[d + 1] = acc[d + 2] = acc[d + 3] = 0.f;
    }
  }
  float m = -INFINITY, l = 0.f;
  for (int c = 0; c < nch; ++c) {
    if (c + 1 < nch) {       // buffer (c + 1) & 1 was released by the __syncwarp that ended chunk c - 1
      load(c + 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncwarp();
    const float* Kc = sm + (c & 1) * (2 * TK * AD);
    const float* Vc = Kc + TK * AD;
    float s[TK];
#pragma unroll
    for (int j = 0; j < TK; ++j) s[j] = 0.f;
#pragma unroll
    for (int d = 0; d < AD; d += 4)
#pragma unroll
      for (int j = 0; j < TK; ++j) {
        const float4 kf = *reinterpret_cast<const float4*>(Kc + j * AD + d);
        s[j] = fmaf(qr[d], kf.x, s[j]);
        s[j] = fmaf(qr[d + 1], kf.y, s[j]);
        s[j] = fmaf(qr[d + 2], kf.z, s[j]);
        s[j] = fmaf(qr[d + 3], kf.w, s[j]);
      }
    // key 0 is in chunk 0 and visible to every query, so mc is finite from the first chunk on; a later chunk that is
    // fully masked for this lane leaves corr = 1 and adds p = 0
    float mc = m;
#pragma unroll
    for (int j = 0; j < TK; ++j) {
      const int t = c * TK + j;
      s[j] = (t < T && (!causal || t <= i)) ? s[j] * scale : -INFINITY;
      mc = fmaxf(mc, s[j]);
    }
    const float corr = expf(m - mc);
    m = mc;
    l *= corr;
#pragma unroll
    for (int d = 0; d < AD; ++d) acc[d] *= corr;
#pragma unroll
    for (int j = 0; j < TK; ++j) {
      const float p = expf(s[j] - mc);
      l += p;
#pragma unroll
      for (int d = 0; d < AD; d += 4) {
        const float4 vf = *reinterpret_cast<const float4*>(Vc + j * AD + d);
        acc[d] = fmaf(p, vf.x, acc[d]);
        acc[d + 1] = fmaf(p, vf.y, acc[d + 1]);
        acc[d + 2] = fmaf(p, vf.z, acc[d + 2]);
        acc[d + 3] = fmaf(p, vf.w, acc[d + 3]);
      }
    }
    __syncwarp();            // every lane is done with this buffer before chunk c + 2 refills it
  }
  if (i >= T) return;
  const float inv = 1.0f / l;
  const size_t off = (row0 + (size_t)i * N) * ldo + col;
#pragma unroll
  for (int d = 0; d < AD; d += 4) {
    const float4 ov = make_float4(acc[d] * inv, acc[d + 1] * inv, acc[d + 2] * inv, acc[d + 3] * inv);
    if (o_hi != nullptr) store_split4(o_hi, o_lo, off + d, ov);
    else *reinterpret_cast<float4*>(o + off + d) = ov;
  }
}

static int launch_temporal_long(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, float* o,
                                uint16_t* o_hi, uint16_t* o_lo, int ldo, int B, int T, int N, int heads, float scale,
                                int causal, cudaStream_t st) {
  static bool done[64];      // the attribute is per device
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && !done[dev]) {
    OMT_CUDA(cudaFuncSetAttribute(attn_temporal_long_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, T_SMEM));
    done[dev] = true;
  }
  const dim3 grid((unsigned)(((long long)B * N + TW - 1) / TW), heads, (T + TQ - 1) / TQ);
  OMT_CUDA(launch_k(attn_temporal_long_kernel, grid, dim3(TW * 32), T_SMEM, st, q, ldq, k, ldk, v, ldv, o, o_hi, o_lo, ldo,
                    B, T, N, scale, causal));
  OMT_LAUNCH_CHECK();
  return OMT_OK;
}

int launch_attn_tc3(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, float* o, uint16_t* o_hi,
                    uint16_t* o_lo, int ldo, int n_seq, int N, int heads, float scale, cudaStream_t st);
int g_attn_kernel = 3;   // N % 128 == 0: 3 = tcgen05 3xTF32, Q / P as TMEM operands (attention_tc3.cu); 1 = CUDA-core fp32

static int set_flash_smem() {
  static bool done[64];      // the attribute is per device
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && !done[dev]) {
    OMT_CUDA(cudaFuncSetAttribute(attn_flash_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
    OMT_CUDA(cudaFuncSetAttribute(attn_flash_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
    done[dev] = true;
  }
  return OMT_OK;
}

}  // namespace omt

using namespace omt;

static int check_attn_ptrs(const char* who, const float* q, int ldq, const float* k, int ldk, const float* v,
                           int ldv, float* o, uint16_t* o_hi, uint16_t* o_lo, int ldo) {
  OMT_REQUIRE(q && k && v && (o || o_hi) && ((o_hi == nullptr) == (o_lo == nullptr)), "%s: null pointer", who);
  OMT_REQUIRE(((uintptr_t)o_hi | (uintptr_t)o_lo) % 8 == 0, "%s: output planes must be 8-byte aligned", who);
  OMT_REQUIRE(ldq % 4 == 0 && ldk % 4 == 0 && ldv % 4 == 0 && ldo % 4 == 0, "%s: leading dims must be multiples of 4", who);
  OMT_REQUIRE(((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)o) % 16 == 0, "%s: pointers must be 16-byte aligned", who);
  return OMT_OK;
}

extern "C" int omt_attn_spatial(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv,
                                float* o, uint16_t* o_hi, uint16_t* o_lo, int ldo, int n_seq, int N, int heads, float scale,
                                omt_stream_t stream) {
  OMT_ENTER();
  int rc = check_attn_ptrs("omt_attn_spatial", q, ldq, k, ldk, v, ldv, o, o_hi, o_lo, ldo);
  if (rc) return rc;
  OMT_REQUIRE(N > 0 && N % 64 == 0, "omt_attn_spatial: N=%d must be a multiple of 64", N);
  OMT_REQUIRE(heads > 0 && heads <= 65535 && n_seq <= 65535, "omt_attn_spatial: grid too large");
  if (n_seq == 0) return OMT_OK;
  if (g_attn_kernel == 3 && N % 128 == 0)
    return launch_attn_tc3(q, ldq, k, ldk, v, ldv, o, o_hi, o_lo, ldo, n_seq, N, heads, scale, (cudaStream_t)stream);
  rc = set_flash_smem();
  if (rc) return rc;
  AttnArgs a{q, ldq, k, ldk, v, ldv, o, ldo, o_hi, o_lo, nullptr, N, 0, 0, 0, scale};
  dim3 grid(N / AQ, heads, n_seq);
  OMT_CUDA(launch_k(attn_flash_kernel<false>, grid, dim3(256), 65536, (cudaStream_t)stream, a));
  OMT_LAUNCH_CHECK();
  return OMT_OK;
}

extern "C" int omt_attn_window(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv,
                               float* o, uint16_t* o_hi, uint16_t* o_lo, int ldo, const float* bias, int n_frames, int h,
                               int w, int ws, int heads, float scale, omt_stream_t stream) {
  OMT_ENTER();
  int rc = check_attn_ptrs("omt_attn_window", q, ldq, k, ldk, v, ldv, o, o_hi, o_lo, ldo);
  if (rc) return rc;
  OMT_REQUIRE(bias != nullptr, "omt_attn_window: null bias");
  OMT_REQUIRE(ws * ws == 64, "omt_attn_window: window %dx%d unsupported (8x8 only)", ws, ws);
  OMT_REQUIRE(h % ws == 0 && w % ws == 0, "omt_attn_window: grid %dx%d not divisible by the window", h, w);
  const long long n_seq = (long long)n_frames * (h / ws) * (w / ws);
  OMT_REQUIRE(n_seq <= 0x7fffffffLL / 64, "omt_attn_window: too many windows");
  if (n_seq == 0) return OMT_OK;
  rc = set_flash_smem();
  if (rc) return rc;
  AttnArgs a{q, ldq, k, ldk, v, ldv, o, ldo, o_hi, o_lo, bias, h * w, h, w, ws, scale};
  dim3 grid((unsigned)n_seq, heads, 1);
  OMT_CUDA(launch_k(attn_flash_kernel<true>, grid, dim3(256), 65536, (cudaStream_t)stream, a));
  OMT_LAUNCH_CHECK();
  return OMT_OK;
}

extern "C" int omt_attn_temporal(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv,
                                 float* o, uint16_t* o_hi, uint16_t* o_lo, int ldo, int B, int T, int N, int heads,
                                 float scale, int causal, omt_stream_t stream) {
  OMT_ENTER();
  int rc = check_attn_ptrs("omt_attn_temporal", q, ldq, k, ldk, v, ldv, o, o_hi, o_lo, ldo);
  if (rc) return rc;
  OMT_REQUIRE(T >= 1, "omt_attn_temporal: T'=%d unsupported (>= 1)", T);
  OMT_REQUIRE(B >= 0 && N >= 0 && heads > 0 && heads <= 65535 && (T + TQ - 1) / TQ <= 65535 &&
              ((long long)B * N + TW - 1) / TW <= 0x7fffffffLL, "omt_attn_temporal: grid too large");
  if ((long long)B * N == 0) return OMT_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (T > 17)
    return launch_temporal_long(q, ldq, k, ldk, v, ldv, o, o_hi, o_lo, ldo, B, T, N, heads, scale, causal, st);
#define OMT_T_CASE(t) case t: return launch_temporal<t>(q, ldq, k, ldk, v, ldv, o, o_hi, o_lo, ldo, B, N, heads, scale, causal, st);
  switch (T) {
    OMT_T_CASE(1) OMT_T_CASE(2) OMT_T_CASE(3) OMT_T_CASE(4) OMT_T_CASE(5) OMT_T_CASE(6) OMT_T_CASE(7)
    OMT_T_CASE(8) OMT_T_CASE(9) OMT_T_CASE(10) OMT_T_CASE(11) OMT_T_CASE(12) OMT_T_CASE(13) OMT_T_CASE(14)
    OMT_T_CASE(15) OMT_T_CASE(16) OMT_T_CASE(17)
  }
#undef OMT_T_CASE
  return OMT_E_ARG;
}
