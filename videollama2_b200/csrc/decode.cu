// Single-token (KV-cache decode) kernels: the M = 1 weight-streaming GEMV with fused RMSNorm, the L2 weight prefetch hint
// and the split-KV attention over the fused-row cache.  HBM / latency-bound; see DESIGN.md section 3 "Decode".
#include "row_common.cuh"

namespace vl2 {

// ---------------------------------------------------------------------------------------------------------
// GEMV (M = 1): y[n] = act(s * dot(W[n,:], x) + bias[n]) (+ residual[n]); s = rsqrt(mean(x^2) + eps) when rms_eps > 0
// (RMSNorm whose gain is folded into W: the norm is linear in x up to the row scale, so it costs one multiply here).
// One warp owns R consecutive rows of W; x is read through L1 (shared by every CTA of the SM).  HBM-bound: 2*N*K bytes.
// Each warp streams its R rows through a private ring of kGemvStages shared-memory stages filled by 1-D bulk copies
// (cp.async.bulk + mbarrier): the bytes in flight are set by the ring depth, not by how many loads the compiler keeps
// in registers, so even N = 4096 (one row per warp, 28 warps per SM) keeps > 100 KB per SM outstanding.
// FP8 = true: W is fp8 E4M3 with one fp32 scale per row (w_scale): y[n] = act(w_scale[n] * s * dot(W8[n,:], x) + ...),
// N*K bytes.  Same ring, barriers, PDL points and epilogue; a stage then holds 2048 weights and a lane consumes 16 weights
// (one 16-byte smem read) and 32 bytes of x per step.  Decode weights only: prefill stays on the bf16 GEMM.
// ---------------------------------------------------------------------------------------------------------
constexpr int kGemvChunk = 2048;                      // bytes of one row per stage (1024 bf16 or 2048 fp8 weights)
constexpr int kGemvWarps = 4;
// Ring depth: R = 1 (N < 8192: o_proj / down_proj / q,k,v) uses 3 stages = 24 KB per CTA so that 7+ CTAs fit on an SM and
// the 1024-CTA grids of the 4096-row projections run as ONE wave (ncu: with 4 stages 6 CTAs fit -> 1.15 waves, the
// second one nearly empty); R = 2 uses 4 stages.  fp8 always runs R = 2 with 2 stages (32 KB per CTA, 6 CTAs per SM):
// its rows are half as long, so a CTA's fixed latency (launch, first stage) is spread over half the bytes, and more
// resident CTAs hide it; 2 x 2 rows x 2 KB per warp in flight still covers a 4096-wide row without a refill.
template <int R, bool FP8 = false> struct GemvCfg { static constexpr int kStages = FP8 ? 2 : (R == 1 ? 3 : 4); };

template <int R, bool RMS, bool FP8>
__global__ void __launch_bounds__(kGemvWarps * 32)
gemv_kernel(const __nv_bfloat16* __restrict__ x, const void* __restrict__ W, const float* __restrict__ bias,
            const __nv_bfloat16* __restrict__ residual, void* __restrict__ y, int out_f32, int N, int K, int act,
            float rms_eps, const float* __restrict__ w_scale) {
  constexpr int kGemvStages = GemvCfg<R, FP8>::kStages;
  extern __shared__ __align__(128) uint8_t gemv_smem[];
  __shared__ uint64_t bars[kGemvWarps][GemvCfg<R, FP8>::kStages];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = (blockIdx.x * kGemvWarps + warp) * R;
  if (n0 >= N) return;                                  // whole warp leaves: no block-wide barrier below
  uint8_t* ring = gemv_smem + (size_t)warp * kGemvStages * R * kGemvChunk;
  uint64_t* bar = bars[warp];
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < kGemvStages; ++s) mbar_init(&bar[s], 1);
    fence_barrier_init();
  }
  __syncwarp();
  const int row_bytes = FP8 ? K : K * 2;
  const int n_chunks = (row_bytes + kGemvChunk - 1) / kGemvChunk;
  const uint8_t* wrow[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    if constexpr (FP8) wrow[r] = static_cast<const uint8_t*>(W) + (int64_t)min(n0 + r, N - 1) * K;
    else wrow[r] = reinterpret_cast<const uint8_t*>(static_cast<const __nv_bfloat16*>(W) + (int64_t)min(n0 + r, N - 1) * K);
  }
  auto issue = [&](int c) {   // lane 0 only
    const int s = c % kGemvStages;
    const int off = c * kGemvChunk;
    const uint32_t bytes = (uint32_t)min(kGemvChunk, row_bytes - off);
    mbar_arrive_expect_tx(&bar[s], bytes * R);
#pragma unroll
    for (int r = 0; r < R; ++r) bulk_load_1d(ring + (s * R + r) * kGemvChunk, wrow[r] + off, bytes, &bar[s]);
  };
  if (lane == 0)
    for (int c = 0; c < kGemvStages - 1 && c < n_chunks; ++c) issue(c);
  pdl_wait();   // weights are constants: their first stages are already in flight while the producer of x drains
  float acc[R];
#pragma unroll
  for (int r = 0; r < R; ++r) acc[r] = 0.f;
  float ss = 0.f;
  const uint4* xp = reinterpret_cast<const uint4*>(x);
  const int nk8 = K >> 3;
  if constexpr (FP8) {
    float acc2[R];    // second chain per row (odd weight pairs): halves the dependent-FMA latency per 16-weight step
#pragma unroll
    for (int r = 0; r < R; ++r) acc2[r] = 0.f;
    for (int c = 0; c < n_chunks; ++c) {
      const int s = c % kGemvStages;
      if (lane == 0 && c + kGemvStages - 1 < n_chunks) issue(c + kGemvStages - 1);
      uint4 xv[kGemvChunk / 256];   // 16 x values (two uint4) per lane per 512-weight step
#pragma unroll
      for (int u = 0; u < kGemvChunk / 512; ++u) {
        const int idx = c * (kGemvChunk / 8) + u * 64 + lane * 2;
        xv[2 * u] = idx < nk8 ? __ldg(xp + idx) : make_uint4(0, 0, 0, 0);
        xv[2 * u + 1] = idx < nk8 ? __ldg(xp + idx + 1) : make_uint4(0, 0, 0, 0);
      }
      mbar_wait(&bar[s], (c / kGemvStages) & 1);
#pragma unroll
      for (int u = 0; u < kGemvChunk / 512; ++u) {
        const int idx = c * (kGemvChunk / 8) + u * 64 + lane * 2;
        if (idx < nk8) {            // K % 16 == 0: both halves of the 16-weight group are in range
          const uint32_t xa[8] = {xv[2 * u].x,     xv[2 * u].y,     xv[2 * u].z,     xv[2 * u].w,
                                  xv[2 * u + 1].x, xv[2 * u + 1].y, xv[2 * u + 1].z, xv[2 * u + 1].w};
          float xf[16];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            xf[2 * j] = bf16_lo(xa[j]);
            xf[2 * j + 1] = bf16_hi(xa[j]);
            if (RMS) {
              ss = fmaf(xf[2 * j], xf[2 * j], ss);
              ss = fmaf(xf[2 * j + 1], xf[2 * j + 1], ss);
            }
          }
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const uint4 wq = *reinterpret_cast<const uint4*>(ring + (s * R + r) * kGemvChunk + (u * 32 + lane) * 16);
            const uint32_t wa[4] = {wq.x, wq.y, wq.z, wq.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float2 w01 = e4m3x2_to_float2(wa[j]);
              const float2 w23 = e4m3x2_to_float2(wa[j] >> 16);
              acc[r] = fmaf(xf[4 * j], w01.x, acc[r]);
              acc[r] = fmaf(xf[4 * j + 1], w01.y, acc[r]);
              acc2[r] = fmaf(xf[4 * j + 2], w23.x, acc2[r]);
              acc2[r] = fmaf(xf[4 * j + 3], w23.y, acc2[r]);
            }
          }
        }
      }
      __syncwarp();
    }
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] += acc2[r];
  } else {
    for (int c = 0; c < n_chunks; ++c) {
      const int s = c % kGemvStages;
      // refill the stage consumed in the previous iteration (every lane passed the __syncwarp at its end)
      if (lane == 0 && c + kGemvStages - 1 < n_chunks) issue(c + kGemvStages - 1);
      uint4 xv[kGemvChunk / 512];
#pragma unroll
      for (int u = 0; u < kGemvChunk / 512; ++u) {
        const int idx = c * (kGemvChunk / 16) + u * 32 + lane;
        xv[u] = idx < nk8 ? __ldg(xp + idx) : make_uint4(0, 0, 0, 0);
      }
      mbar_wait(&bar[s], (c / kGemvStages) & 1);
#pragma unroll
      for (int u = 0; u < kGemvChunk / 512; ++u) {
        const int idx = c * (kGemvChunk / 16) + u * 32 + lane;
        if (idx < nk8) {
          const uint32_t xa[4] = {xv[u].x, xv[u].y, xv[u].z, xv[u].w};
          float xf[8];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            xf[2 * j] = bf16_lo(xa[j]);
            xf[2 * j + 1] = bf16_hi(xa[j]);
            if (RMS) {
              ss = fmaf(xf[2 * j], xf[2 * j], ss);
              ss = fmaf(xf[2 * j + 1], xf[2 * j + 1], ss);
            }
          }
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const uint4 wq = *reinterpret_cast<const uint4*>(ring + (s * R + r) * kGemvChunk + (u * 32 + lane) * 16);
            const uint32_t wa[4] = {wq.x, wq.y, wq.z, wq.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              acc[r] = fmaf(xf[2 * j], bf16_lo(wa[j]), acc[r]);
              acc[r] = fmaf(xf[2 * j + 1], bf16_hi(wa[j]), acc[r]);
            }
          }
        }
      }
      __syncwarp();
    }
  }
  // late PDL trigger: the dependent grid is launched while this one drains (its CTAs only prefetch weights until
  // griddepcontrol.wait releases them), never while this grid still has CTAs waiting for an SM slot
  pdl_launch_dependents();
#pragma unroll
  for (int r = 0; r < R; ++r) acc[r] = warp_sum(acc[r]);
  if (RMS) ss = warp_sum(ss);
  if (lane != 0) return;
  const float s = RMS ? rsqrtf(ss / (float)K + rms_eps) : 1.f;
  float v[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    if constexpr (FP8) v[r] = acc[r] * w_scale[min(n0 + r, N - 1)] * s;
    else v[r] = acc[r] * s;
    if (bias != nullptr && n0 + r < N) v[r] += bias[n0 + r];
  }
  if (act == VL2_ACT_SWIGLU) {   // rows (n0, n0+1) are a (gate, up) pair -> output n0/2      (R == 2)
    const float o = silu(v[0]) * v[R - 1];
    if (out_f32) reinterpret_cast<float*>(y)[n0 >> 1] = o;
    else reinterpret_cast<__nv_bfloat16*>(y)[n0 >> 1] = __float2bfloat16_rn(o);
    return;
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    if (n0 + r >= N) break;
    float o = v[r];
    if (act == VL2_ACT_SILU) o = silu(o);
    else if (act == 100) o = 1.f / (1.f + __expf(-o));
    if (residual != nullptr) o += __bfloat162float(residual[n0 + r]);
    if (out_f32) reinterpret_cast<float*>(y)[n0 + r] = o;
    else reinterpret_cast<__nv_bfloat16*>(y)[n0 + r] = __float2bfloat16_rn(o);
  }
}

// ---------------------------------------------------------------------------------------------------------
// L2 prefetch of a weight range (cp.async.bulk.prefetch.L2): launched on a forked branch of the decode graph while the
// latency-bound attention phase leaves HBM idle, so that the following GEMVs find (part of) their weights in the 126 MB L2.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32)
l2_prefetch_kernel(const uint8_t* __restrict__ base, size_t bytes, unsigned chunk) {
  const size_t n_chunks = (bytes + chunk - 1) / chunk;
  for (size_t c = (size_t)blockIdx.x * 32 + threadIdx.x; c < n_chunks; c += (size_t)gridDim.x * 32) {
    const size_t off = c * chunk;
    const unsigned n = (unsigned)(bytes - off < chunk ? bytes - off : chunk) & ~15u;
    if (n) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(base + off), "r"(n) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------------
// Single-token (decode) attention over a KV cache held as rows of the fused QKV buffer, split over the KV length
// (flash-decoding): grid (kv head, split); a CTA takes the 128-position tiles `split, split + nsplit, ...` of its kv
// head and serves all `group` query heads that share it, so K and V are read from HBM exactly once.
//   scores : thread = position, the whole K row in registers (16-byte loads, all independent -> one memory round trip)
//   softmax: running max / sum per query head across the CTA's tiles
//   P.V    : thread = (position subgroup, 8 output columns), 16-byte V loads, again all independent
// Every (head, split) writes (m, l, o[D]) to the workspace; attn_decode_combine_kernel merges the splits.
// The tile -> split assignment depends only on n_pos, so the graph-replayed variant (n_pos read from device memory,
// grid sized for the cache capacity) is bit-identical to the eager one.
// ---------------------------------------------------------------------------------------------------------
constexpr int kDecTile = 128;

template <int G, int D>
__global__ void __launch_bounds__(128)
attn_decode_split_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ kc,
                         const __nv_bfloat16* __restrict__ vc, float* __restrict__ ws, int64_t ldkv, int n_pos, int group,
                         float scale, const int* __restrict__ pos_ptr) {
  pdl_wait();
  constexpr int NG = D / 8;              // 16-byte column groups per row
  constexpr int NSUB = kDecTile / NG;    // position subgroups in the P.V phase
  constexpr int PV_IT = kDecTile / NSUB; // positions per thread per tile in the P.V phase
  __shared__ __align__(16) float qs[G][D];
  __shared__ float ps[G][kDecTile];
  __shared__ float red[G][4];
  __shared__ float osum[NSUB][D + 4];
  if (pos_ptr != nullptr) n_pos = *pos_ptr + 1;
  const int kvh = blockIdx.x, split = blockIdx.y, nsplit = gridDim.y;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < G * D; i += 128) {
    const int g = i / D, d = i % D;
    qs[g][d] = g < group ? __bfloat162float(q[(kvh * group + g) * D + d]) * scale : 0.f;
  }
  __syncthreads();
  float m_run[G], l_run[G];
  float o[G][8];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    m_run[g] = -INFINITY;
    l_run[g] = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) o[g][e] = 0.f;
  }
  const int n_tiles = (n_pos + kDecTile - 1) / kDecTile;
  if (split >= n_tiles) return;          // no tile for this split: the combine kernel skips its slot
  const int cg = tid % NG, sub = tid / NG;
  for (int tile = split; tile < n_tiles; tile += nsplit) {
    const int pos = tile * kDecTile + tid;
    float sc[G];
#pragma unroll
    for (int g = 0; g < G; ++g) sc[g] = 0.f;
    if (pos < n_pos) {
      const uint4* kr = reinterpret_cast<const uint4*>(kc + (int64_t)pos * ldkv + kvh * D);
      uint4 kv[NG];
#pragma unroll
      for (int c = 0; c < NG; ++c) kv[c] = __ldg(kr + c);
#pragma unroll
      for (int c = 0; c < NG; ++c) {
        const uint32_t ka[4] = {kv[c].x, kv[c].y, kv[c].z, kv[c].w};
        float kf[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          kf[2 * j] = bf16_lo(ka[j]);
          kf[2 * j + 1] = bf16_hi(ka[j]);
        }
#pragma unroll
        for (int g = 0; g < G; ++g) {
          const float4 q0 = *reinterpret_cast<const float4*>(&qs[g][c * 8]);
          const float4 q1 = *reinterpret_cast<const float4*>(&qs[g][c * 8 + 4]);
          sc[g] = fmaf(q0.x, kf[0], sc[g]); sc[g] = fmaf(q0.y, kf[1], sc[g]);
          sc[g] = fmaf(q0.z, kf[2], sc[g]); sc[g] = fmaf(q0.w, kf[3], sc[g]);
          sc[g] = fmaf(q1.x, kf[4], sc[g]); sc[g] = fmaf(q1.y, kf[5], sc[g]);
          sc[g] = fmaf(q1.z, kf[6], sc[g]); sc[g] = fmaf(q1.w, kf[7], sc[g]);
        }
      }
    } else {
#pragma unroll
      for (int g = 0; g < G; ++g) sc[g] = -INFINITY;
    }
    // tile max per query head
#pragma unroll
    for (int g = 0; g < G; ++g) {
      float mx = sc[g];
#pragma unroll
      for (int of = 16; of > 0; of >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, of));
      if (lane == 0) red[g][warp] = mx;
    }
    __syncthreads();
    float alpha[G];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const float mt = fmaxf(fmaxf(red[g][0], red[g][1]), fmaxf(red[g][2], red[g][3]));
      const float m_new = fmaxf(m_run[g], mt);       // finite: every tile holds at least one valid position
      alpha[g] = __expf(m_run[g] - m_new);
      m_run[g] = m_new;
      const float pv = __expf(sc[g] - m_new);
      ps[g][tid] = pv;
    }
    __syncthreads();
    // row sums (every thread computes the same value in the same order: no second reduction tree needed)
#pragma unroll
    for (int g = 0; g < G; ++g) {
      float sm = ps[g][lane] + ps[g][lane + 32] + ps[g][lane + 64] + ps[g][lane + 96];
      sm = warp_sum(sm);
      l_run[g] = l_run[g] * alpha[g] + sm;
#pragma unroll
      for (int e = 0; e < 8; ++e) o[g][e] *= alpha[g];
    }
    // P.V: this thread's positions are sub, sub + NSUB, ...
    uint4 vv[PV_IT];
#pragma unroll
    for (int it = 0; it < PV_IT; ++it) {
      const int pp = tile * kDecTile + it * NSUB + sub;
      vv[it] = pp < n_pos ? __ldg(reinterpret_cast<const uint4*>(vc + (int64_t)pp * ldkv + kvh * D) + cg)
                          : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int it = 0; it < PV_IT; ++it) {
      const uint32_t va[4] = {vv[it].x, vv[it].y, vv[it].z, vv[it].w};
      float vf[8];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        vf[2 * j] = bf16_lo(va[j]);
        vf[2 * j + 1] = bf16_hi(va[j]);
      }
#pragma unroll
      for (int g = 0; g < G; ++g) {
        const float pv = ps[g][it * NSUB + sub];
#pragma unroll
        for (int e = 0; e < 8; ++e) o[g][e] = fmaf(pv, vf[e], o[g][e]);
      }
    }
    __syncthreads();   // ps / red are rewritten by the next tile
  }
  pdl_launch_dependents();
  // combine the position subgroups (fixed order) and publish (m, l, o) of every query head of this kv head
  for (int g = 0; g < G; ++g) {
    if (g >= group) break;
#pragma unroll
    for (int e = 0; e < 8; ++e) osum[sub][cg * 8 + e] = o[g][e];
    __syncthreads();
    float* dst = ws + ((int64_t)(kvh * group + g) * nsplit + split) * (D + 2);
    if (tid < D) {
      float a = 0.f;
#pragma unroll
      for (int sb = 0; sb < NSUB; ++sb) a += osum[sb][tid];
      dst[2 + tid] = a;
    }
    if (tid == 0) {
      dst[0] = m_run[g];
      dst[1] = l_run[g];
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(128)
attn_decode_combine_kernel(const float* __restrict__ ws, __nv_bfloat16* __restrict__ out, int nsplit, int D, int n_pos,
                           const int* __restrict__ pos_ptr) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float wgt[64];
  __shared__ float inv_l;
  if (pos_ptr != nullptr) n_pos = *pos_ptr + 1;
  const int n_tiles = (n_pos + kDecTile - 1) / kDecTile;
  const int n_act = n_tiles < nsplit ? n_tiles : nsplit;   // splits >= n_tiles held no tile and wrote nothing
  const int h = blockIdx.x, tid = threadIdx.x;
  const float* base = ws + (int64_t)h * nsplit * (D + 2);
  if (tid < 32) {      // nsplit <= 64: two entries per lane
    const float m0 = tid < n_act ? base[tid * (D + 2)] : -INFINITY;
    const float m1 = tid + 32 < n_act ? base[(tid + 32) * (D + 2)] : -INFINITY;
    const float l0 = tid < n_act ? base[tid * (D + 2) + 1] : 0.f;
    const float l1 = tid + 32 < n_act ? base[(tid + 32) * (D + 2) + 1] : 0.f;
    float M = fmaxf(m0, m1);
#pragma unroll
    for (int of = 16; of > 0; of >>= 1) M = fmaxf(M, __shfl_xor_sync(0xffffffffu, M, of));
    const float w0 = __expf(m0 - M), w1 = __expf(m1 - M);
    wgt[tid] = w0;
    wgt[tid + 32] = w1;
    const float l = warp_sum(w0 * l0 + w1 * l1);
    if (tid == 0) inv_l = 1.f / l;
  }
  __syncthreads();
  if (tid < D) {
    float a = 0.f;
#pragma unroll 8
    for (int sp = 0; sp < n_act; ++sp) a = fmaf(wgt[sp], base[sp * (D + 2) + 2 + tid], a);
    out[h * D + tid] = __float2bfloat16_rn(a * inv_l);
  }
}

static inline int decode_nsplit(int Hkv) {
  int n = (2 * 148) / Hkv;
  return n < 1 ? 1 : (n > 64 ? 64 : n);
}

}  // namespace vl2

using namespace vl2;
typedef __nv_bfloat16 bf16;

int vl2::launch_gemv(const void* x, const void* W, const float* bias, const void* residual, void* y, int out_f32, int N,
                       int K, int act, float rms_eps, cudaStream_t stream, const float* w_scale) {
  const bool fp8 = w_scale != nullptr;
  const bool two = fp8 || act == VL2_ACT_SWIGLU || N >= 8192;
  const bool rms = rms_eps > 0.f;
  const int rows_per_cta = kGemvWarps * (two ? 2 : 1);
  const int blocks = (N + rows_per_cta - 1) / rows_per_cta;
  const size_t smem = fp8 ? (size_t)kGemvWarps * GemvCfg<2, true>::kStages * 2 * kGemvChunk
                     : two ? (size_t)kGemvWarps * GemvCfg<2>::kStages * 2 * kGemvChunk
                           : (size_t)kGemvWarps * GemvCfg<1>::kStages * kGemvChunk;
#define VL2_GEMV(RR, RMS_, F8)                                                                                              \
  launch_kernel(gemv_kernel<RR, RMS_, F8>, dim3(blocks), dim3(kGemvWarps * 32), smem, stream, 1, (const bf16*)x, W, bias,   \
                (const bf16*)residual, y, out_f32, N, K, act, rms_eps, w_scale)
  if (fp8) {
    if (rms) VL2_GEMV(2, true, true);
    else VL2_GEMV(2, false, true);
  } else {
    VL2_SMEM_OPT_IN((gemv_kernel<2, true, false>), 64 * 1024);
    VL2_SMEM_OPT_IN((gemv_kernel<2, false, false>), 64 * 1024);
    if (two && rms) VL2_GEMV(2, true, false);
    else if (two) VL2_GEMV(2, false, false);
    else if (rms) VL2_GEMV(1, true, false);
    else VL2_GEMV(1, false, false);
  }
#undef VL2_GEMV
  VL2_CHECK_LAUNCH("gemv_kernel");
  return VL2_OK;
}

extern "C" int vl2_gemv_bf16(const void* x, const void* W, const float* bias, const void* residual, void* y, int out_f32,
                             int N, int K, int act, float rms_eps, void* stream) {
  VL2_REQUIRE(N > 0 && K > 0 && K % 8 == 0, VL2_E_BADSHAPE, "vl2_gemv_bf16: need K %% 8 == 0 (N=%d K=%d)", N, K);
  VL2_REQUIRE(x && W && y && aligned16(x) && aligned16(W), VL2_E_BADALIGN, "vl2_gemv_bf16: 16-byte alignment");
  VL2_REQUIRE(act == VL2_ACT_NONE || act == VL2_ACT_SILU || act == 100 || act == VL2_ACT_SWIGLU, VL2_E_UNSUPPORTED,
              "vl2_gemv_bf16: act %d", act);
  VL2_REQUIRE(act != VL2_ACT_SWIGLU || (N % 2 == 0 && residual == nullptr), VL2_E_UNSUPPORTED,
              "vl2_gemv_bf16: SWIGLU needs even N and no residual");
  return launch_gemv(x, W, bias, residual, y, out_f32, N, K, act, rms_eps, (cudaStream_t)stream);
}

extern "C" int vl2_gemv_fp8(const void* x, const void* W8, const float* w_scale, const float* bias, const void* residual,
                            void* y, int out_f32, int N, int K, int act, float rms_eps, void* stream) {
  VL2_REQUIRE(N > 0 && K > 0 && K % 16 == 0, VL2_E_BADSHAPE, "vl2_gemv_fp8: need K %% 16 == 0 (N=%d K=%d)", N, K);
  VL2_REQUIRE(w_scale != nullptr, VL2_E_BADSHAPE, "vl2_gemv_fp8: w_scale (fp32 [N]) is required");
  VL2_REQUIRE(x && W8 && y && aligned16(x) && aligned16(W8), VL2_E_BADALIGN, "vl2_gemv_fp8: 16-byte alignment");
  VL2_REQUIRE(act == VL2_ACT_NONE || act == VL2_ACT_SILU || act == 100 || act == VL2_ACT_SWIGLU, VL2_E_UNSUPPORTED,
              "vl2_gemv_fp8: act %d", act);
  VL2_REQUIRE(act != VL2_ACT_SWIGLU || (N % 2 == 0 && residual == nullptr), VL2_E_UNSUPPORTED,
              "vl2_gemv_fp8: SWIGLU needs even N and no residual");
  return launch_gemv(x, W8, bias, residual, y, out_f32, N, K, act, rms_eps, (cudaStream_t)stream, w_scale);
}

extern "C" int vl2_l2_prefetch(const void* ptr, size_t bytes, void* stream) {
  VL2_REQUIRE(ptr != nullptr && aligned16(ptr), VL2_E_BADALIGN, "vl2_l2_prefetch: pointer must be 16-byte aligned");
  if (bytes < 16) return VL2_OK;
  launch_kernel(l2_prefetch_kernel, dim3(32), dim3(32), 0, (cudaStream_t)stream, 1, (const uint8_t*)ptr, bytes, 16384u);
  VL2_CHECK_LAUNCH("l2_prefetch_kernel");
  return VL2_OK;
}

extern "C" size_t vl2_attention_decode_workspace(int Hq, int Hkv, int D) {
  if (Hq <= 0 || Hkv <= 0 || D <= 0) return 0;
  return (size_t)Hq * decode_nsplit(Hkv) * (D + 2) * sizeof(float);
}

static int launch_decode_attn(const void* q, const void* k_cache, const void* v_cache, void* out, int64_t ldkv, int n_pos,
                              const int32_t* pos_dev, int Hq, int Hkv, int D, float scale, void* workspace,
                              cudaStream_t stream) {
  const int group = Hq / Hkv, nsplit = decode_nsplit(Hkv);
  dim3 grid(Hkv, nsplit);
  float* ws = (float*)workspace;
#define VL2_DEC(GG, DD)                                                                                              \
  launch_kernel(attn_decode_split_kernel<GG, DD>, grid, dim3(128), 0, stream, 1, (const bf16*)q, (const bf16*)k_cache, \
                (const bf16*)v_cache, ws, ldkv, n_pos, group, scale, (const int*)pos_dev)
  if (D == 128 && group <= 4) VL2_DEC(4, 128);
  else if (D == 128) VL2_DEC(8, 128);
  else if (group <= 4) VL2_DEC(4, 64);
  else VL2_DEC(8, 64);
#undef VL2_DEC
  VL2_CHECK_LAUNCH("attn_decode_split_kernel");
  launch_kernel(attn_decode_combine_kernel, dim3(Hq), dim3(128), 0, stream, 1, (const float*)ws, (bf16*)out, nsplit, D, n_pos,
                (const int*)pos_dev);
  VL2_CHECK_LAUNCH("attn_decode_combine_kernel");
  return VL2_OK;
}

extern "C" int vl2_attention_decode(const void* q, const void* k_cache, const void* v_cache, void* out, int64_t ldkv,
                                    int n_pos, int Hq, int Hkv, int D, float scale, void* workspace, void* stream) {
  VL2_REQUIRE(n_pos > 0 && Hq > 0 && Hkv > 0 && Hq % Hkv == 0 && Hq / Hkv <= 8 && (D == 64 || D == 128), VL2_E_BADSHAPE,
              "vl2_attention_decode: bad shape (n_pos=%d Hq=%d Hkv=%d D=%d; group <= 8, D 64|128)", n_pos, Hq, Hkv, D);
  VL2_REQUIRE(workspace != nullptr && ldkv % 8 == 0 && aligned16(k_cache) && aligned16(v_cache), VL2_E_BADALIGN,
              "vl2_attention_decode: workspace missing or misaligned cache");
  return launch_decode_attn(q, k_cache, v_cache, out, ldkv, n_pos, nullptr, Hq, Hkv, D, scale, workspace, (cudaStream_t)stream);
}

extern "C" int vl2_attention_decode_dyn(const void* q, const void* k_cache, const void* v_cache, void* out, int64_t ldkv,
                                        const int32_t* pos_dev, int Hq, int Hkv, int D, float scale, void* workspace,
                                        void* stream) {
  VL2_REQUIRE(pos_dev != nullptr && Hq > 0 && Hkv > 0 && Hq % Hkv == 0 && Hq / Hkv <= 8 && (D == 64 || D == 128),
              VL2_E_BADSHAPE, "vl2_attention_decode_dyn: bad shape (Hq=%d Hkv=%d D=%d)", Hq, Hkv, D);
  VL2_REQUIRE(workspace != nullptr && ldkv % 8 == 0 && aligned16(k_cache) && aligned16(v_cache), VL2_E_BADALIGN,
              "vl2_attention_decode_dyn: workspace missing or misaligned cache");
  return launch_decode_attn(q, k_cache, v_cache, out, ldkv, 0, pos_dev, Hq, Hkv, D, scale, workspace, (cudaStream_t)stream);
}
