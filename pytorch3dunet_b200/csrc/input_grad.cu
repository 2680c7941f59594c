// Gradient with respect to the fp32 network input: the data gradient of the first layer, written straight into the NCDHW fp32 layout
// of x (reference: the autograd of nn.Conv3d on the input volume, pytorch3dunet/unet3d/buildingblocks.py:56, and of ResNetBlock.conv1
// :251 for the residual families).
//
// (a) 3x3x3 conv, padding 1:  dxhat[n,ci,v] = scale * sum_tap sum_co W[co,ci,tap] * dz[n, v - (tap - 1), co]
//     C_in == 1, C_out in {8, 16, 32} (every shipped config): warp-level MMA (mma.sync m16n8k16, fp32 accumulate).  With one input
//     channel the output has one column, so the MMA runs the other way round: per dz voxel u it projects the C_out channels onto the
//     27 taps, Q[u][tap] = sum_co W[co,0,tap] * dz[u,co] (M = 16 voxels, N = 32 >= 27 taps, K = C_out), and the output voxel gathers
//     dxhat[v] = sum_tap Q[v - (tap - 1)][tap] from shared memory.  The volume is streamed plane by plane along D: each dz plane (with a
//     one-voxel halo in H and W) is projected once and adds its three tap planes into three rolling per-thread accumulators, so the
//     halo costs nothing along D and 1.33x along H x W.
//     Other C_in / C_out: one CUDA-core thread per output voxel.
//     Both paths: fixed summation order, no atomics (bit-reproducible); 16-bit operands dz and W (W rounded in the kernel, as
//     b200_prep_dgrad_weights rounds it for every other data gradient); optional per-block partial sums (sum dxhat, sum dxhat*x)
//     [N][P][C_in][2] for the GroupNorm backward of a layer that starts with a GroupNorm, applied afterwards by
//     b200_gn_bwd_apply_ncdhw_f32 (the coefficients need the whole-volume sums, so they cannot be applied in the same pass).
// (b) 1x1x1 conv: dx[n,ci,v] = scale * sum_co W[co,ci] * dy[n,v,co]; one thread per voxel, HBM-bound.
#include "common.cuh"
#include "ew.cuh"

namespace b200 {

#ifdef B200_ACT_F16
#define IG_MMA_TYPES "f16.f16"
#else
#define IG_MMA_TYPES "bf16.bf16"
#endif
__device__ __forceinline__ void ig_mma16816(float c[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32." IG_MMA_TYPES ".f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

constexpr int IG_TH = 8, IG_TW = 32;                    // output tile in H x W (one voxel per thread, 256 threads)
constexpr int IG_HH = IG_TH + 2, IG_HW = IG_TW + 2;     // dz halo plane 10 x 34
constexpr int IG_HALO = IG_HH * IG_HW;                  // 340 voxels
constexpr int IG_MT = (IG_HALO + 15) / 16;              // 22 m-tiles of 16 voxels
constexpr int IG_MT_PER_WARP = (IG_MT + 7) / 8;         // 3
// Q is stored tap-major, Qs[tap][halo voxel]; pitch = 4 (mod 32) makes the fragment stores (8 voxels x 4 tap pairs per instruction)
// and the gathers (32 consecutive voxels) conflict-free
constexpr int IG_PITCH = 356;

// z-chunk length along D: as long as the grid still has >= 512 blocks (or 4 planes), device-independent so that the partials count
// is a pure function of the shape
__host__ __device__ inline int ig_zchunk(int N, int D, int H, int W) {
  const long long tiles = (long long)((H + IG_TH - 1) / IG_TH) * ((W + IG_TW - 1) / IG_TW) * N;
  int zc = 32;
  while (zc > 4 && tiles * ((D + zc - 1) / zc) < 512) zc >>= 1;
  return zc;
}

template <int COUT>
__global__ void __launch_bounds__(256) input_dgrad_mma_kernel(const bf16* __restrict__ dz, const float* __restrict__ Wt, int D, int H, int W,
                                                              int zc, float scale, const float* __restrict__ x, float* __restrict__ dx,
                                                              float* __restrict__ partials) {
  constexpr int KS = (COUT + 15) / 16;  // k-steps of 16 channels (C_out = 8: one, upper half zero)
  __shared__ float Qs[27 * IG_PITCH];
  __shared__ float red[8][2];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tig = lane & 3;
  const int tW = (W + IG_TW - 1) / IG_TW;
  const int x0 = (blockIdx.x % tW) * IG_TW, y0 = (blockIdx.x / tW) * IG_TH;
  const int zb = blockIdx.y * zc, ze = min(D, zb + zc);
  const int n = blockIdx.z;
  const long long plane = (long long)H * W;
  const bf16* dzn = dz + (size_t)n * D * plane * COUT;
  // B fragments: n-tile t = taps 8t..8t+7 (column g), k rows tig*2, +1 and tig*2+8, +9 = channels of k-step ks
  uint32_t bfr[KS][4][2];
#pragma unroll
  for (int ks = 0; ks < KS; ++ks)
#pragma unroll
    for (int t = 0; t < 4; ++t)
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int tap = t * 8 + g, co = ks * 16 + hh * 8 + tig * 2;
        float w0 = 0.f, w1 = 0.f;
        if (tap < 27 && co < COUT) {
          w0 = Wt[(size_t)co * 27 + tap];
          w1 = Wt[(size_t)(co + 1) * 27 + tap];
        }
        bfr[ks][t][hh] = pack2(w0, w1);
      }
  // A fragment rows of this warp's m-tiles: halo voxel r -> (hy, hx); rows past the halo or outside the volume read zeros
  int roff[IG_MT_PER_WARP][2];
#pragma unroll
  for (int i = 0; i < IG_MT_PER_WARP; ++i)
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      const int r = (warp + 8 * i) * 16 + hh * 8 + g;
      const int hy = r / IG_HW, hx = r - hy * IG_HW;
      const int gy = y0 + hy - 1, gx = x0 + hx - 1;
      const bool ok = warp + 8 * i < IG_MT && r < IG_HALO && gy >= 0 && gy < H && gx >= 0 && gx < W;
      roff[i][hh] = ok ? gy * W + gx : -1;
    }
  uint32_t afr[IG_MT_PER_WARP][KS][4];
  auto fetch = [&](int zu) {
    const bool zok = zu >= 0 && zu < D;
    const bf16* src = dzn + (size_t)(zok ? zu : 0) * plane * COUT;
#pragma unroll
    for (int i = 0; i < IG_MT_PER_WARP; ++i)
#pragma unroll
      for (int ks = 0; ks < KS; ++ks)
#pragma unroll
        for (int j = 0; j < 4; ++j) {  // a0: row g, k lo; a1: row g+8, k lo; a2: row g, k hi; a3: row g+8, k hi
          const int o = roff[i][j & 1];
          const int co = ks * 16 + (j >> 1) * 8 + tig * 2;
          afr[i][ks][j] = (zok && o >= 0 && co < COUT) ? __ldg(reinterpret_cast<const uint32_t*>(src + (size_t)o * COUT + co)) : 0u;
        }
  };
  const int ly = warp, lx = lane, gy = y0 + ly, gx = x0 + lx;
  const bool own = gy < H && gx < W;
  float r0 = 0.f, r1 = 0.f, r2 = 0.f;  // output planes zu-1, zu, zu+1
  float s = 0.f, q = 0.f;
  fetch(zb - 1);
  for (int zu = zb - 1; zu <= ze; ++zu) {
    const bool zok = zu >= 0 && zu < D;  // block-uniform
    if (zok) {
      __syncthreads();  // the previous plane's gather is done with Qs
#pragma unroll
      for (int i = 0; i < IG_MT_PER_WARP; ++i) {
        const int mt = warp + 8 * i;
        if (mt >= IG_MT) continue;  // warp-uniform
        float acc[4][4];
#pragma unroll
        for (int t = 0; t < 4; ++t) acc[t][0] = acc[t][1] = acc[t][2] = acc[t][3] = 0.f;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks)
#pragma unroll
          for (int t = 0; t < 4; ++t) ig_mma16816(acc[t], afr[i][ks][0], afr[i][ks][1], afr[i][ks][2], afr[i][ks][3], bfr[ks][t][0], bfr[ks][t][1]);
        const int row = mt * 16 + g;
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const int tap = t * 8 + tig * 2;
          if (tap < 27) {
            Qs[tap * IG_PITCH + row] = acc[t][0];
            Qs[tap * IG_PITCH + row + 8] = acc[t][2];
          }
          if (tap + 1 < 27) {
            Qs[(tap + 1) * IG_PITCH + row] = acc[t][1];
            Qs[(tap + 1) * IG_PITCH + row + 8] = acc[t][3];
          }
        }
      }
      __syncthreads();
    }
    if (zu + 1 <= ze) fetch(zu + 1);  // in flight during the gather
    if (zok) {
      // plane zu adds tap plane a to output plane zu + a - 1: dz at (y - b + 1, x - c + 1) is halo (ly + 2 - b, lx + 2 - c)
      float part[3];
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        float acc = 0.f;
#pragma unroll
        for (int b = 0; b < 3; ++b)
#pragma unroll
          for (int c = 0; c < 3; ++c) acc += Qs[((a * 3 + b) * 3 + c) * IG_PITCH + (ly + 2 - b) * IG_HW + (lx + 2 - c)];
        part[a] = acc;
      }
      r0 += part[0];
      r1 += part[1];
      r2 += part[2];
    }
    const int zo = zu - 1;  // complete now
    if (zo >= zb && zo < ze && own) {
      const float v = r0 * scale;
      const size_t idx = ((size_t)n * D + zo) * plane + (size_t)gy * W + gx;
      dx[idx] = v;
      if (partials) {
        s += v;
        q = fmaf(v, x[idx], q);
      }
    }
    r0 = r1;
    r1 = r2;
    r2 = 0.f;
  }
  if (partials) {
    for (int o = 16; o > 0; o >>= 1) {
      s += __shfl_xor_sync(0xffffffffu, s, o);
      q += __shfl_xor_sync(0xffffffffu, q, o);
    }
    if (lane == 0) {
      red[warp][0] = s;
      red[warp][1] = q;
    }
    __syncthreads();
    if (threadIdx.x < 2) {
      float a = 0.f;
      for (int wv = 0; wv < 8; ++wv) a += red[wv][threadIdx.x];
      const int P = gridDim.x * gridDim.y;
      partials[((size_t)n * P + blockIdx.y * gridDim.x + blockIdx.x) * 2 + threadIdx.x] = a;
    }
  }
}

// CUDA-core path: one thread per output voxel and input channel at a time; grid (P, N), P = ceil(vox / 256)
__global__ void __launch_bounds__(256) input_dgrad_direct_kernel(const bf16* __restrict__ dz, const float* __restrict__ Wt, int D, int H,
                                                                 int W, int Cin, int Cout, float scale, const float* __restrict__ x,
                                                                 float* __restrict__ dx, float* __restrict__ partials) {
  extern __shared__ float red[];  // [8 warps][Cin][2]
  const long long vox = (long long)D * H * W;
  const int n = blockIdx.y;
  const long long v = (long long)blockIdx.x * 256 + threadIdx.x;
  const bool own = v < vox;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int z = 0, y = 0, xx = 0;
  if (own) {
    xx = (int)(v % W);
    y = (int)((v / W) % H);
    z = (int)(v / ((long long)W * H));
  }
  const bf16* dzn = dz + (size_t)n * vox * Cout;
  for (int ci = 0; ci < Cin; ++ci) {
    float acc = 0.f;
    if (own) {
      for (int tap = 0; tap < 27; ++tap) {
        const int sz = z - tap / 9 + 1, sy = y - (tap / 3) % 3 + 1, sx = xx - tap % 3 + 1;
        if (sz < 0 || sz >= D || sy < 0 || sy >= H || sx < 0 || sx >= W) continue;
        const bf16x8* src = reinterpret_cast<const bf16x8*>(dzn + (((size_t)sz * H + sy) * W + sx) * Cout);
        const float* wr = Wt + (size_t)ci * 27 + tap;
        for (int c8 = 0; c8 < Cout / 8; ++c8) {
          float f[8];
          unpack8(src[c8], f);
#pragma unroll
          for (int k = 0; k < 8; ++k) acc = fmaf(bf16_round(__ldg(wr + (size_t)(c8 * 8 + k) * Cin * 27)), f[k], acc);
        }
      }
    }
    const size_t idx = ((size_t)n * Cin + ci) * vox + v;
    const float val = acc * scale;
    if (own) dx[idx] = val;
    if (partials) {
      float a = own ? val : 0.f, b = own ? val * x[idx] : 0.f;
      for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
      }
      if (lane == 0) {
        red[(warp * Cin + ci) * 2] = a;
        red[(warp * Cin + ci) * 2 + 1] = b;
      }
    }
  }
  if (partials) {
    __syncthreads();
    for (int i = threadIdx.x; i < Cin * 2; i += 256) {
      float a = 0.f;
      for (int wv = 0; wv < 8; ++wv) a += red[wv * Cin * 2 + i];
      partials[((size_t)n * gridDim.x + blockIdx.x) * Cin * 2 + i] = a;
    }
  }
}

static bool input_dgrad_mma_ok(int Cin, int Cout) { return Cin == 1 && (Cout == 8 || Cout == 16 || Cout == 32); }

// out[n,c,v] = scale * (A*dxhat + B*x + Cc), coef[n][c] = (A, B, Cc); grid (blocks, N*C)
__global__ void gn_bwd_apply_ncdhw_f32_kernel(const float* __restrict__ dxhat, const float* __restrict__ x, const float* __restrict__ coef,
                                              long long vox, float scale, float* __restrict__ out) {
  const int nc = blockIdx.y;
  const float A = coef[nc * 3] * scale, B = coef[nc * 3 + 1] * scale, Cc = coef[nc * 3 + 2] * scale;
  const size_t base = (size_t)nc * vox;
  for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < vox; v += (long long)gridDim.x * blockDim.x)
    out[base + v] = fmaf(A, dxhat[base + v], fmaf(B, x[base + v], Cc));
}

// dx[n,ci,v] = scale * sum_co W[co][ci] dy[n,v,co]; grid (ceil(vox/256), N), W staged in shared memory
__global__ void __launch_bounds__(256) pointwise_dgrad_f32_kernel(const bf16* __restrict__ dy, const float* __restrict__ Wm, long long vox,
                                                                  int Cin, int Cout, float scale, float* __restrict__ dx) {
  extern __shared__ float wsm[];  // [Cout][Cin]
  for (int i = threadIdx.x; i < Cout * Cin; i += blockDim.x) wsm[i] = Wm[i];
  __syncthreads();
  const int n = blockIdx.y;
  const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= vox) return;
  const bf16x8* row = reinterpret_cast<const bf16x8*>(dy + ((size_t)n * vox + v) * Cout);
  for (int ci = 0; ci < Cin; ++ci) {
    float acc = 0.f;
    for (int c8 = 0; c8 < Cout / 8; ++c8) {
      float f[8];
      unpack8(row[c8], f);
#pragma unroll
      for (int k = 0; k < 8; ++k) acc = fmaf(wsm[(c8 * 8 + k) * Cin + ci], f[k], acc);
    }
    dx[((size_t)n * Cin + ci) * vox + v] = acc * scale;
  }
}

}  // namespace b200

using namespace b200;
#define ST(s) ((cudaStream_t)(s))

extern "C" {

int b200_input_dgrad_partials_count(int N, int D, int H, int W, int Cin, int Cout) {
  if (input_dgrad_mma_ok(Cin, Cout)) {
    const int zc = ig_zchunk(N, D, H, W);
    return ((H + IG_TH - 1) / IG_TH) * ((W + IG_TW - 1) / IG_TW) * ((D + zc - 1) / zc);
  }
  return ceil_div((long long)D * H * W, 256);
}

int b200_input_dgrad_conv3(const void* dz, const float* W, int N, int D, int H, int Wd, int Cin, int Cout, float scale, const float* x,
                           float* dx, float* partials, b200_stream_t s) {
  B200_CHECK_ARG(Cin >= 1 && Cout % 8 == 0 && Cout >= 8, "input_dgrad_conv3: Cin=%d Cout=%d (Cout must be a multiple of 8)", Cin, Cout);
  B200_CHECK_ARG(!partials || x, "input_dgrad_conv3: partial sums need x");
  if (input_dgrad_mma_ok(Cin, Cout)) {
    const int zc = ig_zchunk(N, D, H, Wd);
    dim3 grid(((H + IG_TH - 1) / IG_TH) * ((Wd + IG_TW - 1) / IG_TW), (D + zc - 1) / zc, N);
    if (Cout == 8)
      input_dgrad_mma_kernel<8><<<grid, 256, 0, ST(s)>>>((const bf16*)dz, W, D, H, Wd, zc, scale, x, dx, partials);
    else if (Cout == 16)
      input_dgrad_mma_kernel<16><<<grid, 256, 0, ST(s)>>>((const bf16*)dz, W, D, H, Wd, zc, scale, x, dx, partials);
    else
      input_dgrad_mma_kernel<32><<<grid, 256, 0, ST(s)>>>((const bf16*)dz, W, D, H, Wd, zc, scale, x, dx, partials);
    B200_CHECK_LAUNCH("input_dgrad_mma");
    return 0;
  }
  B200_CHECK_ARG(Cin <= 384, "input_dgrad_conv3: Cin=%d too large", Cin);
  dim3 grid(ceil_div((long long)D * H * Wd, 256), N);
  input_dgrad_direct_kernel<<<grid, 256, partials ? 8 * Cin * 2 * sizeof(float) : 0, ST(s)>>>((const bf16*)dz, W, D, H, Wd, Cin, Cout, scale,
                                                                                              x, dx, partials);
  B200_CHECK_LAUNCH("input_dgrad_direct");
  return 0;
}

int b200_gn_bwd_apply_ncdhw_f32(const float* dxhat, const float* x, const float* coef, int N, int C, long long voxels, float scale,
                                float* out, b200_stream_t s) {
  long long b = (voxels + 255) / 256;
  dim3 grid((unsigned)(b > 1024 ? 1024 : (b < 1 ? 1 : b)), N * C);
  gn_bwd_apply_ncdhw_f32_kernel<<<grid, 256, 0, ST(s)>>>(dxhat, x, coef, voxels, scale, out);
  B200_CHECK_LAUNCH("gn_bwd_apply_ncdhw_f32");
  return 0;
}

int b200_pointwise_dgrad_f32(const void* dy, const float* W, int N, long long voxels, int Cin, int Cout, float scale, float* dx,
                             b200_stream_t s) {
  B200_CHECK_ARG(Cout % 8 == 0 && (size_t)Cin * Cout * sizeof(float) <= 48 * 1024, "pointwise_dgrad_f32: Cin=%d Cout=%d unsupported", Cin,
                 Cout);
  dim3 grid(ceil_div(voxels, 256), N);
  pointwise_dgrad_f32_kernel<<<grid, 256, (size_t)Cin * Cout * sizeof(float), ST(s)>>>((const bf16*)dy, W, voxels, Cin, Cout, scale, dx);
  B200_CHECK_LAUNCH("pointwise_dgrad_f32");
  return 0;
}

}  // extern "C"
