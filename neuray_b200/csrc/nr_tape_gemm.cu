// Weight gradients from the backward tapes: for every Linear layer, dW[out][in] = sum over rows of dz[out] x[in] and
// db[out] = sum of dz[out] (one extra "input" that is constantly 1).  All layers of a pass in ONE launch.
//
// The tapes are slot-major (a slot's values for consecutive rows are contiguous), so a K-chunk of 64 rows of a layer's
// operands is n_in + n_out coalesced 256-byte reads.  A CTA takes (layer, a contiguous range of chunks): the chunk goes to
// shared memory (row stride 68 floats: conflict-free fragment loads) and is multiplied on the tensor cores (warp-level
// m16n8k8 TF32 MMAs, 3xTF32 split for fp32 accuracy); see tape_gemm_kernel.
// cuBLAS runs these shapes (M, N <= 64, K = 262 144) as sgemm_largek at ~320 us each, 26 per pass; the fp32 SIMT version of
// this kernel took 1.8 ms per pass (LDS/FMA bound).
#include "nr_train_math.cuh"

namespace nr {
namespace tg {

constexpr int MAXD = 48;
constexpr int KC = 64;       // rows (the contraction index) per chunk: half a tape tile
constexpr int LDK = KC + 4;  // shared-memory row stride: bank = (4 * operand row + k) mod 32, distinct for the 32 lanes of a fragment load
constexpr int MAXU = 9;      // m16n8 output tiles per warp: 4 x 18 tiles at most (64 outputs, 140 + 1 inputs) over 8 warps

struct Args {
  NrGemmDesc d[MAXD];
  const float* tape[4];      // 0 row tape, 1 row gradients, 2 point tape, 3 point gradients
  long long rows[4];
  int slots[4];
  float* out;
  int first_cta[MAXD + 1];   // CTAs [first_cta[l], first_cta[l+1]) work on layer l (shares proportional to the layer's cost)
  int n_desc;
};

__device__ __forceinline__ void cp_async4(float* dst, const float* src, bool valid) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
  const int n = valid ? 4 : 0;                                   // src-size 0: the destination is zero-filled
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(d), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async16(float* dst, const float* src) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// D (16x8, fp32) += A (16x8, tf32, row) * B (8x8, tf32, col) on the tensor cores (warp-level MMA)
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
// x = hi + lo, hi exact in tf32 (low 13 mantissa bits cleared), lo = x - hi exact in fp32
__device__ __forceinline__ void split(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}

// One CTA = (layer, contiguous range of 64-row chunks).  dW = dz * x^T is a GEMM whose contraction index is the ROW
// (K = 262 144 at the training shape) with at most 64 x 141 outputs, so it runs as warp-level tensor-core MMAs with the
// operands taken straight from the K-major tape chunks in shared memory:  A = dz [out][k],  B = x [in][k]  (both "row"
// of the tape = contiguous k), fp32-accurate through the 3xTF32 split (hi*hi + lo*hi + hi*lo) done on the fragments.
// A warp owns output tiles (16 outputs x 8 inputs) x a share of the chunk's eight k-steps; accumulators stay in registers
// over all chunks and are added to the result with atomics at the end.
__global__ void __launch_bounds__(256) tape_gemm_kernel(const __grid_constant__ Args a) {
  extern __shared__ __align__(16) float sm[];
  int layer = 0;
  while (layer + 1 < a.n_desc && int(blockIdx.x) >= a.first_cta[layer + 1]) ++layer;
  const int part = int(blockIdx.x) - a.first_cta[layer], parts = a.first_cta[layer + 1] - a.first_cta[layer];
  const NrGemmDesc& d = a.d[layer];
  const int n_in = d.n_in + 1, n_out = d.n_out;                  // + the constant-1 input (bias)
  const float* __restrict__ X = a.tape[d.x_tape] + (long long)d.x_slot * tr::TILE;      // + tile * slots * 128
  const float* __restrict__ Z = a.tape[d.g_tape] + (long long)d.g_slot * tr::TILE;
  const long long xt = (long long)a.slots[d.x_tape] * tr::TILE, zt = (long long)a.slots[d.g_tape] * tr::TILE;   // floats per tape tile
  const long long M = a.rows[d.x_tape];
  const int buf_floats = (n_in + n_out) * LDK;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t4 = lane & 3;
  const int mt_n = (n_out + 15) >> 4, nt_n = (n_in + 7) >> 3, tiles = mt_n * nt_n;
  // few tiles: split the chunk's 8 k-steps over the spare warps (ksplit = 1, 2, 4 or 8)
  int ksplit = 1;
  while (ksplit < 8 && tiles * ksplit * 2 <= 8) ksplit <<= 1;
  const int units = tiles * ksplit;
  float acc[MAXU][4];
#pragma unroll
  for (int u = 0; u < MAXU; ++u)
#pragma unroll
    for (int e = 0; e < 4; ++e) acc[u][e] = 0.f;
  // a CTA walks a contiguous range of 64-row chunks (sequential streams per operand slot), double buffered: the
  // cp.async copies of chunk c+1 are in flight while chunk c is multiplied
  const long long chunks = (M + KC - 1) / KC;
  const long long per = (chunks + parts - 1) / parts;
  const long long ch0 = (long long)part * per, ch_end = min(chunks, ch0 + per);
  auto stage = [&](long long ch, float* buf) {
    const long long tile = ch >> 1;
    const int half = int(ch & 1) * KC;
    const long long k0 = ch * KC;
    const int kn = int(M - k0 < KC ? M - k0 : KC);
    const float* __restrict__ xsrc = X + tile * xt + half;
    const float* __restrict__ zsrc = Z + tile * zt + half;
    if (kn == KC) {                                  // full chunk: 16-byte copies
      const int n = (n_in - 1 + n_out) * (KC / 4);
      for (int idx = threadIdx.x; idx < n; idx += 256) {
        const int row = idx / (KC / 4), k = (idx - row * (KC / 4)) * 4;
        const float* src = row < n_in - 1 ? xsrc + row * tr::TILE + k : zsrc + (row - (n_in - 1)) * tr::TILE + k;
        cp_async16(buf + (row < n_in - 1 ? row : row + 1) * LDK + k, src);                // row n_in - 1 is the constant input
      }
    } else {                                         // the last, partial chunk: element-wise with zero fill
      const int n = (n_in - 1 + n_out) * KC;
      for (int idx = threadIdx.x; idx < n; idx += 256) {
        const int row = idx / KC, k = idx - row * KC;
        const float* src = row < n_in - 1 ? xsrc + row * tr::TILE + k : zsrc + (row - (n_in - 1)) * tr::TILE + k;
        cp_async4(buf + (row < n_in - 1 ? row : row + 1) * LDK + k, src, k < kn);
      }
    }
  };
  for (int i = threadIdx.x; i < 2 * KC; i += 256) sm[(i / KC) * buf_floats + (n_in - 1) * LDK + (i % KC)] = 1.f;
  if (ch0 < ch_end) stage(ch0, sm);
  cp_async_commit();
  for (long long ch = ch0; ch < ch_end; ++ch) {
    float* buf = sm + int((ch - ch0) & 1) * buf_floats;
    if (ch + 1 < ch_end) stage(ch + 1, sm + int((ch - ch0 + 1) & 1) * buf_floats);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const float* xs = buf;                       // [n_in][LDK]
    const float* zs = buf + n_in * LDK;          // [n_out][LDK]
#pragma unroll
    for (int u = 0; u < MAXU; ++u) {
      const int unit = warp + 8 * u;
      if (unit < units) {                        // warp-uniform
        const int tile = unit / ksplit, kpart = unit - tile * ksplit;
        const int mt = tile / nt_n, nt = tile - mt * nt_n;
        // fragment rows, clamped into the operand (outputs beyond n_out / n_in are discarded at the end)
        const float* za = zs + min(16 * mt + g, n_out - 1) * LDK + t4;
        const float* zb = zs + min(16 * mt + g + 8, n_out - 1) * LDK + t4;
        const float* xb = xs + min(8 * nt + g, n_in - 1) * LDK + t4;
        // The tensor cores truncate their fp32 accumulator (about 1e-7 of the running sum per MMA, toward zero; see the
        // conv kernel in nr_encoder.cu).  Chained over every chunk of a CTA (up to ~4 100 MMAs at the training shape) that
        // lost 1.2e-4 of a same-sign sum (tests/test_backward_gpu.py, accuracy test).  So a chunk accumulates from zero and
        // is added to the running sum with a rounding FADD: 1.9e-6.
        float part[4] = {0.f, 0.f, 0.f, 0.f};
        for (int ks = kpart; ks < KC / 8; ks += ksplit) {
          const int k = 8 * ks;
          uint32_t ah[4], al[4], bh[2], bl[2];
          split(za[k], ah[0], al[0]); split(zb[k], ah[1], al[1]); split(za[k + 4], ah[2], al[2]); split(zb[k + 4], ah[3], al[3]);
          split(xb[k], bh[0], bl[0]); split(xb[k + 4], bh[1], bl[1]);
          mma_tf32(part, al, bh);
          mma_tf32(part, ah, bl);
          mma_tf32(part, ah, bh);
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[u][e] += part[e];
      }
    }
    __syncthreads();                             // the buffer is refilled by the prefetch of the iteration after next
  }
  float* out = a.out + d.out_off;
#pragma unroll
  for (int u = 0; u < MAXU; ++u) {
    const int unit = warp + 8 * u;
    if (unit < units) {
      const int tile = unit / ksplit;
      const int mt = tile / nt_n, nt = tile - mt * nt_n;
      // accumulator layout of m16n8: c0 (g, 2 t4), c1 (g, 2 t4 + 1), c2 (g + 8, 2 t4), c3 (g + 8, 2 t4 + 1)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int o = 16 * mt + g + (e >> 1) * 8, i = 8 * nt + 2 * t4 + (e & 1);
        if (o < n_out && i < n_in) atomicAdd(out + o * n_in + i, acc[u][e]);
      }
    }
  }
}

}  // namespace tg
}  // namespace nr

extern "C" int nr_tape_gemms(const NrGemmDesc* descs, int n_desc, const float* tape_row, const float* grad_row, long long rows,
                             const float* tape_point, const float* grad_point, long long points, float* out, void* stream) {
  using namespace nr;
  NR_CHECK_ARG(descs != nullptr && n_desc >= 1 && n_desc <= tg::MAXD, "descriptor count");
  NR_CHECK_ARG(tape_row && grad_row && tape_point && grad_point && out, "null device pointer");
  tg::Args a;
  int max_rows = 0;
  for (int i = 0; i < n_desc; ++i) {
    const NrGemmDesc& d = descs[i];
    NR_CHECK_ARG(d.n_out >= 1 && d.n_out <= 64 && d.n_in >= 1 && d.n_in <= 140 && d.x_tape >= 0 && d.x_tape < 4 && d.g_tape >= 0 && d.g_tape < 4,
                 "descriptor");
    NR_CHECK_ARG(((d.n_out + 15) / 16) * ((d.n_in + 8) / 8) <= tg::MAXU * 8, "layer too large");
    a.d[i] = d;
    if (d.n_in + 1 + d.n_out > max_rows) max_rows = d.n_in + 1 + d.n_out;
  }
  a.tape[0] = tape_row; a.tape[1] = grad_row; a.tape[2] = tape_point; a.tape[3] = grad_point;
  a.rows[0] = rows; a.rows[1] = rows; a.rows[2] = points; a.rows[3] = points;
  a.slots[0] = tr::R_SLOTS; a.slots[1] = tr::G_SLOTS; a.slots[2] = tr::P_SLOTS; a.slots[3] = tr::GP_SLOTS;
  a.out = out;
  const size_t smem = 2 * size_t(max_rows) * tg::LDK * sizeof(float);     // two chunk buffers
  if (smem > 48 * 1024)   // per-device attribute, set per launch: no per-process state
    cudaFuncSetAttribute(tg::tape_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
  // CTAs per layer in proportion to its cost (bytes staged + MMAs issued per chunk), so that the 64 x 141 layers do not
  // leave a tail behind the 1 x 9 ones: ~8 CTAs per SM in total, every layer at least one
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  double cost[tg::MAXD], total = 0.0;
  for (int i = 0; i < n_desc; ++i) {
    const NrGemmDesc& d = descs[i];
    const double tiles = double((d.n_out + 15) / 16) * double((d.n_in + 8) / 8);
    cost[i] = double(a.rows[d.x_tape]) * (double(d.n_in + d.n_out) + 6.0 * tiles);
    total += cost[i];
  }
  const int target = sms * 8;
  a.n_desc = n_desc;
  a.first_cta[0] = 0;
  for (int i = 0; i < n_desc; ++i) {
    const long long chunks = (a.rows[descs[i].x_tape] + tg::KC - 1) / tg::KC;
    long long n = (long long)(target * cost[i] / (total > 0 ? total : 1.0) + 0.5);
    if (n > chunks) n = chunks;
    if (n < 1) n = 1;
    a.first_cta[i + 1] = a.first_cta[i] + int(n);
  }
  tg::tape_gemm_kernel<<<a.first_cta[n_desc], 256, smem, (cudaStream_t)stream>>>(a);
  NR_CHECK_LAUNCH("tape_gemms");
  return NR_OK;
}
