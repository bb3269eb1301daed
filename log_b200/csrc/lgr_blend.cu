// Per-tile front-to-back alpha compositing (forward) and the gradient sweep (backward).
//
// One CTA of 256 threads per 16x16 tile; warp w owns the 8x4 pixel sub-tile ((w&1)*8, (w>>1)*4), one pixel per
// lane.  The tile's depth-sorted list is staged through shared memory 256 splats at a time (coalesced id read,
// 3 x 16-byte gather per splat, 48-byte staged record).  The staging thread also tests its splat's conservative
// alpha>=1/255 box against the eight sub-tiles and publishes one byte of hit bits, so a warp finds its hits among 32
// staged splats with one byte load and a ballot, and only walks the hits (lane = pixel, broadcast LDS).  With small
// splats this skips ~90 % of the (pixel, splat) pairs the classic per-thread loop evaluates.
// Backward: the same front-to-back walk (closed form of the published recurrence, see below).  Per contributing hit every
// lane publishes two scalars; every 8 hits the warp contracts them against fixed per-pixel weights (pixel-coordinate
// moments and cotangent-weighted sums) on the tensor cores (mma.sync m16n8k8, split TF32 = fp32 accuracy); the moments
// become gradients right after each contraction, then 3 vector atomics per (warp, hit).  With View::contrib the forward records which
// sub-tiles composited each list entry and the backward (REC) walks exactly those pairs, stopping every pixel after its
// last contributor (the forward's n_contrib) instead of re-testing boxes and transmittances.
#include "lgr_common.cuh"
#include "lgr_prof.cuh"

namespace lgr {

constexpr int BLEND_THREADS = TILE_PIX;   // 256
// minimum resident CTAs per SM the compiler must make room for (register cap = 65536 / (256 * N)); measured, see DESIGN.md
#ifndef LGR_FWD_MIN_CTAS
#define LGR_FWD_MIN_CTAS 5
#endif
#ifndef LGR_BWD_MIN_CTAS
#define LGR_BWD_MIN_CTAS 4
#endif
constexpr int BATCH = 256;
constexpr unsigned FULL = 0xffffffffu;

struct SubTile {
  int x, y;          // this lane's pixel
  bool inside;
};

__device__ __forceinline__ SubTile make_subtile(const View& v, int tile, int lane, int warp) {
  SubTile s;
  const int tx = tile % v.gx, ty = v.row0 + tile / v.gx;
  const int sx = tx * TILE + (warp & 1) * 8, sy = ty * TILE + (warp >> 1) * 4;
  s.x = sx + (lane & 7); s.y = sy + (lane >> 3);
  s.inside = s.x < v.W && s.y < v.H;
  return s;
}

// Which of the tile's eight 8x4 sub-tiles (bit w = warp w) can the conservative {alpha >= 1/255} box of a splat reach?
// (tx0, ty0) = pixel coordinates of the tile's corner.  Conservative (never misses a contributing pair), so skipping on
// it never changes a result.
__device__ __forceinline__ unsigned subtile_bits(const float4 r0, const float4 r1, float tx0, float ty0) {
  const float xlo = r0.x - r1.z, xhi = r0.x + r1.z, ylo = r0.y - r1.w, yhi = r0.y + r1.w;
  unsigned xm = 0u, m = 0u;
  if (xhi >= tx0 && xlo <= tx0 + 7.0f) xm |= 1u;
  if (xhi >= tx0 + 8.0f && xlo <= tx0 + 15.0f) xm |= 2u;
#pragma unroll
  for (int r = 0; r < 4; r++)
    if (yhi >= ty0 + 4.0f * r && ylo <= ty0 + 4.0f * r + 3.0f) m |= xm << (2 * r);
  return m;
}

// The skip decisions (power > 0, alpha < 1/255, T < 1e-4) must come out IDENTICAL in the forward and the backward
// kernel (the backward re-walks the list front to back and must stop where the forward stopped).  Explicitly rounded
// intrinsics are never contracted or re-associated, so both kernels execute the same arithmetic.
// The conic in the splat record is pre-multiplied by log2(e): alpha = o * 2^(power2).
__device__ __forceinline__ float eval_power2(const float4 r0, const float con_z, float dx, float dy) {
  const float q = __fmaf_rn(r0.z, __fmul_rn(dx, dx), __fmul_rn(con_z, __fmul_rn(dy, dy)));   // cx dx^2 + cz dy^2
  return __fmaf_rn(-0.5f, q, -__fmul_rn(r0.w, __fmul_rn(dx, dy)));
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float eval_alpha(float opacity, float G) { return fminf(ALPHA_MAX, __fmul_rn(opacity, G)); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float2 lds_f2(uint32_t addr) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
  return v;
}
// keep a shared-window address in a register (the compiler otherwise rebuilds it from SR_CgaCtaId inside hot loops)
__device__ __forceinline__ uint32_t pin_reg(uint32_t v) {
  asm volatile("" : "+r"(v));
  return v;
}
__device__ __forceinline__ void red_shared_max_u32(uint32_t addr, unsigned v) {
  asm volatile("red.shared.max.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void sts_f32(uint32_t addr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// pull the 128-byte line(s) of a record the NEXT batch will gather into L2 while this batch is walked
__device__ __forceinline__ void prefetch_l2(const float* p) {
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}
// TF32 split of an fp32 value.  The tensor core reads only sign, exponent and the upper 10 mantissa bits of a .tf32
// operand, i.e. it multiplies with trunc(x) when handed the raw fp32 bits; tf32_lo(x) = x - trunc(x) is exact in fp32 and
// |lo| < 2^-10 |x|, so trunc(x) + trunc(lo) carries x to ~2^-20 relative.  (cvt.rna.tf32 costs 4 SASS instructions per
// value on sm_100a -- a range check, an integer add, a select and a mask; this is one LOP3 and one FADD.)
__device__ __forceinline__ float tf32_lo(float x) { return x - __uint_as_float(__float_as_uint(x) & 0xffffe000u); }
// Four 8x8 b16 matrices = four blocks of 8 rows x 4 fp32: lane l supplies the address of row l%8 of block l/8 and
// receives, per block, the fp32 at (row l/4, column l%4) -- exactly the B fragment of mma.m16n8k8.tf32 when a row is
// one hit and the columns are pixels.
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
// D(16x8) += A(16x8, row) * B(8x8, col), TF32 inputs, fp32 accumulate.  Lane (g = l/4, t = l%4) holds
// a0 = A[g][t], a1 = A[g+8][t], a2 = A[g][t+4], a3 = A[g+8][t+4];  b0 = B[t][g], b1 = B[t+4][g];
// d0 = D[g][2t], d1 = D[g][2t+1], d2 = D[g+8][2t], d3 = D[g+8][2t+1].
__device__ __forceinline__ void mma_tf32(float& d0, float& d1, float& d2, float& d3, uint32_t a0, uint32_t a1, uint32_t a2,
                                         uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d0), "+f"(d1), "+f"(d2), "+f"(d3) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// Staged splat: three consecutive float4 per list entry (48-byte stride: conflict-free for 128-bit accesses),
//   [0] = (px, py, conic_x', conic_y')   [1] = (conic_z', opacity, hx, hy)   [2] = (r, g, b, id as int bits)
// plus one byte of sub-tile hit bits.
// recorded: the entry's byte of View::contrib (backward, when the forward recorded which sub-tiles composited it) or nullptr
__device__ __forceinline__ void stage_splat(float4* s_rec, unsigned char* s_bits, int slot, const float* __restrict__ splat,
                                            int id, float tx0, float ty0, const uint8_t* __restrict__ recorded = nullptr) {
  const float* rec = splat + (int64_t)id * LGR_SPLAT_FLOATS;
  const float4 r0 = ldg4(rec), r1 = ldg4(rec + 4);
  float4 r2 = ldg4(rec + 8);
  r2.w = __int_as_float(id);
  s_rec[3 * slot] = r0; s_rec[3 * slot + 1] = r1; s_rec[3 * slot + 2] = r2;
  s_bits[slot] = recorded ? *recorded : (unsigned char)subtile_bits(r0, r1, tx0, ty0);
}

// ---------------------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------------------
// REC: also record, per tile-list entry, the sub-tiles that composited it (View::contrib), for the backward
template <bool AUX, bool REC>
__global__ void __launch_bounds__(BLEND_THREADS, LGR_FWD_MIN_CTAS)
blend_fwd_kernel(View v, const int32_t* __restrict__ tile_start, const int32_t* __restrict__ sorted_ids,
                 const float* __restrict__ splat, float* __restrict__ image, float* __restrict__ final_T,
                 int32_t* __restrict__ n_contrib, int32_t* __restrict__ pid_pixel, float* __restrict__ pw_pixel,
                 unsigned* __restrict__ point_weight_bits, int32_t* __restrict__ point_count) {
  __shared__ float4 s_rec[BATCH * 3];
  __shared__ unsigned s_w[AUX ? BATCH : 1];
  __shared__ unsigned char s_bits[BATCH];
  __shared__ unsigned s_cb[REC ? (BLEND_THREADS / 32) * (BATCH / 32) : 1];      // per warp: bit e = a pixel of this warp took staged splat e
  const int tile = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const SubTile st = make_subtile(v, tile, lane, warp);
  const float pxf = (float)st.x, pyf = (float)st.y;
  const float tx0 = (float)((tile % v.gx) * TILE), ty0 = (float)((v.row0 + tile / v.gx) * TILE);
  const int beg = tile_start[tile], len = tile_start[tile + 1] - beg;
  const uint32_t s_w_addr = smem_u32(s_w);
  const uint32_t s_rec_addr = pin_reg(smem_u32(s_rec));

  float T = 1.0f, C0 = 0.f, C1 = 0.f, C2 = 0.f, wmax = 0.f;
  int last = 0, wid = -1;
  int done = st.inside ? 0 : 1;
  int id_next = tid < len ? sorted_ids[beg + tid] : -1;

  // Two barriers per batch.  A thread stages, flushes and re-stages only ITS OWN slot (record tid, hit bits tid, aux word
  // tid), so the flush of batch b and the staging of batch b+1 need no barrier between them:
  //     stage(0) | A | walk(0) | B | flush(0), stage(1) | A | walk(1) | B | ...
  int base = 0, cnt = min(BATCH, len);
  auto stage = [&]() {
    if (tid < cnt) stage_splat(s_rec, s_bits, tid, splat, id_next, tx0, ty0);
    else s_bits[tid] = 0;
    if (AUX) s_w[tid] = 0u;
    id_next = base + BATCH + tid < len ? sorted_ids[beg + base + BATCH + tid] : -1;
    if (id_next >= 0) prefetch_l2(splat + (int64_t)id_next * LGR_SPLAT_FLOATS);
  };
  if (len > 0) stage();
  while (base < len) {
    __syncthreads();                         // A: the batch is staged
    if (REC) {      // a warp owns its BATCH/32 words of s_cb: cleared here, written below, read by others only after B
      if (lane < BATCH / 32) s_cb[warp * (BATCH / 32) + lane] = 0u;
      __syncwarp();
    }
    if (!__all_sync(FULL, done)) {
      for (int c0 = 0; c0 < cnt; c0 += 32) {
        const int e_l = c0 + lane;
        unsigned mask = __ballot_sync(FULL, (s_bits[e_l] >> warp) & 1u);
        unsigned own_w = 0u;                 // max weight of the splat this lane tested, over this warp's pixels
        unsigned took = 0u;                  // bit j: some pixel of this warp composited staged splat c0 + j
        while (mask) {
          // two hits per iteration: loads and alpha evaluation of both overlap, the transmittance updates are sequential
          const int jA = __ffs(mask) - 1;
          mask &= mask - 1;
          const bool two = mask != 0u;
          const int jB = two ? __ffs(mask) - 1 : jA;
          mask &= mask - 1;
          const uint32_t recA = s_rec_addr + 48u * (uint32_t)(c0 + jA), recB = s_rec_addr + 48u * (uint32_t)(c0 + jB);
          const float4 r0A = lds_f4(recA), r0B = lds_f4(recB);
          const float2 r1A = lds_f2(recA + 16u), r1B = lds_f2(recB + 16u);                  // (conic_z, opacity)
          const float dxA = __fsub_rn(r0A.x, pxf), dyA = __fsub_rn(r0A.y, pyf);
          const float dxB = __fsub_rn(r0B.x, pxf), dyB = __fsub_rn(r0B.y, pyf);
          const float powerA = eval_power2(r0A, r1A.x, dxA, dyA), powerB = eval_power2(r0B, r1B.x, dxB, dyB);
          const float alphaA = eval_alpha(r1A.y, ex2_approx(powerA)), alphaB = eval_alpha(r1B.y, ex2_approx(powerB));
          float wA = 0.f, wB = 0.f;
          if (!done && powerA <= 0.0f && alphaA >= ALPHA_MIN) {
            const float test_T = __fmul_rn(T, __fsub_rn(1.0f, alphaA));
            if (test_T < T_STOP) done = 1;
            else {
              wA = alphaA * T;
              const float4 r2 = lds_f4(recA + 32u);
              C0 = fmaf(r2.x, wA, C0); C1 = fmaf(r2.y, wA, C1); C2 = fmaf(r2.z, wA, C2);
              T = test_T;
              last = base + c0 + jA + 1;
              if (AUX && wA > wmax) { wmax = wA; wid = __float_as_int(r2.w); }
            }
          }
          if (two && !done && powerB <= 0.0f && alphaB >= ALPHA_MIN) {
            const float test_T = __fmul_rn(T, __fsub_rn(1.0f, alphaB));
            if (test_T < T_STOP) done = 1;
            else {
              wB = alphaB * T;
              const float4 r2 = lds_f4(recB + 32u);
              C0 = fmaf(r2.x, wB, C0); C1 = fmaf(r2.y, wB, C1); C2 = fmaf(r2.z, wB, C2);
              T = test_T;
              last = base + c0 + jB + 1;
              if (AUX && wB > wmax) { wmax = wB; wid = __float_as_int(r2.w); }
            }
          }
          if (AUX) {
            const unsigned mA = __reduce_max_sync(FULL, __float_as_uint(wA));   // w >= 0: uint order == float order
            const unsigned mB = __reduce_max_sync(FULL, __float_as_uint(wB));
            if (lane == jA) own_w = mA;
            if (two && lane == jB) own_w = mB;
          } else if (REC) {
            if (__any_sync(FULL, wA != 0.f)) took |= 1u << jA;
            if (__any_sync(FULL, wB != 0.f)) took |= 1u << jB;
          }
        }
        // fork flavour: the lane that staged a splat holds its max weight over this warp's pixels; non-zero <=> composited here
        // (a composited pixel has w = alpha T >= 1/255 * 1e-4 > 0): one ballot per 32 staged splats
        if (AUX && REC) took = __ballot_sync(FULL, own_w != 0u);
        if (REC && lane == 0) s_cb[warp * (BATCH / 32) + (c0 >> 5)] = took;
        if (AUX && own_w) red_shared_max_u32(s_w_addr + 4u * e_l, own_w);
        if (__all_sync(FULL, done)) break;
      }
    }
    const int all_done = __syncthreads_and(done);      // B: every warp has left the walk
    if (AUX && tid < cnt && s_w[tid]) atomicMax(point_weight_bits + __float_as_int(s_rec[3 * tid + 2].w), s_w[tid]);
    if (REC && tid < cnt) {      // for the backward: which sub-tiles composited this list entry
      unsigned byte = 0u;
#pragma unroll
      for (int w = 0; w < BLEND_THREADS / 32; w++) byte |= ((s_cb[w * (BATCH / 32) + (tid >> 5)] >> (tid & 31)) & 1u) << w;
      v.contrib[beg + base + tid] = (uint8_t)byte;
    }
    base += BATCH;
    if (all_done || base >= len) break;
    cnt = min(BATCH, len - base);
    stage();
  }
  if (st.inside) {
    const int64_t pix = (int64_t)st.y * v.W + st.x, HW = (int64_t)v.H * v.W;
    image[pix] = C0 + T * __ldg(v.bg);
    image[HW + pix] = C1 + T * __ldg(v.bg + 1);
    image[2 * HW + pix] = C2 + T * __ldg(v.bg + 2);
    final_T[pix] = T;
    n_contrib[pix] = last;
    if (AUX) {
      pid_pixel[pix] = (v.pid_map && wid >= 0) ? v.pid_map[wid] : wid; pw_pixel[pix] = wmax;
      if (point_count && wid >= 0) atomicAdd(point_count + wid, 1);      // histogram of the per-pixel winners
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------------------
// The sweep runs FRONT TO BACK, exactly like the forward: T_j comes from the same multiplications (no division
// chain).  With R_j = sum_c dL/dC_c * (colour of everything from splat j on, incl. bg T_final) -- a scalar that starts at
// sum_c dL/dC_c * pixel_c and loses (c_j . dL/dC) a_j T_j at every contributing splat --
//   dL/da_j = (c_j . dL/dC) T_j - R_{j+1} / (1 - a_j)
// which is the published back-to-front recurrence written in closed form.
//
// Reduction over the warp's pixels.  Every one of the 9 per-splat outputs is a FIXED-weight linear functional of two
// per-lane scalars of the hit, wG = dL/dG * G and w = alpha * T:
//     M00, M10, M01, M20, M11, M02 = sum_l wG_l * {1, u, v, u^2, uv, v^2}_l      (u, v: pixel coordinates about the warp's sub-tile centre)
//     C0, C1, C2                   = sum_l w_l * dL/dC_{0,1,2; l}
// i.e. a [hits x 32] x [32 x 9] contraction.  Each lane publishes (wG, w) of a contributing hit as one row element of two
// [8 hits][32 pixels] shared-memory blocks; when 8 hits are pending (or the batch ends) the warp runs the contraction
// on the tensor cores: A (16 rows = 8 wG rows + 8 w rows) straight from the blocks with ldmatrix, B = the weights (moment
// weights are quarter-integers, |u^2| <= 12.25: exact in TF32; the cotangent weights are split hi + lo once per
// kernel), every A value split hi + lo, fp32 accumulation -- 8 + 12 mma.m16n8k8 per 8 hits, error ~2^-20 relative.
// Right after the contraction the 4 lanes of hit g's fragment group gather its 9 sums with 4 shuffles, turn the moments
// into d/dmean2D, d/dconic, d/dopacity (X = splat centre in the same coordinates):
//     sum wG dx = X M00 - M10,   sum wG dx^2 = X^2 M00 - 2 X M10 + M20,   sum wG dx dy = XY M00 - X M01 - Y M10 + M11 ...
// and add them into dsplat with one vector atomic each (fire-and-forget RED, no shared-memory accumulators).
constexpr int HITS = 8;          // hits per contraction (half the m of mma.m16n8k8: 8 wG rows + 8 w rows)
constexpr int XROW = 36;         // floats per published row: 32 pixels + 4 pad, so the 8 rows of an ldmatrix block hit 8 bank groups
constexpr int BWD_SMEM = BATCH * 48 + (BLEND_THREADS / 32) * (2 * HITS * XROW + 192 + 192) * 4 + BATCH;
static_assert(BWD_SMEM <= 48 * 1024, "the backward launches without the large-shared-memory opt-in");

// REC: the forward recorded (View::contrib) which sub-tiles composited each list entry and (View::last_contrib = its
// n_contrib output) where every pixel's last contributor sits; the sweep then meets exactly the contributing (sub-tile,
// splat) pairs and a pixel is finished once the walk has passed its last contributor -- no box tests, no T < 1e-4 test.
template <bool REC>
__global__ void __launch_bounds__(BLEND_THREADS, LGR_BWD_MIN_CTAS)
blend_bwd_kernel(View v, const int32_t* __restrict__ tile_start, const int32_t* __restrict__ sorted_ids,
                 const float* __restrict__ splat, const float* __restrict__ image,
                 const float* __restrict__ dL_dimage, float* __restrict__ dsplat) {
  extern __shared__ float4 smem_f4[];
  float4* s_rec = smem_f4;                                                        // [BATCH * 3]
  float* s_x = reinterpret_cast<float*>(s_rec + BATCH * 3);                       // per warp: wG[8][36] | w[8][36]
  float* s_cw = s_x + (BLEND_THREADS / 32) * 2 * HITS * XROW;                     // per warp: cotangent weights, B-fragment order
  float* s_mw = s_cw + (BLEND_THREADS / 32) * 192;                                // per warp: moment weights, B-fragment order
  unsigned char* s_bits = reinterpret_cast<unsigned char*>(s_mw + (BLEND_THREADS / 32) * 192);      // [BATCH]
  const int tile = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const SubTile st = make_subtile(v, tile, lane, warp);
  const float pxf = (float)st.x, pyf = (float)st.y;
  const float tx0 = (float)((tile % v.gx) * TILE), ty0 = (float)((v.row0 + tile / v.gx) * TILE);
  const int beg = tile_start[tile], len = tile_start[tile + 1] - beg;
  const uint32_t s_rec_addr = pin_reg(smem_u32(s_rec));
  const uint32_t xg_addr = pin_reg(smem_u32(s_x) + (uint32_t)warp * (2 * HITS * XROW * 4));
  const uint32_t xlane_addr = pin_reg(xg_addr + 4u * (uint32_t)lane);
  // ldmatrix row address of this lane: row lane%8 of block lane/8; blocks = (wG, chunk 2s), (w, chunk 2s), (wG, chunk 2s+1), (w, chunk 2s+1)
  const uint32_t xrow = pin_reg(xg_addr + (uint32_t)(lane & 7) * (XROW * 4) + (uint32_t)((lane >> 3) & 1) * (HITS * XROW * 4) +
                                (uint32_t)(lane >> 4) * 16u);
  const float ucx = (warp & 1) * 8 + 3.5f, ucy = (warp >> 1) * 4 + 1.5f;   // moment origin: this warp's sub-tile centre
  const float tcx = tx0 + ucx, tcy = ty0 + ucy;
  const int g = lane >> 2, t = lane & 3;        // mma fragment coordinates of this lane

  float Rd = 0.f, dp0 = 0.f, dp1 = 0.f, dp2 = 0.f;
  int last = 0;                                  // REC: list index + 1 of this pixel's last contributor (0: none)
  if (st.inside) {
    const int64_t pix = (int64_t)st.y * v.W + st.x, HW = (int64_t)v.H * v.W;
    dp0 = dL_dimage[pix]; dp1 = dL_dimage[HW + pix]; dp2 = dL_dimage[2 * HW + pix];
    Rd = image[pix] * dp0 + image[HW + pix] * dp1 + image[2 * HW + pix] * dp2;
    if (REC) last = v.last_contrib[pix];
  }
  // B fragments of the weights, per warp in shared memory, lane-major per k-step so that the load of k-step s reads
  // consecutive addresses (one LDS.64 / LDS.128 over 192 bytes).  Only the lanes of the used columns have an entry:
  // g < 6 (lanes 0..23) for the moments, g < 3 (lanes 0..11) for the cotangents.  The other lanes load the last entry
  // again (a broadcast, no extra wavefront, no branch): it lands in D columns that are never read (moments 6, 7 of t = 3;
  // colour columns >= 3).
  // Moments: s_mw[(s*24 + lane)*2 + {0,1}] = weight of output g at the pixel of k-step s with k = t (column t, row s of the
  // sub-tile) / k = t + 4 (column t + 4).  Multiples of 0.25, |values| <= 12.25: exact in TF32.
  const uint32_t mw_addr = pin_reg(smem_u32(s_mw) + (uint32_t)warp * (192 * 4) + (uint32_t)min(lane, 23) * 8u);
  for (int k = lane; k < 192; k += 32) {
    const int which = k & 1, s_ = (k >> 1) / 24, l_ = (k >> 1) % 24, t_ = l_ & 3, g_ = l_ >> 2;
    const float u = (float)((warp & 1) * 8 + t_ + 4 * which) - ucx, vv = (float)((warp >> 1) * 4 + s_) - ucy;
    const float f = g_ == 0 ? 1.f : g_ == 1 ? u : g_ == 2 ? vv : g_ == 3 ? u * u : g_ == 4 ? u * vv : vv * vv;
    s_mw[warp * 192 + k] = f;
  }
  // Cotangents (columns 0..2 = channel): s_cw[(s*12 + c*4 + t)*4 + {0,1,2,3}] = hi(k=t), hi(k=t+4), lo(k=t), lo(k=t+4)
  const uint32_t cw_addr = pin_reg(smem_u32(s_cw) + (uint32_t)warp * (192 * 4) + (uint32_t)min(lane, 11) * 16u);
  {
    float* cw = s_cw + warp * 192;
    const int col = lane & 7, s = lane >> 3, tt = col & 3, which = col >> 2;
    const float dpc[3] = {dp0, dp1, dp2};
#pragma unroll
    for (int c = 0; c < 3; c++) {
      cw[(s * 12 + c * 4 + tt) * 4 + which] = dpc[c];                  // read as trunc(x) by the tensor core
      cw[(s * 12 + c * 4 + tt) * 4 + 2 + which] = tf32_lo(dpc[c]);
    }
  }
  __syncwarp();

  float T = 1.0f;
  int done = st.inside ? (REC ? (last == 0) : 0) : 1;
  int id_next = tid < len ? sorted_ids[beg + tid] : -1;

  // Two barriers per batch: A (the batch is staged) and B (every warp has left the walk, so slot tid may be re-staged).
  // Thread tid stages only slot tid (record and hit bits).
  int base = 0, cnt = min(BATCH, len);
  auto stage = [&]() {
    if (tid < cnt) {
      // with View::contrib: walk exactly the (sub-tile, splat) pairs that composited something in the forward
      stage_splat(s_rec, s_bits, tid, splat, id_next, tx0, ty0, REC ? v.contrib + beg + base + tid : nullptr);
    } else {
      s_bits[tid] = 0;
    }
    id_next = base + BATCH + tid < len ? sorted_ids[beg + base + BATCH + tid] : -1;
    if (id_next >= 0) prefetch_l2(splat + (int64_t)id_next * LGR_SPLAT_FLOATS);
  };
  if (len > 0) stage();
  while (base < len) {
    __syncthreads();                         // A: the batch is staged
    if (!__all_sync(FULL, done)) {
      int c0 = -32, pend = 0, my_e = 0;
      unsigned mask = 0u;
      bool fin = false;
      while (true) {
        if (mask == 0u) {      // next group of 32 staged splats with a hit
          do {
            c0 += 32;
            fin = c0 >= cnt || __all_sync(FULL, done);
            if (fin) break;
            mask = __ballot_sync(FULL, (s_bits[c0 + lane] >> warp) & 1u);
          } while (mask == 0u);
        }
        if (!fin) {
          // Two hits per iteration: their loads and the evaluation of alpha are independent and overlap; only the
          // transmittance / colour-behind updates are sequential (A before B).
          const int jA = __ffs(mask) - 1;
          mask &= mask - 1;
          const bool two = mask != 0u;
          const int jB = two ? __ffs(mask) - 1 : jA;
          mask &= mask - 1;
          const int eA = c0 + jA, eB = c0 + jB;
          const uint32_t recA = s_rec_addr + 48u * (uint32_t)eA, recB = s_rec_addr + 48u * (uint32_t)eB;
          const float4 r0A = lds_f4(recA), r0B = lds_f4(recB);
          const float2 r1A = lds_f2(recA + 16u), r1B = lds_f2(recB + 16u);                  // (conic_z, opacity)
          const float dxA = __fsub_rn(r0A.x, pxf), dyA = __fsub_rn(r0A.y, pyf);
          const float dxB = __fsub_rn(r0B.x, pxf), dyB = __fsub_rn(r0B.y, pyf);
          const float powerA = eval_power2(r0A, r1A.x, dxA, dyA), powerB = eval_power2(r0B, r1B.x, dxB, dyB);
          const float GA = ex2_approx(powerA), GB = ex2_approx(powerB);
          const float alphaA = eval_alpha(r1A.y, GA), alphaB = eval_alpha(r1B.y, GB);
          const float omA = __fsub_rn(1.0f, alphaA), omB = __fsub_rn(1.0f, alphaB);
          bool cA = false, cB = false;
          const float TA = T;
          float TB;
          if (REC) {
            // every visited splat in front of the pixel's last contributor with alpha >= 1/255 was composited by the forward
            // (it would otherwise have stopped the pixel there); same multiplications, so T follows the forward bit for bit
            cA = !done && powerA <= 0.0f && alphaA >= ALPHA_MIN;
            if (cA) T = __fmul_rn(T, omA);
            done = (base + eA + 1 >= last);
            TB = T;
            cB = two && !done && powerB <= 0.0f && alphaB >= ALPHA_MIN;
            if (cB) T = __fmul_rn(T, omB);
            if (two) done = (base + eB + 1 >= last);
          } else {
            if (!done && powerA <= 0.0f && alphaA >= ALPHA_MIN) {
              const float tt = __fmul_rn(T, omA);
              if (tt < T_STOP) done = 1; else { cA = true; T = tt; }
            }
            TB = T;
            if (two && !done && powerB <= 0.0f && alphaB >= ALPHA_MIN) {
              const float tt = __fmul_rn(T, omB);
              if (tt < T_STOP) done = 1; else { cB = true; T = tt; }
            }
          }
          const bool anyA = __any_sync(FULL, cA), anyB = __any_sync(FULL, cB);
          if (anyA) {
            float wG = 0.f, w = 0.f;
            if (cA) {
              const float4 r2 = lds_f4(recA + 32u);
              w = alphaA * TA;
              const float cdot = r2.x * dp0 + r2.y * dp1 + r2.z * dp2;
              Rd = fmaf(-cdot, w, Rd);                          // what is behind the splat (+ bg T_final), dotted with dL/dC
              const float dL_dalpha = cdot * TA - Rd * rcp_approx(omA);
              wG = r1A.y * dL_dalpha * GA;                      // dL/dG * G   (the 0.99 clamp is straight-through)
            }
            const uint32_t row = xlane_addr + (uint32_t)pend * (XROW * 4);
            sts_f32(row, wG); sts_f32(row + HITS * XROW * 4, w);
            if (lane == pend) my_e = eA;
            pend++;
          }
          if (anyB) {
            float wG = 0.f, w = 0.f;
            if (cB) {
              const float4 r2 = lds_f4(recB + 32u);
              w = alphaB * TB;
              const float cdot = r2.x * dp0 + r2.y * dp1 + r2.z * dp2;
              Rd = fmaf(-cdot, w, Rd);
              const float dL_dalpha = cdot * TB - Rd * rcp_approx(omB);
              wG = r1B.y * dL_dalpha * GB;
            }
            const uint32_t row = xlane_addr + (uint32_t)pend * (XROW * 4);
            sts_f32(row, wG); sts_f32(row + HITS * XROW * 4, w);
            if (lane == pend) my_e = eB;
            pend++;
          }
        }
        if (pend >= HITS - 1 || (fin && pend > 0)) {      // fewer than two free rows, or the batch is over
          // ---- contract the pending hits on the tensor cores ----
          // A (16 x 32 pixels): rows 0..7 = wG of the 8 hits, rows 8..15 = w of the same hits; one ldmatrix.x4 per k-step
          // delivers (a0, a1, a2, a3) in place.  B (32 pixels x 8): the weights -- Bm moments (6 columns, exact), Bc the
          // cotangents (3 columns, hi + lo).  D1 = A Bm (rows 0..7 used), D2 = A Bc (rows 8..15 used): two independent chains.
          __syncwarp();
          float d0 = 0.f, d1 = 0.f, z0 = 0.f, z1 = 0.f, y0 = 0.f, y1 = 0.f, d2 = 0.f, d3 = 0.f;
#pragma unroll
          for (int s = 0; s < 4; s++) {
            uint32_t a0, a1, a2, a3;
            ldsm_x4(xrow + 32u * s, a0, a1, a2, a3);
            const uint32_t l0 = __float_as_uint(tf32_lo(__uint_as_float(a0))), l1 = __float_as_uint(tf32_lo(__uint_as_float(a1)));
            const uint32_t l2 = __float_as_uint(tf32_lo(__uint_as_float(a2))), l3 = __float_as_uint(tf32_lo(__uint_as_float(a3)));
            const float2 bm = lds_f2(mw_addr + 192u * s);
            const float4 bc = lds_f4(cw_addr + 192u * s);
            mma_tf32(d0, d1, z0, z1, a0, a1, a2, a3, __float_as_uint(bm.x), __float_as_uint(bm.y));
            mma_tf32(y0, y1, d2, d3, a0, a1, a2, a3, __float_as_uint(bc.x), __float_as_uint(bc.y));
            mma_tf32(d0, d1, z0, z1, l0, l1, l2, l3, __float_as_uint(bm.x), __float_as_uint(bm.y));
            mma_tf32(y0, y1, d2, d3, l0, l1, l2, l3, __float_as_uint(bc.x), __float_as_uint(bc.y));
            mma_tf32(y0, y1, d2, d3, a0, a1, a2, a3, __float_as_uint(bc.z), __float_as_uint(bc.w));
          }
          // lane (g, t): d0/d1 = moments 2t, 2t+1 of hit g (t < 3) ; d2/d3 = colour sums 2t, 2t+1 of hit g (t = 0: 0, 1; t = 1: 2)
          const int e = __shfl_sync(FULL, my_e, g);
          // Gather within the lane group, 4 shuffles: t = 0 (d/dmean2D, d/dconic_xy) needs M01, M20 (from t = 1) and M11
          // (t = 2); t = 1 (d/dconic_z, d/dopacity, d/drg) needs M00, C0, C1 (t = 0) and M02 (t = 2); t = 2 (d/db) needs
          // C2 (t = 1).  Source lane of x2: t = 0 <- 2, 1 <- 0, 2 <- 1.
          const int src = (lane & ~3) | ((0x3102 >> (4 * t)) & 3);
          const float x0 = __shfl_xor_sync(FULL, d0, 1);                      // t = 0: M01   t = 1: M00
          const float x1 = __shfl_down_sync(FULL, d1, 1);                     // t = 0: M20   t = 1: M02
          const float x2 = __shfl_sync(FULL, t == 2 ? d0 : d2, src);          // t = 0: M11   t = 1: C0   t = 2: C2
          const float x3 = __shfl_xor_sync(FULL, d3, 1);                      //              t = 1: C1
          if (g < pend && t < 3) {
            const uint32_t rec = s_rec_addr + 48u * (uint32_t)e;
            const float4 r0 = lds_f4(rec);                                    // (px, py, conic_x', conic_y')
            const float2 r1 = lds_f2(rec + 16u);                              // (conic_z', opacity)
            float* dst = dsplat + (int64_t)__float_as_int(lds_f2(rec + 40u).y) * LGR_GRAD_FLOATS;
            const float X = r0.x - tcx, Y = r0.y - tcy;
            float4 part;                               // float4 t of the splat's gradient row: one vector atomic per lane
            if (t == 0) {
              const float M00 = d0, M10 = d1, M01 = x0, M20 = x1, M11 = x2;
              const float Sx = fmaf(X, M00, -M10), Sy = fmaf(Y, M00, -M01);                       // sum wG dx, sum wG dy
              const float Sxx = fmaf(X, fmaf(X, M00, -2.f * M10), M20);                           // sum wG dx^2
              const float Sxy = fmaf(X, fmaf(Y, M00, -M01), fmaf(-Y, M10, M11));                  // sum wG dx dy
              part.x = -(r0.z * Sx + r0.w * Sy);       // d/dpx  (x log2e: the conic in the record is pre-scaled)
              part.y = -(r1.x * Sy + r0.w * Sx);       // d/dpy  (x log2e)
              part.z = -0.5f * Sxx;                    // d/dconic_x
              part.w = -Sxy;                           // d/dconic_y
            } else if (t == 1) {
              const float M00 = x0, M01 = d0, M02 = x1;
              part.x = -0.5f * fmaf(Y, fmaf(Y, M00, -2.f * M01), M02);                             // d/dconic_z = -sum wG dy^2 / 2
              part.y = M00 * rcp_approx(r1.y);         // d/dopacity = sum G dL/dalpha = sum wG / o
              part.z = x2; part.w = x3;                // d/dr, d/dg
            } else {
              part = make_float4(x2, 0.f, 0.f, 0.f);   // d/db; the row's 3 padding floats stay 0
            }
            atomicAdd(reinterpret_cast<float4*>(dst) + t, part);
          }
          __syncwarp();
          pend = 0;
        }
        if (fin) break;
      }
    }
    const int all_done = __syncthreads_and(done);      // B: every warp has left the walk
    base += BATCH;
    if (all_done || base >= len) break;
    cnt = min(BATCH, len - base);
    stage();
  }
}

// ---------------------------------------------------------------------------------------------------------
int launch_blend_fwd(const View& v, const int32_t* tile_start, const int32_t* sorted_ids, const float* splat,
                     float* image, float* final_T, int32_t* n_contrib, int32_t* pid_pixel, float* pw_pixel,
                     float* point_weight, int32_t* point_count, cudaStream_t st) {
  const int ntiles = v.gx * (v.row1 - v.row0);
  if (ntiles <= 0) return 0;
  ProfScope ps(K_BLEND_FWD, st);
  unsigned* pwb = reinterpret_cast<unsigned*>(point_weight);
  const bool rec = v.contrib != nullptr;
  if (v.want_aux && rec)
    blend_fwd_kernel<true, true><<<ntiles, BLEND_THREADS, 0, st>>>(v, tile_start, sorted_ids, splat, image, final_T, n_contrib, pid_pixel, pw_pixel, pwb, point_count);
  else if (v.want_aux)
    blend_fwd_kernel<true, false><<<ntiles, BLEND_THREADS, 0, st>>>(v, tile_start, sorted_ids, splat, image, final_T, n_contrib, pid_pixel, pw_pixel, pwb, point_count);
  else if (rec)
    blend_fwd_kernel<false, true><<<ntiles, BLEND_THREADS, 0, st>>>(v, tile_start, sorted_ids, splat, image, final_T, n_contrib, pid_pixel, pw_pixel, pwb, point_count);
  else
    blend_fwd_kernel<false, false><<<ntiles, BLEND_THREADS, 0, st>>>(v, tile_start, sorted_ids, splat, image, final_T, n_contrib, pid_pixel, pw_pixel, pwb, point_count);
  LGR_CHECK_LAUNCH();
  return 0;
}

int launch_blend_bwd(const View& v, const int32_t* tile_start, const int32_t* sorted_ids, const float* splat,
                     const float* image, const float* dL_dimage, float* dsplat, cudaStream_t st) {
  const int ntiles = v.gx * (v.row1 - v.row0);
  if (ntiles <= 0) return 0;
  const bool rec = v.contrib != nullptr && v.last_contrib != nullptr;
  ProfScope ps(K_BLEND_BWD, st);
  if (rec) blend_bwd_kernel<true><<<ntiles, BLEND_THREADS, BWD_SMEM, st>>>(v, tile_start, sorted_ids, splat, image, dL_dimage, dsplat);
  else blend_bwd_kernel<false><<<ntiles, BLEND_THREADS, BWD_SMEM, st>>>(v, tile_start, sorted_ids, splat, image, dL_dimage, dsplat);
  LGR_CHECK_LAUNCH();
  return 0;
}

}  // namespace lgr
