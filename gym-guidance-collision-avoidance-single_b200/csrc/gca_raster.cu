// gca_raster.cu - image observation of SingleAircraftStackEnv on the device (sm_100a).
//
// Reference: PKG/SingleAircraftStackEnv.py:179-214 (render: 800x800 RGB GL frame) and :104-108
// (preprocess_frame: RGB2GRAY + INTER_AREA / 4).  The per-sample arithmetic is the specification in
// gca_raster_spec.h (shared with the CPU oracle); this file evaluates exactly that arithmetic, with
// exact-equivalence shortcuts only (argued where they are made).
//
// Persistent CTAs (2 per SM), each looping over environments.  The 1.9 MB full-resolution frame never
// exists, and the 40 KB output plane is assembled in SHARED memory and leaves with one TMA bulk store:
//   0. once per CTA: the three 32x32 RGBA textures are expanded to float4 in shared memory; every
//      bilinear footprint (33x33 corners per texture) is classified: 0 = four transparent texels
//      (the blend is the identity), 2 = four identical opaque texels (the blend is a replacement),
//      1 = anything else (the general blend); a summed-area table counts the non-transparent
//      footprints of any index rectangle;
//   1. per env: sprite poses in draw order (ownship, goal, intruders) -> shared memory; the plane is
//      filled with white; every sprite ORs its bit into the <= 2x2 cells (16x16 output pixels) it reaches;
//   2. one warp per sprite walks the <= 13x13 output pixels of the sprite's bounding box, 32 at a time.
//      A pixel is LIVE for a sprite if its 4x4 sample block can meet the rotated quad and the footprints
//      those samples can land on are not all transparent (summed-area query).  The warp keeps the pixels
//      that are live for its sprite and for no sprite drawn earlier - so every pixel that can differ from
//      white is shaded exactly once - together with the (<= 4) sprites that are live on it;
//   3. the kept pixels are shaded two at a time, lane = one of the 16 samples of a pixel.  Pixels on which only
//      this sprite is live (the destination is white: ~98 % of them) take a deferred path: transparent and
//      uniform-opaque footprints are settled at once, the samples that need the general bilinear blend are
//      queued and blended 32 at a time with every lane busy, their grays added by shared-memory atomics.  The
//      others take the ordered path: colour state in registers, the live sprites blended in draw order.  Then
//      gray, warp-wide packed integer reduction, 4x4 area mean (round half to even), one byte into the plane;
//   4. fence.proxy.async + cp.async.bulk shared -> global of the whole plane (UBLKCP); the next env's
//      fill waits only for the bulk copy to have READ the plane.
// Output bytes: 40 000 per env-step, written once, fully coalesced.
#include "gca_launch.h"
#include "gca_raster_spec.h"

namespace gca {

constexpr int kRasterThreads = 384;
constexpr int kRasterWarps = kRasterThreads / 32;
constexpr int kMaxSprites = GCA_RASTER_MAX_INTRUDERS + 2;   // 128 -> 4 mask words per cell
constexpr int kCorner = GCA_SPRITE + 1;                     // bilinear footprints per axis: iu in [-1, 31]
constexpr int kSat = kCorner + 1;                           // summed-area table side
constexpr int kListCap = 40;                                // >= 1 carried + 32 new pixels + 1 odd simple pixel
constexpr int kCellShift = 4;                               // cell = 16 x 16 output pixels
constexpr float kMagic = 12582912.0f;                       // 1.5 * 2^23: x + kMagic rounds x to an integer (RN-even)
// half extent of the quad (16) + half diagonal of the 4x4 sample block (1.5 * sqrt 2 = 2.1214) + slack
constexpr float kHitReach = 18.25f;
constexpr uint32_t kScanCell = 0xfefefefeu;                 // more than 4 live sprites: walk the whole cell mask

struct RasterArgs {
  DevState s;
  int faithful;
  int W, H;                 // full-resolution canvas
  int ow, oh;               // output size (W/4, H/4)
  int cells_x, cells_y;     // 8x8-output-pixel cells
  const uint8_t* sprites;
  uint8_t* frames;
  long long env_stride, plane_stride;
  int n_planes, slot;
  const uint8_t* clear_mask;
  int bulk_ok;              // plane addresses / size are 16-byte aligned: TMA bulk store
};

// floor of t for t in [-0.5, 31.5] without a conversion instruction: s = RN(t + kMagic) is kMagic + n with n the
// nearest integer, exactly; n - (n > t) is the floor.  Returns the integer, writes the float.
__device__ __forceinline__ int floor_small(float t, float* fl) {
  const float s = __fadd_rn(t, kMagic);
  const float n = __fadd_rn(s, -kMagic);
  const int adj = n > t ? 1 : 0;
  *fl = n > t ? __fadd_rn(n, -1.0f) : n;
  return (__float_as_int(s) - 0x4B400000) - adj;
}

// The spec's clamp((int)rintf(v), 0, 255), kept in float.  v = src * alpha + dst * (1 - alpha) with src <= 255 (1 + 2e-6),
// 0 <= dst <= 255, 0 <= alpha <= 1 + 2e-6 lies in (-0.01, 255.01), so rintf(v) is already in [0, 255] and the clamp is
// the identity; (v + kMagic) - kMagic is rintf(v) (round to nearest even) for |v| < 2^22.
__device__ __forceinline__ float quantise_u8(float v) { return __fadd_rn(__fadd_rn(v, kMagic), -kMagic); }

// gca_raster_sample (gca_raster_spec.h) with the 8-bit colour kept in float registers.  Same operations in the
// same order; the two shortcuts are exact:
//  * class 0 (four texels with alpha 0): the spec's a255 is 0.0f and it returns without blending;
//  * class 2 (four texels equal, alpha 255): every bilinear value is c(1+e), |e| < 2e-6, alpha is 1+e', |e'| < 2e-6,
//    so v = c + d with |d| < 2e-3 for c, dst <= 255 and rintf(v) = c: the blend writes the texel colour.
// where a sample falls in a sprite's texture: false if outside the quad
__device__ __forceinline__ bool sample_locate(const float4 pose, float wx, float wy, int& iu, int& iv, float& tu, float& tv,
                                              float& fu0, float& fv0) {
  const float dx = __fadd_rn(wx, -pose.x), dy = __fadd_rn(wy, -pose.y);
  const float lx = __fadd_rn(__fmul_rn(pose.z, dx), __fmul_rn(pose.w, dy));
  const float ly = __fadd_rn(__fmul_rn(pose.z, dy), -__fmul_rn(pose.w, dx));
  if (!(lx >= -GCA_SPRITE_HALF && lx < GCA_SPRITE_HALF && ly >= -GCA_SPRITE_HALF && ly < GCA_SPRITE_HALF)) return false;
  tu = __fadd_rn(lx, 15.5f);
  tv = __fadd_rn(ly, 15.5f);
  iu = floor_small(tu, &fu0);
  iv = floor_small(tv, &fv0);
  return true;
}

// the general bilinear fetch + alpha blend of one located sample (t: the sprite's 32x32 float4 texture)
__device__ __forceinline__ void sample_blend(const float4* __restrict__ t, int iu, int iv, float tu, float tv, float fu0,
                                             float fv0, float& r, float& g, float& b) {
  const int u0 = max(iu, 0), u1 = min(iu + 1, 31), v0 = max(iv, 0), v1 = min(iv + 1, 31);
  const float4 t00 = t[(31 - v0) * GCA_SPRITE + u0];
  const float4 t10 = t[(31 - v0) * GCA_SPRITE + u1];
  const float4 t01 = t[(31 - v1) * GCA_SPRITE + u0];
  const float4 t11 = t[(31 - v1) * GCA_SPRITE + u1];
  const float fu = __fadd_rn(tu, -fu0), fv = __fadd_rn(tv, -fv0);
  const float gu = __fadd_rn(1.0f, -fu), gv = __fadd_rn(1.0f, -fv);
#define GCA_BIL(k)                                                                                  \
  __fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(t00.k, gu), __fmul_rn(t10.k, fu)), gv),                   \
            __fmul_rn(__fadd_rn(__fmul_rn(t01.k, gu), __fmul_rn(t11.k, fu)), fv))
  const float a255 = GCA_BIL(w);
  if (a255 == 0.0f) return;
  const float alpha = __fmul_rn(a255, 0.003921568859368563f);
  const float beta = __fadd_rn(1.0f, -alpha);
  r = quantise_u8(__fadd_rn(__fmul_rn(GCA_BIL(x), alpha), __fmul_rn(r, beta)));
  g = quantise_u8(__fadd_rn(__fmul_rn(GCA_BIL(y), alpha), __fmul_rn(g, beta)));
  b = quantise_u8(__fadd_rn(__fmul_rn(GCA_BIL(z), alpha), __fmul_rn(b, beta)));
#undef GCA_BIL
}

__device__ __forceinline__ void raster_sample_fast(const float4 pose, const int tex, const float4* __restrict__ texf,
                                                   const uint8_t* __restrict__ cls, float wx, float wy, float& r,
                                                   float& g, float& b) {
  int iu, iv;
  float tu, tv, fu0, fv0;
  if (!sample_locate(pose, wx, wy, iu, iv, tu, tv, fu0, fv0)) return;
  const int c = cls[tex * (kCorner * kCorner) + (iv + 1) * kCorner + (iu + 1)];
  if (c == 0) return;
  const float4* t = texf + tex * (GCA_SPRITE * GCA_SPRITE);
  if (c == 2) {
    const float4 t00 = t[(31 - max(iv, 0)) * GCA_SPRITE + max(iu, 0)];
    r = t00.x; g = t00.y; b = t00.z;
    return;
  }
  sample_blend(t, iu, iv, tu, tv, fu0, fv0, r, g, b);
}

// cv2 RGB2GRAY in exact float arithmetic (every intermediate is an integer < 2^24), then >> 15
__device__ __forceinline__ int gray_of(float r, float g, float b) {
  const float gx = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(9798.0f, r), __fmul_rn(19235.0f, g)), __fmul_rn(3735.0f, b)), 16384.0f);
  return __float2int_rn(gx) >> 15;
}

__device__ __forceinline__ int floor_int(float t) {        // floor for |t| < 2^22, no conversion instruction
  const float s = __fadd_rn(t, kMagic);
  return (__float_as_int(s) - 0x4B400000) - (__fadd_rn(s, -kMagic) > t ? 1 : 0);
}

// Is the output pixel centred on (pcx, pcy) LIVE for the sprite: can one of its 16 samples (offsets +-0.5, +-1.5)
// fall inside the quad on a footprint that is not fully transparent?  Conservative (never false for a sample
// the spec would blend), deterministic (every warp evaluates the same function, so ownership is consistent).
__device__ __forceinline__ bool pixel_live(const float4 pose, const uint16_t* __restrict__ sat, float pcx, float pcy) {
  const float dx = pcx - pose.x, dy = pcy - pose.y;
  const float lx = pose.z * dx + pose.w * dy, ly = pose.z * dy - pose.w * dx;
  if (!(fabsf(lx) <= kHitReach && fabsf(ly) <= kHitReach)) return false;
  // the samples' local coordinates lie within +-rad of the centre's on each axis
  const float rad = 1.5f * (fabsf(pose.z) + fabsf(pose.w)) + 0.01f;
  const float tu = lx + 15.5f, tv = ly + 15.5f;
  const int a0 = min(max(floor_int(tu - rad), -1), 31) + 1, a1 = min(max(floor_int(tu + rad), -1), 31) + 2;
  const int b0 = min(max(floor_int(tv - rad), -1), 31) + 1, b1 = min(max(floor_int(tv + rad), -1), 31) + 2;
  const int n = (int)sat[b1 * kSat + a1] - (int)sat[b0 * kSat + a1] - (int)sat[b1 * kSat + a0] + (int)sat[b0 * kSat + a0];
  return n > 0;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__global__ void __launch_bounds__(kRasterThreads, 2) raster_kernel(const RasterArgs a) {
  extern __shared__ __align__(16) uint8_t rsm[];
  const DevState& s = a.s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n_sprites = 2 + s.N;
  const int n_cells = a.cells_x * a.cells_y;
  const int plane_bytes = a.ow * a.oh;
  float4* texf = reinterpret_cast<float4*>(rsm);                                   // [3][32][32] RGBA as float
  uint8_t* plane = rsm + 3 * GCA_SPRITE * GCA_SPRITE * sizeof(float4);             // [oh][ow]
  uint4* cell_mask = reinterpret_cast<uint4*>(plane + ((plane_bytes + 15) & ~15)); // [n_cells]
  float4* pose = reinterpret_cast<float4*>(cell_mask + n_cells);                   // [128] (cx, cy, rc, rs)
  short4* box = reinterpret_cast<short4*>(pose + kMaxSprites);                     // [128] output-pixel bounding boxes
  uint2* list = reinterpret_cast<uint2*>(box + kMaxSprites) + warp * kListCap;     // per warp: (ox | oy << 16, sprite ids)
  uint32_t* wsm = reinterpret_cast<uint32_t*>(reinterpret_cast<uint2*>(box + kMaxSprites) + kRasterWarps * kListCap) + warp * 96;
  uint32_t* slist = wsm;                                                           // per warp: 32 simple pixels (ox | oy << 16)
  int* acc = reinterpret_cast<int*>(wsm + 32);                                     //           their gray sums
  uint16_t* queue = reinterpret_cast<uint16_t*>(wsm + 64);                         //           deferred samples (slot << 4 | sample)
  uint16_t* sat_all = reinterpret_cast<uint16_t*>(reinterpret_cast<uint32_t*>(reinterpret_cast<uint2*>(box + kMaxSprites) + kRasterWarps * kListCap) + kRasterWarps * 96);
  uint8_t* cls = reinterpret_cast<uint8_t*>(sat_all + 3 * kSat * kSat);            // [3][33][33]
  __shared__ int next_sprite;                                                      // dynamic sprite -> warp assignment

  // ---- 0. textures, footprint classes and their summed-area tables, once per CTA
  for (int i = tid; i < 3 * GCA_SPRITE * GCA_SPRITE; i += kRasterThreads) {
    const uchar4 q = reinterpret_cast<const uchar4*>(a.sprites)[i];
    texf[i] = make_float4((float)q.x, (float)q.y, (float)q.z, (float)q.w);
  }
  for (int i = tid; i < 3 * kCorner * kCorner; i += kRasterThreads) {
    const int t = i / (kCorner * kCorner), c = i % (kCorner * kCorner);
    const int iv = c / kCorner - 1, iu = c % kCorner - 1;
    const int u0 = max(iu, 0), u1 = min(iu + 1, 31), v0 = max(iv, 0), v1 = min(iv + 1, 31);
    const uint32_t* tx = reinterpret_cast<const uint32_t*>(a.sprites) + t * GCA_SPRITE * GCA_SPRITE;
    const uint32_t q00 = tx[(31 - v0) * GCA_SPRITE + u0], q10 = tx[(31 - v0) * GCA_SPRITE + u1];
    const uint32_t q01 = tx[(31 - v1) * GCA_SPRITE + u0], q11 = tx[(31 - v1) * GCA_SPRITE + u1];
    int k = 1;
    if (((q00 | q10 | q01 | q11) >> 24) == 0u) k = 0;
    else if ((q00 >> 24) == 255u && q00 == q10 && q00 == q01 && q00 == q11) k = 2;
    cls[i] = (uint8_t)k;
  }
  __syncthreads();
  // sat[t][b][a] = number of non-transparent footprints with row < b and column < a (rows / columns shifted by +1)
  for (int i = tid; i < 3 * kSat; i += kRasterThreads) {                            // row prefix sums
    const int t = i / kSat, b = i % kSat;
    uint16_t* row = sat_all + (t * kSat + b) * kSat;
    int acc = 0;
    row[0] = 0;
    for (int c = 1; c < kSat; ++c) {
      if (b >= 1) acc += cls[t * kCorner * kCorner + (b - 1) * kCorner + (c - 1)] != 0;
      row[c] = (uint16_t)acc;
    }
  }
  __syncthreads();
  for (int i = tid; i < 3 * kSat; i += kRasterThreads) {                            // column prefix sums
    const int t = i / kSat, c = i % kSat;
    uint16_t* col = sat_all + t * kSat * kSat + c;
    int acc = 0;
    for (int b = 0; b < kSat; ++b) { acc += col[b * kSat]; col[b * kSat] = (uint16_t)acc; }
  }

  for (int env = blockIdx.x; env < s.B; env += gridDim.x) {
    // the bulk store of the previous plane must have read shared memory before it is filled again
    if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncthreads();

    // ---- 1. sprite poses in draw order: ownship, goal, intruders (PKG/SingleAircraftStackEnv.py:192-212)
    if (tid < n_sprites) {
      float4 p;
      if (tid == 0) {
        const float2 pos = s.own_pos[env];
        const double2 hs = s.own_hs[env];
        double sn, cs;
        gca_sincos(hs.x, &sn, &cs);
        p = make_float4(pos.x, pos.y, (float)sn, -(float)cs);             // cos(h - pi/2) = sin h, sin(h - pi/2) = -cos h
      } else if (tid == 1) {
        const double2 g = s.goal[env];
        p = make_float4((float)g.x, (float)g.y, 1.0f, 0.0f);
      } else {
        const int i = tid - 2;
        float px, py;
        const uint8_t* pl = s.ipos + (size_t)(s.counters[env].z & 1) * s.pos_plane;   // the env's current positions
        if (a.faithful) {
          const double2 q = *reinterpret_cast<const double2*>(pl + ipos_offset(s, true, (size_t)env, i));
          px = (float)q.x; py = (float)q.y;
        } else {
          const float2 q = *reinterpret_cast<const float2*>(pl + ipos_offset(s, false, (size_t)env, i));
          px = q.x; py = q.y;
        }
        const float2 v = *reinterpret_cast<const float2*>(s.ivel + ivel_offset(s, (size_t)env, i));
        // the intruder's heading is constant for life (:207-211); its direction is that of the velocity
        // (a zero velocity - only gca_set_state can make one - has no direction: drawn with heading 0, never a NaN pose)
        const float len = __fsqrt_rn(__fadd_rn(__fmul_rn(v.x, v.x), __fmul_rn(v.y, v.y)));
        const float ch = len > 0.0f ? __fdiv_rn(v.x, len) : 1.0f, sh = len > 0.0f ? __fdiv_rn(v.y, len) : 0.0f;
        p = make_float4(px, py, sh, -ch);
      }
      pose[tid] = p;
      // bounding box in output pixels (x0 > x1 or y0 > y1: nothing on the canvas)
      const float ytop = (float)a.H - p.y;
      const float fx0 = floorf((p.x - GCA_SPRITE_REACH) * 0.25f), fx1 = floorf((p.x + GCA_SPRITE_REACH) * 0.25f);
      const float fy0 = floorf((ytop - GCA_SPRITE_REACH) * 0.25f), fy1 = floorf((ytop + GCA_SPRITE_REACH) * 0.25f);
      box[tid] = make_short4((short)fminf(fmaxf(fx0, 0.0f), (float)a.ow), (short)fminf(fmaxf(fx1, -1.0f), (float)(a.ow - 1)),
                             (short)fminf(fmaxf(fy0, 0.0f), (float)a.oh), (short)fminf(fmaxf(fy1, -1.0f), (float)(a.oh - 1)));
    }
    for (int i = tid; i < n_cells; i += kRasterThreads) cell_mask[i] = make_uint4(0u, 0u, 0u, 0u);
    if (tid == 0) next_sprite = 0;
    {
      uint4* o4 = reinterpret_cast<uint4*>(plane);                        // white clear
      const uint4 white = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
      for (int i = tid; i < (plane_bytes + 15) / 16; i += kRasterThreads) o4[i] = white;
    }
    // VecFrameStack: a finished env starts from an all-zero stack (vec_frame_stack.py:19-23)
    uint8_t* env_base = a.frames + (long long)env * a.env_stride;
    if (a.clear_mask && a.clear_mask[env]) {
      const int words = plane_bytes / 4;
      for (int pl = 0; pl < a.n_planes; ++pl) {
        if (pl == a.slot) continue;
        uint32_t* dst = reinterpret_cast<uint32_t*>(env_base + (long long)pl * a.plane_stride);
        for (int i = tid; i < words; i += kRasterThreads) dst[i] = 0u;
      }
    }
    __syncthreads();

    // ---- bin the sprites into cells (their bounding boxes, in output pixels)
    if (tid < n_sprites) {
      const short4 bb = box[tid];
      for (int cy = bb.z >> kCellShift; cy <= (bb.w >> kCellShift) && bb.z <= bb.w; ++cy)
        for (int cx = bb.x >> kCellShift; cx <= (bb.y >> kCellShift) && bb.x <= bb.y; ++cx)
          atomicOr(reinterpret_cast<unsigned int*>(&cell_mask[cy * a.cells_x + cx]) + (tid >> 5), 1u << (tid & 31));
    }
    __syncthreads();

    // ---- 2 + 3. one warp per sprite
    const int half = lane >> 4, sidx = lane & 15;
    const float sxo = (float)(sidx & 3) + 0.5f, syo = (float)(sidx >> 2) + 0.5f;
    // shade list[i] (lanes 0-15) and list[i + 1] (lanes 16-31, if two)
    auto shade_pair = [&](int i, bool two) {
      const bool valid = half == 0 || two;
      const uint2 e = list[valid ? i + half : i];
      const int ox = (int)(e.x & 0xffffu), oy = (int)(e.x >> 16);
      const float wx = __fadd_rn((float)(4 * ox), sxo);
      const float wy = __fadd_rn((float)a.H, -__fadd_rn((float)(4 * oy), syo));
      float r = 255.0f, g = 255.0f, b = 255.0f;                            // white clear
      if (e.y != kScanCell) {
        uint32_t ids = e.y;                                                // <= 4 sprites in draw order, 0xff ends
        while ((ids & 0xffu) != 0xffu) {
          const int j = (int)(ids & 0xffu);
          ids = (ids >> 8) | 0xff000000u;
          raster_sample_fast(pose[j], min(j, 2), texf, cls, wx, wy, r, g, b);
        }
      } else {
        const uint4 m = cell_mask[(oy >> kCellShift) * a.cells_x + (ox >> kCellShift)];
        const uint32_t words[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          uint32_t bits = words[w];
          while (bits) {
            const int j = w * 32 + __ffs(bits) - 1;
            bits &= bits - 1;
            raster_sample_fast(pose[j], min(j, 2), texf, cls, wx, wy, r, g, b);
          }
        }
      }
      const int gray = gray_of(r, g, b);
      const int both = __reduce_add_sync(0xffffffffu, gray << (half * 16));
      if (sidx == 0 && valid) plane[oy * a.ow + ox] = (uint8_t)gca_area16_u8((both >> (half * 16)) & 0xffff);
    };

    for (;;) {
      int k0 = 0;
      if (lane == 0) k0 = atomicAdd(&next_sprite, 1);                      // sprites own disjoint pixels: any order
      k0 = __shfl_sync(0xffffffffu, k0, 0);
      if (k0 >= n_sprites) break;
      const float4 me = pose[k0];
      const uint16_t* my_sat = sat_all + min(k0, 2) * kSat * kSat;
      const short4 mb = box[k0];
      const int bx0 = mb.x, by0 = mb.z;
      const int nx = mb.y - mb.x + 1, ny = mb.w - mb.z + 1;
      if (nx <= 0 || ny <= 0) continue;
      int cnt = 0;
      for (int base = 0; base < nx * ny; base += 32) {
        // 2. pixels this sprite owns: live for it and for no sprite drawn earlier
        const int p = base + lane;
        bool keep = false;
        uint2 entry = make_uint2(0u, 0u);
        if (p < nx * ny) {
          const int oy = by0 + p / nx, ox = bx0 + p % nx;
          const float pcx = (float)(4 * ox) + 2.0f, pcy = (float)a.H - ((float)(4 * oy) + 2.0f);
          if (pixel_live(me, my_sat, pcx, pcy)) {
            const uint4 m = cell_mask[(oy >> kCellShift) * a.cells_x + (ox >> kCellShift)];
            const uint32_t words[4] = {m.x, m.y, m.z, m.w};
            uint32_t ids = 0xffffff00u | (uint32_t)k0;
            int nid = 1;
            keep = true;
#pragma unroll
            for (int w = 0; w < 4; ++w) {
              uint32_t bits = words[w];
              while (bits && keep) {
                const int j = w * 32 + __ffs(bits) - 1;
                bits &= bits - 1;
                if (j == k0) continue;
                const short4 jb = box[j];
                if (ox >= jb.x && ox <= jb.y && oy >= jb.z && oy <= jb.w &&
                    pixel_live(pose[j], sat_all + min(j, 2) * kSat * kSat, pcx, pcy)) {
                  if (j < k0) keep = false;                                // an earlier sprite owns this pixel
                  else if (nid < 4) { ids = (ids & ~(0xffu << (8 * nid))) | ((uint32_t)j << (8 * nid)); ++nid; }
                  else ids = kScanCell;
                }
              }
            }
            entry = make_uint2((uint32_t)ox | ((uint32_t)oy << 16), nid > 4 || ids == kScanCell ? kScanCell : ids);
          }
        }
        // simple pixels (this sprite is the only live one: the destination is white, blending order is moot) take the
        // deferred path below; the others, and an odd simple one, the ordered path
        const bool simple = keep && entry.y == (0xffffff00u | (uint32_t)k0);
        const uint32_t bs = __ballot_sync(0xffffffffu, simple);
        const uint32_t bc = __ballot_sync(0xffffffffu, keep && !simple);
        const int ns = __popc(bs) & ~1;                                    // simple pixels shaded in pairs
        if (simple) {
          const int rk = __popc(bs & ((1u << lane) - 1u));
          if (rk < ns) slist[rk] = entry.x;
          else list[cnt + __popc(bc)] = entry;                             // the odd one out
        }
        if (keep && !simple) list[cnt + __popc(bc & ((1u << lane) - 1u))] = entry;
        cnt += __popc(bc) + (__popc(bs) & 1);
        __syncwarp();
        // 3a. simple pixels: lane = sample; transparent and uniform-opaque footprints are settled at once, the general
        // blends are queued and done 32 at a time with every lane busy
        {
          const float4* mytex = texf + min(k0, 2) * (GCA_SPRITE * GCA_SPRITE);
          const uint8_t* mycls = cls + min(k0, 2) * (kCorner * kCorner);
          int qn = 0;
          auto flush = [&](int start, int n) {
            if (lane < n) {
              const int q = queue[start + lane], slot = q >> 4, sm = q & 15;
              const uint32_t e = slist[slot];
              const float wx = __fadd_rn((float)(4 * (int)(e & 0xffffu)), (float)(sm & 3) + 0.5f);
              const float wy = __fadd_rn((float)a.H, -__fadd_rn((float)(4 * (int)(e >> 16)), (float)(sm >> 2) + 0.5f));
              int iu, iv;
              float tu, tv, fu0, fv0;
              float r = 255.0f, g = 255.0f, b = 255.0f;                    // white clear
              if (sample_locate(me, wx, wy, iu, iv, tu, tv, fu0, fv0)) sample_blend(mytex, iu, iv, tu, tv, fu0, fv0, r, g, b);
              atomicAdd(&acc[slot], gray_of(r, g, b));
            }
            __syncwarp();
          };
          for (int i = 0; i < ns; i += 2) {
            const uint32_t e = slist[i + half];
            const float wx = __fadd_rn((float)(4 * (int)(e & 0xffffu)), sxo);
            const float wy = __fadd_rn((float)a.H, -__fadd_rn((float)(4 * (int)(e >> 16)), syo));
            int iu, iv;
            float tu, tv, fu0, fv0;
            int gray = 255;                                                // outside the quad / transparent: white
            bool defer = false;
            if (sample_locate(me, wx, wy, iu, iv, tu, tv, fu0, fv0)) {
              const int c = mycls[(iv + 1) * kCorner + (iu + 1)];
              if (c == 2) {
                const float4 t00 = mytex[(31 - max(iv, 0)) * GCA_SPRITE + max(iu, 0)];
                gray = gray_of(t00.x, t00.y, t00.z);
              } else if (c == 1) {
                defer = true;
                gray = 0;
              }
            }
            const int both = __reduce_add_sync(0xffffffffu, gray << (half * 16));
            if (sidx == 0) acc[i + half] = (both >> (half * 16)) & 0xffff;
            const uint32_t bd = __ballot_sync(0xffffffffu, defer);
            if (defer) queue[qn + __popc(bd & ((1u << lane) - 1u))] = (uint16_t)(((i + half) << 4) | sidx);
            qn += __popc(bd);
            __syncwarp();
            if (qn >= 32) {
              flush(qn - 32, 32);
              qn -= 32;
            }
          }
          if (qn) flush(0, qn);
          for (int l = lane; l < ns; l += 32) {
            const uint32_t e = slist[l];
            plane[(int)(e >> 16) * a.ow + (int)(e & 0xffffu)] = (uint8_t)gca_area16_u8(acc[l]);
          }
          __syncwarp();
        }
        // 3b. the ordered path: two pixels per pass, lane = sample; an odd one is carried to the next batch
        int i = 0;
        for (; i + 1 < cnt; i += 2) shade_pair(i, true);
        if (i < cnt) {
          const uint2 last = list[i];
          __syncwarp();
          if (lane == 0) list[0] = last;
          cnt = 1;
        } else {
          cnt = 0;
        }
        __syncwarp();
      }
      if (cnt) shade_pair(0, false);
      __syncwarp();
    }
    __syncthreads();

    // ---- 4. the finished plane leaves shared memory
    uint8_t* out = env_base + (long long)a.slot * a.plane_stride;
    if (a.bulk_ok) {
      if (tid == 0) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                     :: "l"(out), "r"(smem_u32(plane)), "r"(plane_bytes) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    } else {
      for (int i = tid; i < plane_bytes / 4; i += kRasterThreads)
        reinterpret_cast<uint32_t*>(out)[i] = reinterpret_cast<const uint32_t*>(plane)[i];
    }
  }
  if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

size_t raster_smem_bytes(int ow, int oh) {
  const int cs = 1 << kCellShift;
  const int cells = ((ow + cs - 1) / cs) * ((oh + cs - 1) / cs);
  return 3 * GCA_SPRITE * GCA_SPRITE * sizeof(float4) + (((size_t)ow * oh + 15) & ~(size_t)15) + sizeof(uint4) * (size_t)cells +
         (sizeof(float4) + sizeof(short4)) * kMaxSprites + sizeof(uint2) * kRasterWarps * kListCap +
         sizeof(uint32_t) * kRasterWarps * 96 +
         sizeof(uint16_t) * 3 * kSat * kSat + ((3 * kCorner * kCorner + 15) & ~15);
}

cudaError_t launch_raster(const DevState& s, bool faithful, int W, int H, const uint8_t* sprites, uint8_t* frames,
                          long long env_stride, long long plane_stride, int n_planes, int slot,
                          const uint8_t* clear_mask, cudaStream_t st) {
  RasterArgs a{};
  a.s = s; a.faithful = faithful ? 1 : 0; a.W = W; a.H = H; a.ow = W / 4; a.oh = H / 4;
  a.cells_x = (a.ow + (1 << kCellShift) - 1) >> kCellShift; a.cells_y = (a.oh + (1 << kCellShift) - 1) >> kCellShift;
  a.sprites = sprites; a.frames = frames; a.env_stride = env_stride; a.plane_stride = plane_stride;
  a.n_planes = n_planes; a.slot = slot; a.clear_mask = clear_mask;
  a.bulk_ok = ((a.ow * a.oh) % 16 == 0 && env_stride % 16 == 0 && plane_stride % 16 == 0 &&
               reinterpret_cast<uintptr_t>(frames) % 16 == 0) ? 1 : 0;
  const size_t smem = raster_smem_bytes(a.ow, a.oh);
  if (smem > kRasterSmemMax || a.ow > 32767 || a.oh > 32767) return cudaErrorInvalidValue;
  cudaError_t e = cudaFuncSetAttribute(raster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int per_sm = smem * 2 + 2048 <= kRasterSmemMax ? 2 : 1;
  const unsigned grid = (unsigned)min((long long)s.B, (long long)sms * per_sm);
  raster_kernel<<<grid, kRasterThreads, smem, st>>>(a);
  return cudaGetLastError();
}

}  // namespace gca
