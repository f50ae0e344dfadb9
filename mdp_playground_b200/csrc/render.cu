// Image-observation renderers (K4 ImageMultiDiscrete, K5 ImageContinuous).
//
// K4 restates spaces/image_multi_discrete.py:129-270: polygon -> rotate ->
// flip -> transpose, as ONE gather per output byte: the final pixel is mapped
// back through the flip and Pillow's 16.16 fixed-point rotation to the polygon
// image, where a bit of the (state, R, vertex-variant) mask decides 0 / 255.
// K5 restates spaces/image_continuous.py:116-246: background 208, black
// terminal rectangles, green target disc, blue agent disc (painter's order),
// relevant and irrelevant sub-images stacked along x.
//
// K4: one warp renders one image.  The image is zero-filled with 128-bit
// streaming stores first; the shape is then assembled as column bitmaps of the
// FINAL image in shared memory and only its non-empty 4-byte words are stored
// again.  K5: one CTA per (sub-)image, 16 output bytes per thread and store.
#include <cstdlib>
#include <string>

#include "internal.h"
#include "philox.cuh"

namespace mdpp {

constexpr int kRBlock = 128;
constexpr int kMaskRows = 64;
constexpr int kMaskCentre = 31;
constexpr int kRotCols = 80;  // bounding box of the rotated polygon: <= 2*30+7+2
// zero columns either side of the polygon mask: the rotation gather reads up to
// 15 samples past the mask box (see the segment test) without a bounds test
constexpr int kMaskPad = 24;
constexpr int kMaskCols = kMaskRows + 2 * kMaskPad;

struct RenderDParams {
  // the tables of a single-config launch; in a grouped launch group 0's
  // (width, height and n_sub_images are common) with has_rotate = any group's
  mdpp_image_discrete_tables tb;
  const mdpp_image_discrete_group* groups;  // grouped launch: the descriptors
  const uint16_t* env_group;                //   and the env -> group map
  const int64_t* states;
  const int32_t* params_in;
  int32_t* params_out;
  uint8_t* out;
  int64_t n_images, n_envs;
  uint32_t k0, k1, stream;
  uint64_t step_index;
  const uint64_t* step_index_dev;
  int64_t env_id_offset;
};

// floor(a / b) for |a| < 2^15, 0 < b < 2^15: (a + 0.5) / b is at least 0.5 / b
// away from every integer, far more than the error of the fp32 product.
__device__ __forceinline__ int floor_div_small(int a, int b, float inv_b) {
  return b == 1 ? a : (int)floorf(((float)a + 0.5f) * inv_b);
}

// One WARP renders one image (4 images per CTA): the kernel is issue-bound
// -- several hundred scalar instructions of per-image set-up against 625
// vector stores -- so the set-up must not be replicated over several warps,
// and warp barriers replace CTA barriers.  All lanes compute the (uniform)
// transform parameters redundantly; lane-parallel work is the zero fill, the
// mask load, the rotation gather and the box stores.  (Computing the set-up of
// the CTA's four images once, in lanes 0-3 of warp 0, saves ~250 of ~1900 warp
// instructions per image but measured 8 % SLOWER: three warps wait at a CTA
// barrier for the dependent loads of the fourth.)
constexpr int kImagesPerCta = kRBlock / 32;

// Everything the lane-parallel phases need to know about one image.
struct ImageSetup {
  int32_t R, sw, sh, rot, flip;  // transform parameters (rot < 0: unrotated)
  int32_t id;                    // mask of (state, R, vertex variants)
  // Final-image geometry of the box-local column bitmaps `fmask`: bit b of
  // column c is final pixel (xbase + c, ybase + b), ybase a multiple of 4 so
  // that a nibble of the bitmap is one aligned 4-byte word of the output;
  // columns c_lo..c_hi / bits b_lo..b_hi can be set (c_hi < 0: nothing).
  int32_t xbase, ybase, c_lo, c_hi, b_lo, b_hi;
  // rotation gather: 16.16 source coordinates, pre-shifted into mask space
  // (mx = X >> 16, my = Y >> 16), as linear forms of the box-local (column c,
  // row k):  X = X00 + c cX + k dX,  Y = Y00 + c cY + k dY
  int32_t X00, Y00, cX, cY, dX, dY;
  uint32_t rows_lo, rows_hi;     // mask rows whose pixel lies inside the image
};

// R = r_min + #{thresholds <= u}: one threshold per lane and a ballot (all 32
// lanes hold the same u).  `thr0` = this lane's threshold of the first 32,
// loaded by the caller ahead of the dependent chain (+inf past the end).
__device__ __forceinline__ int scaled_radius(const mdpp_image_discrete_tables& tb,
                                             uint32_t word, int lane, double thr0) {
  int R = tb.r_min;
  if (!tb.has_scale) return R;
  const double u = uniform32(word);
  R += __popc(__ballot_sync(0xffffffffu, thr0 <= u));
  for (int base = 32; base < tb.n_radii - 1; base += 32) {
    const int k = base + lane;
    const bool le = k < tb.n_radii - 1 && tb.r_thresholds[k] <= u;
    R += __popc(__ballot_sync(0xffffffffu, le));
  }
  return R;
}

// The scalar set-up of image m (see ImageSetup).  Restates the draw order of
// the reference (:149-181, :251, :258-259): one Philox call per image, w0
// scale, w1 / w2 shifts, w3 rotation + flip bits.  Uniform over the warp.
// `tb`: the image's tables; `id_base`: the Philox id of env 0 of them (mod
// 2^32), the id of env e being id_base + e.
__device__ __forceinline__ ImageSetup image_setup(const RenderDParams& p,
                                                  const mdpp_image_discrete_tables& tb,
                                                  uint32_t id_base, int64_t m,
                                                  int lane, double thr0) {
  const int W = tb.width, H = tb.height;
  ImageSetup g;
  int state = (int)p.states[m];
  state = min(max(state, 0), tb.n_states - 1);
  int R, sw, sh, rot, flip;
  if (p.params_in) {
    const int32_t* q = p.params_in + m * 5;
    R = q[0]; sw = q[1]; sh = q[2]; rot = q[3]; flip = q[4];
  } else {
    // (n_images < 2^31, checked by the caller: 32-bit arithmetic; the usual
    // shapes -- one or two sub-images, one step per launch -- divide nothing)
    uint32_t e = (uint32_t)m, sub = 0;  // (step, env); sub-image `sub` of it
    if (tb.n_sub_images == 2) { sub = e & 1u; e >>= 1; }
    else if (tb.n_sub_images > 2) { sub = e % (uint32_t)tb.n_sub_images; e /= (uint32_t)tb.n_sub_images; }
    uint32_t t_rel = 0;
    if (e >= (uint32_t)p.n_envs) { t_rel = e / (uint32_t)p.n_envs; e -= t_rel * (uint32_t)p.n_envs; }
    const uint32_t gid = id_base + e;
    const uint64_t step = p.step_index + (uint64_t)t_rel +
                          (p.step_index_dev ? *p.step_index_dev : 0ull);
    U4 w = philox4x32_10(gid, (uint32_t)step, (uint32_t)(step >> 32),
                         p.stream + 16u * sub, p.k0, p.k1);
    R = scaled_radius(tb, w.x, lane, thr0);
    sw = W / 2; sh = H / 2;
    if (tb.has_shift) {  // integers(-m + 1, m), m = W/2 - R, then quantise
      const int mw = W / 2 - R, mh = H / 2 - R;
      const int aw = -mw + 1 + (int)__umulhi(w.y, (uint32_t)max(2 * mw - 1, 1));
      const int ah = -mh + 1 + (int)__umulhi(w.z, (uint32_t)max(2 * mh - 1, 1));
      const float inv_q = 1.0f / (float)tb.sh_quant;
      sw += floor_div_small(aw, tb.sh_quant, inv_q) * tb.sh_quant;
      sh += floor_div_small(ah, tb.sh_quant, inv_q) * tb.sh_quant;
    }
    rot = -1;
    if (tb.has_rotate) {
      rot = (int)__umulhi(w.w, 360u);
      rot = floor_div_small(rot, tb.ro_quant, 1.0f / (float)tb.ro_quant) * tb.ro_quant;
    }
    flip = 0;
    if (tb.has_flip && (w.w & 1u) == 0) flip = (w.w & 2u) == 0 ? 1 : 2;
  }
  if (lane == 0 && p.params_out) {
    int32_t* q = p.params_out + m * 5;
    q[0] = R; q[1] = sw; q[2] = sh; q[3] = rot; q[4] = flip;
  }
  g.R = R; g.sw = sw; g.sh = sh; g.rot = rot; g.flip = flip;
  g.X00 = g.Y00 = g.cX = g.cY = g.dX = g.dY = 0;
  if (rot < 0) {
    // unrotated: the mask itself, mirrored for the flips and shifted by s bits
    const int y_off = flip == 2 ? H - 33 - sh : sh - kMaskCentre;
    g.ybase = y_off & ~3;
    const int s = y_off - g.ybase;
    g.xbase = flip == 1 ? W - 33 - sw : sw - kMaskCentre;
    g.c_lo = max(kMaskCentre - R - 2, 0); g.c_hi = min(kMaskCentre + R + 3, kMaskRows - 1);
    g.b_lo = g.c_lo + s; g.b_hi = g.c_hi + s;
  } else {
    const int32_t* c = tb.rot_coeff + (rot >= 360 ? rot % 360 : rot) * 6;
    const int a0 = c[0], a1 = c[1], a2 = c[2], a3 = c[3], a4 = c[4], a5 = c[5];
    // bounding box of the polygon (disc of radius R around the centre) in the
    // FINAL image: forward-map the centre through the rotation and the flip
    const float X = (float)sw * 65536.f - (float)a2, Y = (float)sh * 65536.f - (float)a5;
    // (a bounding box with 3 pixels of slack: an approximate reciprocal will do)
    const float inv_det = __frcp_rn((float)a0 * (float)a4 - (float)a1 * (float)a3);
    float cx = ((float)a4 * X - (float)a1 * Y) * inv_det;
    float cy = ((float)a0 * Y - (float)a3 * X) * inv_det;
    if (flip == 1) cx = (float)(W - 1) - cx;
    if (flip == 2) cy = (float)(H - 1) - cy;
    const int bx0 = max((int)floorf(cx) - R - 3, 0);
    const int bx1 = min(min((int)ceilf(cx) + R + 3, W - 1), bx0 + kRotCols - 1);
    const int by0 = max((int)floorf(cy) - R - 3, 0) & ~3;
    const int by1 = min(min((int)ceilf(cy) + R + 3, H - 1), by0 + 127);
    g.xbase = bx0; g.ybase = by0;
    g.c_lo = 0; g.c_hi = bx1 - bx0;  // may be negative: nothing to draw
    g.b_lo = 0; g.b_hi = by1 - by0;
    const int sx = flip == 1 ? -1 : 1, sy = flip == 2 ? -1 : 1;  // d(fx)/d(x), d(fy)/d(y)
    const int fx0 = flip == 1 ? W - 1 - bx0 : bx0;
    const int fy0 = flip == 2 ? H - 1 - by0 : by0;
    g.dX = a1 * sy; g.dY = a4 * sy;
    g.cX = a0 * sx; g.cY = a3 * sx;
    g.X00 = a2 + a1 * fy0 + a0 * fx0 + (kMaskCentre - sw) * 65536;
    g.Y00 = a5 + a4 * fy0 + a3 * fx0 + (kMaskCentre - sh) * 65536;
  }
  {
    const int ri = min(max(R - tb.r_min, 0), tb.n_radii - 1);
    const int cell = state * tb.n_radii + ri;
    // (the mask ids of ALL vertex variants of the cell, one per lane, are
    // fetched together with the two variant maps instead of after them: one
    // dependent global load less per image)
    const int n_var = tb.n_xvar * tb.n_yvar;
    int cand = 0;
    if (n_var <= 32 && lane < n_var) cand = tb.mask_index[(int64_t)cell * n_var + lane];
    const int xv = tb.xvar[(int64_t)cell * W + min(max(sw, 0), W - 1)];
    const int yv = tb.yvar[(int64_t)cell * H + min(max(sh, 0), H - 1)];
    if (n_var <= 32) g.id = __shfl_sync(0xffffffffu, cand, xv * tb.n_yvar + yv);
    else g.id = tb.mask_index[((int64_t)cell * tb.n_xvar + xv) * tb.n_yvar + yv];
    // A quantised shift can push the polygon up to q-1 pixels over the image
    // edge (Pillow clips it there): clear the mask bits whose pixel lies
    // outside the image, so "inside the mask" implies "inside the image".
    const int lo = max(0, kMaskCentre - sh), hi = min(63, H - 1 + kMaskCentre - sh);
    uint64_t rows = 0;
    if (hi >= lo) rows = (hi - lo == 63 ? ~0ull : ((1ull << (hi - lo + 1)) - 1ull)) << lo;
    g.rows_lo = (uint32_t)rows; g.rows_hi = (uint32_t)(rows >> 32);
  }
  return g;
}

// (10 CTAs = 40 images per SM at 48 registers: the rotation gather keeps more
// shared-memory loads in flight than at 40 registers / 12 CTAs, and 16 384
// images are 2.8 instead of 2.3 waves: 43.0 -> 40.4 us rotated, 33.4 -> 31.2
// us unrotated; 8 CTAs at 59 registers: 39.9 / 32.6 us.  Two warps or one per
// CTA instead of four, so that a slow image does not hold its neighbours'
// slots: 39.7 / 39.5 us rotated, i.e. within 1-2 %.)
//
// kGrouped: the tables come from the image's config group (p.groups, found
// through p.env_group) instead of the kernel parameters.  Each warp copies
// its group's 128-byte descriptor to shared memory before the
// griddepcontrol.wait below -- static tables, like r_thresholds -- so the
// overlap with the step kernel is kept.
static_assert(sizeof(mdpp_image_discrete_group) == 128, "one word per lane");
template <int V, bool kGrouped>  // V: experiment switches (MDPP_RENDER_VARIANT); none at present
__global__ void __launch_bounds__(kRBlock, 10)
render_discrete_kernel(const __grid_constant__ RenderDParams p) {
  __shared__ uint64_t mask_s[kImagesPerCta][kMaskCols];    // polygon column bitmaps
  __shared__ uint64_t fmask_s[kImagesPerCta][kRotCols][2];  // ... of the final image
  __shared__ mdpp_image_discrete_group desc_s[kGrouped ? kImagesPerCta : 1];
  // The next kernel of the stream, when launched with programmatic stream
  // serialisation (the next step kernel), may start its prologue now; it
  // still waits for this grid to complete before touching the env state.
  // (image step(): 45.7 -> 43.3 us rotated, 37.6 -> 36.3 us unrotated)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t m = (int64_t)blockIdx.x * kImagesPerCta + warp;
  if (m >= p.n_images) return;  // whole warp; only warp-level barriers below
  uint64_t* mask = mask_s[warp] + kMaskPad;
  uint64_t (*fmask)[2] = fmask_s[warp];
  int gi = 0;
  if (kGrouped) {  // the image's env (see image_setup) -> its group; used below
    uint32_t e = (uint32_t)m;
    if (p.tb.n_sub_images == 2) e >>= 1;
    else if (p.tb.n_sub_images > 2) e /= (uint32_t)p.tb.n_sub_images;
    if (e >= (uint32_t)p.n_envs) e %= (uint32_t)p.n_envs;  // a [T][N] block
    gi = p.env_group[e];
  }
  const mdpp_image_discrete_tables& tb = kGrouped ? desc_s[warp].tb : p.tb;
  const int W = p.tb.width, H = p.tb.height;
  const int total = W * H;
  uint8_t* out = p.out + m * (int64_t)total;
  // 16-byte zero fill + aligned 4-byte words per column
  const bool fast = total % 16 == 0 && H % 4 == 0;
  // phase 1: the image is mostly background -- stream zeros everywhere, FIRST:
  // these stores need nothing but the output pointer, so they drain while the
  // dependent loads of the set-up below (state -> Philox -> variant maps ->
  // mask id -> mask bits) are in flight.  The warp barriers of the set-up
  // order them before the box stores of phase 2.
  uint4* out4 = reinterpret_cast<uint4*>(out);
  const uint4 z = make_uint4(0u, 0u, 0u, 0u);
  const int n16 = total / 16;
  int zi = lane;  // next 16-byte word this lane zeroes
  // (rotated images: only a third of the fill up front, the rest is issued
  // between the gather iterations so that the stores drain under the math:
  // 68 -> 62 us per 16 384 images against the whole fill first)
  const int n_first = p.tb.has_rotate ? n16 / 3 : n16;
  if (fast) {
    for (; zi + 96 < n_first; zi += 128) {
      __stcs(out4 + zi, z); __stcs(out4 + zi + 32, z);
      __stcs(out4 + zi + 64, z); __stcs(out4 + zi + 96, z);
    }
    if (n_first == n16)
      for (; zi < n16; zi += 32) __stcs(out4 + zi, z);
  }
  for (int w = lane; w < 2 * kRotCols; w += 32) (&fmask[0][0])[w] = 0ull;
  if (lane < kMaskPad) { mask[-1 - lane] = 0ull; mask[kMaskRows + lane] = 0ull; }
  // (static tables may be read ahead of the wait below)
  uint32_t id_base = (uint32_t)p.env_id_offset;
  if (kGrouped) {
    reinterpret_cast<uint32_t*>(&desc_s[warp])[lane] =
        reinterpret_cast<const uint32_t*>(p.groups + gi)[lane];
    __syncwarp();
    id_base += (uint32_t)(desc_s[warp].global_id_base - desc_s[warp].env_begin);
  }
  const double thr0 = tb.has_scale && lane < tb.n_radii - 1 ? tb.r_thresholds[lane]
                                                            : __longlong_as_double(0x7ff0000000000000ll);
  // launched with MDPP_LAUNCH_OVERLAP_PREVIOUS: everything above overlapped the
  // previous kernel of the stream (the step that produces `states`); wait for
  // it now.  Returns at once in an ordinary launch.
  asm volatile("griddepcontrol.wait;" ::: "memory");

  const ImageSetup g = image_setup(p, tb, id_base, m, lane, thr0);
  __syncwarp();  // fmask is cleared
  const int sw = g.sw, sh = g.sh, rot = g.rot, flip = g.flip;
  const int xbase = g.xbase, ybase = g.ybase;
  const int c_lo = g.c_lo, c_hi = g.c_hi, b_lo = g.b_lo, b_hi = g.b_hi;
  {
    const uint64_t rows = ((uint64_t)g.rows_hi << 32) | g.rows_lo;
    const int s = (flip == 2 ? H - 33 - sh : sh - kMaskCentre) & 3;
#pragma unroll
    for (int mc = lane; mc < kMaskRows; mc += 32) {
      uint64_t col = tb.mask_bits[(int64_t)g.id * kMaskRows + mc] & rows;
      if ((unsigned)(mc + sw - kMaskCentre) >= (unsigned)W) col = 0;
      if (rot >= 0) {
        mask[mc] = col;  // source of the rotation gather below
      } else {
        if (flip == 2) col = __brevll(col);
        const int c = flip == 1 ? 63 - mc : mc;
        fmask[c][0] = col << s;
        fmask[c][1] = s ? col >> (64 - s) : 0ull;
      }
    }
  }
  __syncwarp();
  // Rotated images: gather the polygon ONCE into the final-image column
  // bitmaps.  Work item = 16 consecutive rows of one column = one 16-bit slot,
  // owned by exactly one lane (no atomics); the inverse affine of Pillow's
  // NEAREST rotation (16.16 fixed point) is stepped incrementally along y.
  if (rot >= 0 && c_hi >= 0 && b_hi >= 0) {
    const int ncols = c_hi + 1, nrows = b_hi + 1;
    // (rows per work item; 8 measured 8 % slower: more per-item set-up than
    // the tighter fit to the box saves)
    constexpr int kSeg = 16;
    uint16_t* slots = reinterpret_cast<uint16_t*>(&fmask[0][0]);
    const int segs = (nrows + kSeg - 1) / kSeg;  // slots past it stay zero (cleared above)
    // set mask bits (R clamped: replayed parameters are caller-supplied, and
    // the padding of `mask` covers 15 columns beyond this box only)
    const int Rc = min(max(g.R, 0), kMaskCentre - 1);
    const int m_lo = kMaskCentre - Rc - 2, m_hi = kMaskCentre + Rc + 3;
    const int dX = g.dX, dY = g.dY;
    const float inv_segs = 1.0f / (float)segs;
    // Mask bits outside the image were cleared at load, so the image-bounds
    // test of the rotation is implied by the mask lookup.
    for (int w = lane; w < ncols * segs; w += 32) {
      // (w + 0.5) / segs is at least 0.5 / segs away from an integer: exact
      const int c = (int)(((float)w + 0.5f) * inv_segs);
      const int sgm = w - c * segs;
      const int k0 = sgm * kSeg;                            // box-local rows
      int X = g.X00 + c * g.cX + k0 * dX;
      int Y = g.Y00 + c * g.cY + k0 * dY;
      // the 16 samples lie on a segment: if both ends are on the same outer
      // side of the polygon's mask box, none of them can hit a set bit
      const int mxa = X >> 16, mxb = (X + (kSeg - 1) * dX) >> 16;
      const int mya = Y >> 16, myb = (Y + (kSeg - 1) * dY) >> 16;
      uint32_t bits = 0;
      if (!(max(mxa, mxb) < m_lo || min(mxa, mxb) > m_hi ||
            max(mya, myb) < m_lo || min(mya, myb) > m_hi)) {
        // every sample lies between the two ends, i.e. at most 15 columns
        // outside [m_lo, m_hi]: inside the zero padding of `mask`; a row
        // outside 0..63 shifts everything out (shr.b64 clamps its amount).
        // Bit k enters at the top and slides down.
#pragma unroll
        for (int k = 0; k < kSeg; ++k) {
          uint64_t v;
          asm("shr.b64 %0, %1, %2;" : "=l"(v) : "l"(mask[X >> 16]), "r"(Y >> 16));
          bits = __funnelshift_r(bits, (uint32_t)v, 1);
          X += dX; Y += dY;
        }
        bits >>= 32 - kSeg;
        // (rows past the box need no masking: they are exact samples too, and
        // phase 2 stores whole 4-row words up to b_hi only -- inside the image)
      }
      slots[c * 8 + sgm] = (uint16_t)bits;  // little-endian: slot s = bits 16s..
      if (fast) {  // the next slice of the zero fill
#pragma unroll
        for (int q = 0; q < 4; ++q, zi += 32)
          if (zi < n16) __stcs(out4 + zi, z);
      }
    }
    __syncwarp();
  }
  if (fast && n_first != n16) {  // what is left of the zero fill
    for (; zi < n16; zi += 32) __stcs(out4 + zi, z);
    __syncwarp();
  }
  if (fast) {
    // phase 2: the 4-byte words of the box whose nibble is not empty (the
    // barriers above order these stores after the zero fill of phase 1).  No
    // set bit lies outside the image (see the mask load / the gather bounds),
    // so the nibble test is also the bounds test.
    const uint8_t* fb = reinterpret_cast<const uint8_t*>(&fmask[0][0]);
    uint8_t* obase = out + ((int64_t)xbase * H + ybase);
    // 8 lanes per column (a byte of the bitmap = 8 rows = 2 words each), 4
    // columns per pass; boxes taller than 64 rows take a second round.
    // (Two lanes per column with 8 words each: same speed rotated, 25 %
    // slower unrotated.)
    const int sub = lane & 7;
    for (int jb = (b_lo >> 3) + sub; jb <= min(b_hi >> 3, 15); jb += 8) {
      // (rows past b_hi hold samples too, possibly below the image: the upper
      // word of the last byte is dropped when it starts past b_hi)
      const uint32_t keep = 8 * jb + 4 <= b_hi ? 0xFFu : 0x0Fu;
      const int c0 = c_lo + (lane >> 3);
      const uint8_t* src = fb + jb + c0 * 16;
      uint32_t* q = reinterpret_cast<uint32_t*>(obase + 8 * jb + (int64_t)c0 * H);
      // (no "byte != 0" branch around the two predicated stores, running
      // pointers instead of per-column address arithmetic: 40.1 -> 39.1 us)
      for (int c = c0; c <= c_hi; c += 4, src += 64, q += H) {
        const uint32_t byte = *src & keep;
        const uint32_t lo = byte & 0xFu, hi = byte >> 4;
        if (lo) __stcs(q, ((lo * 0x00204081u) & 0x01010101u) * 0xFFu);
        if (hi) __stcs(q + 1, ((hi * 0x00204081u) & 0x01010101u) * 0xFFu);
      }
    }
  } else {  // odd image sizes: one byte per lane and step
    for (int idx = lane; idx < total; idx += 32) {
      const int c = idx / H - xbase, b = idx % H - ybase;
      uint32_t v = 0;
      if ((unsigned)c < (unsigned)kRotCols && (unsigned)b < 128u)
        v = (uint32_t)(fmask[c][b >> 6] >> (b & 63)) & 1u;
      out[idx] = v ? 255 : 0;
    }
  }
}

struct RenderCParams {
  // single-config launch: the configuration; grouped: group 0's (the sizes,
  // dim and dtype are common)
  mdpp_image_continuous_config cfg;
  const mdpp_image_continuous_group* groups;  // grouped launch: the configs
  const uint16_t* env_group;                  //   and the env -> group map
  int64_t n_envs;
  const void* states;
  uint8_t* out;
};

// kGrouped: the CTA first stages its image's group configuration in shared
// memory; everything after that is the single-config kernel.
template <typename R, bool kGrouped>
__global__ void __launch_bounds__(kRBlock)
render_continuous_kernel(const __grid_constant__ RenderCParams p) {
  constexpr int kCfgWords = sizeof(mdpp_image_continuous_config) / 4;
  static_assert(sizeof(mdpp_image_continuous_config) % 16 == 0, "uint4 copy");
  __shared__ __align__(16) uint32_t cfg_s[kGrouped ? kCfgWords : 1];
  const int n_sub = p.cfg.n_sub_images;
  const int64_t m = blockIdx.x / n_sub;
  const int sub = blockIdx.x % n_sub;  // 0 relevant, 1 irrelevant
  if (kGrouped) {
    const int gi = p.env_group[m % p.n_envs];
    const uint4* src = reinterpret_cast<const uint4*>(&p.groups[gi].cfg);
    for (int i = threadIdx.x; i < kCfgWords / 4; i += kRBlock)
      reinterpret_cast<uint4*>(cfg_s)[i] = src[i];
    __syncthreads();
  }
  const mdpp_image_continuous_config& c =
      kGrouped ? *reinterpret_cast<const mdpp_image_continuous_config*>(cfg_s) : p.cfg;
  const int W = c.width, H = c.height;
  const R* st = reinterpret_cast<const R*>(p.states) + m * c.dim;
  // convert_to_pixel (:248-277): ((v - lo) / (hi - lo)) in dtype_s, promoted
  // to float64 by the integer image shape, truncated
  int px[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const R v = st[sub == 0 ? c.rel_index[k] : c.irr_index[k]];
    const R lo = (R)c.feat_low[k], hi = (R)c.feat_high[k];
    R frac;
    if (sizeof(R) == 4) frac = (R)__fdiv_rn(__fsub_rn((float)v, (float)lo),
                                           __fsub_rn((float)hi, (float)lo));
    else frac = (R)__ddiv_rn(__dsub_rn((double)v, (double)lo),
                             __dsub_rn((double)hi, (double)lo));
    px[k] = (int)__dmul_rn((double)frac, (double)(k == 0 ? W : H));
  }
  const int rad = c.stamp_radius;
  const bool rel = sub == 0;
  auto in_stamp = [&](int x, int y, int cx, int cy) -> bool {
    const int r = y - cy + rad;
    if ((unsigned)r >= (unsigned)c.stamp_rows) return false;
    const int dx = x - cx - c.stamp[r][0];
    return (unsigned)dx < (unsigned)c.stamp[r][1];
  };
  auto colour = [&](int x, int y, int ch) -> uint32_t {
    if (in_stamp(x, y, px[0], px[1])) return ch == 2 ? 255u : 0u;  // agent, blue
    if (rel) {
      if (c.has_target && in_stamp(x, y, c.target_pixel[0], c.target_pixel[1]))
        return ch == 1 ? 255u : 0u;                                 // target, green
      for (int b = 0; b < c.n_rects; ++b)
        if (x >= c.rect[b][0] && x <= c.rect[b][2] && y >= c.rect[b][1] &&
            y <= c.rect[b][3])
          return 0u;                                                // terminal, black
    }
    // grid lines (white), drawn first by the reference, so tested last
    if ((unsigned)x < 256u && (unsigned)y < 256u &&
        (((c.vline[sub][x >> 6] >> (x & 63)) | (c.hline[sub][y >> 6] >> (y & 63))) & 1ull))
      return 255u;
    return 208u;
  };
  const int total = W * H * 3;
  uint8_t* out = p.out + ((int64_t)m * c.n_sub_images + sub) * (int64_t)total;
  if (total % 16 == 0) {
    uint4* out4 = reinterpret_cast<uint4*>(out);
    for (int i = threadIdx.x; i < total / 16; i += kRBlock) {
      uint32_t w[4] = {0u, 0u, 0u, 0u};
      int pix = (i * 16) / 3, ch = (i * 16) % 3;
      int x = pix / H, y = pix - x * H;
#pragma unroll
      for (int b = 0; b < 16; ++b) {
        w[b >> 2] |= colour(x, y, ch) << ((b & 3) * 8);
        if (++ch == 3) { ch = 0; if (++y == H) { y = 0; ++x; } }
      }
      __stcs(out4 + i, make_uint4(w[0], w[1], w[2], w[3]));
    }
  } else {
    for (int idx = threadIdx.x; idx < total; idx += kRBlock) {
      const int pix = idx / 3;
      out[idx] = (uint8_t)colour(pix / H, pix % H, idx % 3);
    }
  }
}

}  // namespace mdpp

using namespace mdpp;

namespace {

// The parameters of a discrete render call that do not depend on where the
// tables come from.
void fill_render_params(RenderDParams& p, const int64_t* states,
                        const int32_t* params_in, int32_t* params_out,
                        uint8_t* out, int64_t n_images, int64_t n_envs,
                        int32_t image_stream, const mdpp_step_opts* opts) {
  p.states = states;
  p.params_in = params_in;
  p.params_out = params_out;
  p.out = out;
  p.n_images = n_images;
  p.n_envs = n_envs;
  p.k0 = (uint32_t)opts->seed;
  p.k1 = (uint32_t)(opts->seed >> 32);
  p.stream = (uint32_t)image_stream;
  p.step_index = opts->step_index;
  p.step_index_dev = opts->step_index_dev;
  p.env_id_offset = opts->env_id_offset;
}

template <bool kGrouped>
int launch_render_discrete(mdpp_ctx* ctx, const RenderDParams& p,
                           const mdpp_step_opts* opts, void* cuda_stream) {
  const unsigned grid = (unsigned)((p.n_images + kImagesPerCta - 1) / kImagesPerCta);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kRBlock);
  cfg.stream = (cudaStream_t)cuda_stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (opts->flags & MDPP_LAUNCH_OVERLAP_PREVIOUS) ? 1 : 0;
  static const int variant = [] {  // experiment knob
    const char* e = std::getenv("MDPP_RENDER_VARIANT");
    return e ? std::atoi(e) : 0;
  }();
  switch (variant) {
    case 1: MDPP_CUDA(ctx, cudaLaunchKernelEx(&cfg, render_discrete_kernel<1, kGrouped>, p)); break;
    default: MDPP_CUDA(ctx, cudaLaunchKernelEx(&cfg, render_discrete_kernel<0, kGrouped>, p));
  }
  MDPP_CUDA(ctx, cudaGetLastError());
  return MDPP_OK;
}

template <bool kGrouped>
int launch_render_continuous(mdpp_ctx* ctx, const RenderCParams& p,
                             int64_t n_images, void* cuda_stream) {
  const unsigned grid = (unsigned)(n_images * p.cfg.n_sub_images);
  if (p.cfg.is_f64)
    render_continuous_kernel<double, kGrouped><<<grid, kRBlock, 0, (cudaStream_t)cuda_stream>>>(p);
  else
    render_continuous_kernel<float, kGrouped><<<grid, kRBlock, 0, (cudaStream_t)cuda_stream>>>(p);
  MDPP_CUDA(ctx, cudaGetLastError());
  return MDPP_OK;
}

inline int n_sub_of(const mdpp_image_discrete_tables& tb) {
  return tb.n_sub_images < 1 ? 1 : tb.n_sub_images;
}

}  // namespace

extern "C" int mdpp_render_discrete(mdpp_ctx* ctx,
                                    const mdpp_image_discrete_tables* tb,
                                    const int64_t* states,
                                    const int32_t* params_in,
                                    int32_t* params_out, uint8_t* out,
                                    int64_t n_images, int64_t n_envs,
                                    int32_t image_stream,
                                    const mdpp_step_opts* opts,
                                    void* cuda_stream) {
  if (!ctx) return MDPP_EINVAL;
  if (!tb || !states || !out || !opts || n_images < 1 || n_envs < 1)
    return fail(ctx, MDPP_EINVAL, "render_discrete: bad arguments");
  if (tb->width < 1 || tb->height < 1 || !tb->mask_bits || !tb->mask_index ||
      !tb->xvar || !tb->yvar || !tb->rot_coeff)
    return fail(ctx, MDPP_EINVAL, "render_discrete: incomplete tables");
  if (tb->has_scale && tb->n_radii > 1 && !tb->r_thresholds)
    return fail(ctx, MDPP_EINVAL, "render_discrete: missing r_thresholds");
  if (n_images > 0x7fffffffLL)
    return fail(ctx, MDPP_EINVAL, "render_discrete: too many images per call");
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  RenderDParams p;
  p.tb = *tb;
  p.groups = nullptr;
  p.env_group = nullptr;
  fill_render_params(p, states, params_in, params_out, out, n_images, n_envs,
                     image_stream, opts);
  return launch_render_discrete<false>(ctx, p, opts, cuda_stream);
}

extern "C" int mdpp_render_continuous(mdpp_ctx* ctx,
                                      const mdpp_image_continuous_config* cfg,
                                      const void* states, uint8_t* out,
                                      int64_t n_images, void* cuda_stream) {
  if (!ctx) return MDPP_EINVAL;
  if (!cfg || !states || !out || n_images < 1)
    return fail(ctx, MDPP_EINVAL, "render_continuous: bad arguments");
  if (cfg->n_sub_images < 1 || cfg->n_sub_images > 2 ||
      cfg->stamp_rows > MDPP_MAX_STAMP_ROWS || cfg->n_rects > MDPP_MAX_TERM_BOXES)
    return fail(ctx, MDPP_EINVAL, "render_continuous: bad configuration");
  if (n_images * cfg->n_sub_images > 0x7fffffffLL)
    return fail(ctx, MDPP_EINVAL, "render_continuous: too many images per call");
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  RenderCParams p;
  p.cfg = *cfg;
  p.groups = nullptr;
  p.env_group = nullptr;
  p.n_envs = 0;
  p.states = states;
  p.out = out;
  return launch_render_continuous<false>(ctx, p, n_images, cuda_stream);
}

extern "C" int mdpp_set_image_discrete_groups(mdpp_ctx* ctx,
                                              const mdpp_image_discrete_group* groups,
                                              int32_t n_groups) {
  if (!ctx) return MDPP_EINVAL;
  int rc = validate_groups(ctx, __func__, groups, n_groups, /*env_map=*/true);
  if (rc) return rc;
  const mdpp_image_discrete_tables& t0 = groups[0].tb;
  mdpp_image_discrete_tables first = t0;
  for (int g = 0; g < n_groups; ++g) {
    const mdpp_image_discrete_tables& t = groups[g].tb;
    const std::string which = "set_image_discrete_groups: group " + std::to_string(g);
    if (t.width != t0.width || t.height != t0.height || n_sub_of(t) != n_sub_of(t0))
      return fail(ctx, MDPP_EINVAL, which + " differs from group 0 in width, height "
                  "or n_sub_images");
    if (t.width < 1 || t.height < 1 || t.n_states < 1 || t.n_radii < 1)
      return fail(ctx, MDPP_EINVAL, which + ": bad sizes");
    if (!t.mask_bits || !t.mask_index || !t.xvar || !t.yvar || !t.rot_coeff ||
        (t.has_scale && t.n_radii > 1 && !t.r_thresholds))
      return fail(ctx, MDPP_EINVAL, which + ": missing table pointer");
    first.has_rotate |= t.has_rotate;  // (the kernel's zero-fill schedule)
  }
  rc = install_groups(ctx, ctx->img_d_set, groups, n_groups, /*block=*/0);
  if (rc) return rc;
  ctx->img_d_first = first;
  return MDPP_OK;
}

extern "C" int mdpp_render_discrete_groups(mdpp_ctx* ctx, const int64_t* states,
                                           const int32_t* params_in,
                                           int32_t* params_out, uint8_t* out,
                                           int64_t n_images, int64_t n_envs,
                                           int32_t image_stream,
                                           const mdpp_step_opts* opts,
                                           void* cuda_stream) {
  if (!ctx) return MDPP_EINVAL;
  if (!ctx->img_d_set.groups)
    return fail(ctx, MDPP_EINVAL, "render_discrete_groups: no image groups set");
  if (!states || !out || !opts || n_images < 1 || n_envs < 1)
    return fail(ctx, MDPP_EINVAL, "render_discrete_groups: bad arguments");
  int rc = bind_groups(ctx, ctx->img_d_set, "render_discrete_groups", n_envs);
  if (rc) return rc;
  if (n_images > 0x7fffffffLL)
    return fail(ctx, MDPP_EINVAL, "render_discrete_groups: too many images per call");
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  RenderDParams p;
  p.tb = ctx->img_d_first;
  p.groups = static_cast<const mdpp_image_discrete_group*>(ctx->img_d_set.groups);
  p.env_group = ctx->img_d_set.env_group;
  fill_render_params(p, states, params_in, params_out, out, n_images, n_envs,
                     image_stream, opts);
  return launch_render_discrete<true>(ctx, p, opts, cuda_stream);
}

extern "C" int mdpp_set_image_continuous_groups(mdpp_ctx* ctx,
                                                const mdpp_image_continuous_group* groups,
                                                int32_t n_groups) {
  if (!ctx) return MDPP_EINVAL;
  int rc = validate_groups(ctx, __func__, groups, n_groups, /*env_map=*/true);
  if (rc) return rc;
  const mdpp_image_continuous_config& c0 = groups[0].cfg;
  for (int g = 0; g < n_groups; ++g) {
    const mdpp_image_continuous_config& c = groups[g].cfg;
    const std::string which = "set_image_continuous_groups: group " + std::to_string(g);
    if (c.width != c0.width || c.height != c0.height || c.n_sub_images != c0.n_sub_images)
      return fail(ctx, MDPP_EINVAL, which + " differs from group 0 in width, height "
                  "or n_sub_images");
    if (c.dim != c0.dim || c.is_f64 != c0.is_f64)
      return fail(ctx, MDPP_EINVAL, which + " differs from group 0 in dim or is_f64");
    if (c.width < 1 || c.height < 1 || c.n_sub_images < 1 || c.n_sub_images > 2 ||
        c.stamp_rows > MDPP_MAX_STAMP_ROWS || c.n_rects > MDPP_MAX_TERM_BOXES)
      return fail(ctx, MDPP_EINVAL, which + ": bad configuration");
  }
  rc = install_groups(ctx, ctx->img_c_set, groups, n_groups, /*block=*/0);
  if (rc) return rc;
  ctx->img_c_first = c0;
  return MDPP_OK;
}

extern "C" int mdpp_render_continuous_groups(mdpp_ctx* ctx, const void* states,
                                             uint8_t* out, int64_t n_images,
                                             int64_t n_envs, void* cuda_stream) {
  if (!ctx) return MDPP_EINVAL;
  if (!ctx->img_c_set.groups)
    return fail(ctx, MDPP_EINVAL, "render_continuous_groups: no image groups set");
  if (!states || !out || n_images < 1 || n_envs < 1)
    return fail(ctx, MDPP_EINVAL, "render_continuous_groups: bad arguments");
  int rc = bind_groups(ctx, ctx->img_c_set, "render_continuous_groups", n_envs);
  if (rc) return rc;
  if (n_images * ctx->img_c_first.n_sub_images > 0x7fffffffLL)
    return fail(ctx, MDPP_EINVAL, "render_continuous_groups: too many images per call");
  MDPP_CUDA(ctx, cudaSetDevice(ctx->device));
  RenderCParams p;
  p.cfg = ctx->img_c_first;
  p.groups = static_cast<const mdpp_image_continuous_group*>(ctx->img_c_set.groups);
  p.env_group = ctx->img_c_set.env_group;
  p.n_envs = n_envs;
  p.states = states;
  p.out = out;
  return launch_render_continuous<true>(ctx, p, n_images, cuda_stream);
}
