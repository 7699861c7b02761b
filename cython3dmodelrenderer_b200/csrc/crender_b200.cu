// crender_b200.cu -- B200 (sm_100a) implementation of the Version C rendering hot path of
// oKatanaaa/Cython3DModelRenderer, behind the C ABI in include/crender_b200.h.
//
// Reference being replaced ("pyx" = crender/cy/pixel_buffer_filler/advanced_pixel_buffer_filler.pyx,
// "mu" = crender/cy/pixel_buffer_filler/math_utils.pyx):
//   pyx:106-130  project_on_screen_multithread          -> k_setup (phase 1: transform + projection)
//   pyx:202-211  back-face cull, pixel rectangle         -> k_setup (phase 2: setup, cull, bbox, tile counts)
//   pyx:213-224  per-pixel barycentrics, depth, z-test   -> k_raster (shared-memory tile, 64-bit packed-key min)
//   pyx:226-242  attribute interpolation + buffer writes -> k_raster (deferred shading of the winning triangle)
//
// Design (see DESIGN.md): the reference walks triangles and fights over pixels with per-pixel locks; here the
// screen is cut into TW x TH tiles, every tile is owned by exactly one CTA, visibility is resolved inside shared
// memory with a deterministic min over key = (orderable depth bits << 32 | ~triangle index), and only the winner
// of each pixel is shaded and written -- once, with full 128-byte lines.  Results equal the reference's
// n_threads=1 output bit for bit; all arithmetic is IEEE binary32, one rounding per operation (this file MUST be
// compiled with -fmad=false; divisions and square roots are the correctly rounded defaults).
//
// Not a port: nothing here mirrors the reference's loop structure, locking or memory layout.

#include <cuda.h>
#include <cuda_runtime.h>

#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <atomic>
#include <mutex>
#include <thread>
#include <vector>

#include "crender_b200.h"

// ------------------------------------------------------------------------------------------------------------
// constants
// ------------------------------------------------------------------------------------------------------------
namespace {

constexpr int TW = 32;          // tile width in pixels  (one 128-byte line of z, three of colour / normals)
constexpr int TH = 32;          // tile height in pixels
constexpr int NT = 256;         // threads per CTA in every kernel but the tile rasterizer
// The tile rasterizer is instantiated in two CTA shapes (RasterShape / RasterLarge / RasterSmall, further down); the macros below
// are the large shape's parameters, the CRB_SMALL_* ones the small shape's.
#ifndef CRB_RT
#define CRB_RT 128              // threads per CTA of k_raster (a multiple of 32)
#endif
#ifdef CRB_ABLATION
#define DBG(F, bit) (((F).flags & (bit)) != 0u)
#else
#define DBG(F, bit) ((void)(bit), false)
#endif
constexpr unsigned FLAG_DBG_ONEREC = 0x100000u;   // ablation: every pixel shades from record 0 (measures the cost of the gathers; wrong image)
constexpr unsigned FLAG_DBG_NOCLEAR = 0x10000u, FLAG_DBG_NOSHADE = 0x20000u, FLAG_DBG_NOROWS = 0x40000u, FLAG_DBG_NOOUT = 0x80000u;  // ablation switches (CRB_DEBUG_SKIP)
constexpr unsigned FLAG_OUT_DIRECT = 0x200u;   // experiment: shaded pixels stored straight from registers (12-byte strided stores)
constexpr unsigned FLAG_OUT_TMA = 0x100u;   // internal Frame.flags bit: shaded colour / normal rows leave through TMA boxes
constexpr unsigned CRB_TEX_FLAGS = CRB_TEXTURE | CRB_TEX_PERSPECTIVE | CRB_TEX_BILINEAR | CRB_TEX_TRILINEAR;   // per-pixel texturing and its modes
#ifndef CRB_CH
#define CRB_CH 96               // triangles staged in shared memory per pass of the tile rasterizer
#endif
constexpr unsigned SPLIT_N = 48;  // single-view launches: tiles with more triangles than this are rasterized by SPLIT_BANDS CTAs, 8 rows each
constexpr int SPLIT_BANDS = 4;
#ifndef CRB_CLEAR_EVERY
#define CRB_CLEAR_EVERY 4
#endif
constexpr unsigned CE = CRB_CLEAR_EVERY;  // every CE-th CTA of k_raster is a clear CTA (power of two)
constexpr int WIDE_TILES = 12;    // a triangle whose pixel rectangle touches more tiles than this is binned by its whole warp
constexpr unsigned HEAVY_N = 64;  // tiles with more triangles than this are rasterized first (longest first: shorter kernel tail)
#ifndef CRB_FQ
#define CRB_FQ 256              // fragments a warp compacts per round (8 per row)
#endif
#ifndef CRB_KEY_STRIDE
#define CRB_KEY_STRIDE 35
#endif
// 64-bit keys, row stride 35 = 3 (mod 16 bank pairs): the fragments a warp evaluates together are a few consecutive pixels of
// consecutive rows (a small triangle), and with a shift of three bank pairs per row they spread over all the banks
// (stride 33 shifted one pair per row: 60 % of the key accesses were bank-conflict replays)
constexpr int KEY_STRIDE = CRB_KEY_STRIDE;
constexpr unsigned long long KEY_EMPTY = 0xFFFFFFFFFFFFFFFFull;
constexpr float Z_INIT = 1e6f;  // pyx:67
constexpr float REJ_EPS = 1e-6f;      // fast-reject guard band on barycentric numerators (see tri_fast_setup)
constexpr float L3_MIN = 1e-30f, L3_MAX = 1e30f;
constexpr int MAX_DIM = 65535;  // bbox corners are packed in 16 bits
#ifndef CRB_CLEAR_ROWS
#define CRB_CLEAR_ROWS 16       // rows per TMA box of the fused clear (the constant pattern must fit the staging area it shares)
#endif
constexpr int BOX_ROWS = 8;       // rows per TMA box (clear pattern and shaded rows go out 8 tile rows at a time)
constexpr int HSTAT_WORDS = 4;    // 64-bit words of busy-tile statistics k_raster posts per position in a batch of launches (8 positions)
constexpr size_t HSTAT_BYTES = 8 * HSTAT_WORDS * 8;
constexpr int PROF_MAX = 8192;  // k_raster launches that can be timed between two crb_profile_read calls

static_assert(TW == 32, "a tile row is one warp wide");

// Per-(view,triangle) records written by k_setup.
//   shade record: ONE 128-byte line = 8 float4, everything the shading pass needs for a pixel (a single L2 round trip,
//   prefetched into L1 when a tile stages the triangle):
//     S_A (x0 y0 x1 y1)  S_B (x2 y2 z0 z1)  S_C (z2 l03 l13 l23)      screen-space vertices + denominators of mu:14,17,20
//     S_N0 (n0.xyz n1.x)  S_N1 (n1.yz n2.xy)  S_X (n2.z c0.xyz)  S_C1 (c1.xyz c2.x)  S_C2 (c2.yz flags -)
//                                    (c_k: the colour, or with CRB_TEXTURE (u, v, -), with CRB_TEX_PERSPECTIVE (u*w, v*w, w), w = 1/z)
//   recE (bbox x, bbox y, local, flags)  packed half-open pixel rectangle of a DRAWN triangle; the entries of a 256-triangle chunk are
//                                    dense: chunk c of view v has alive[v,c] entries at [v*T + c*256, ...), entry j = triangle
//                                    c*256 + local (k_fill and the atomic path walk drawn triangles only, with full warps)
enum ShadeRec { S_A = 0, S_B, S_C, S_N0, S_N1, S_X, S_C1, S_C2, SREC };

struct ProjC {
    float p[16];   // row-major 4x4, proj_mat of pyx:85-90
    float xs, ys;  // (float)(w/2.0), (float)(h/2.0)  pyx:109
};

struct Frame {
    ProjC proj;
    int W, H;            // full image size
    int row0, row1;      // rows owned by this filler (band); buffers hold rows [row0,row1)
    int tilesX, tilesY, nTiles;
    long long T;         // triangles per view
    int nViews;
    unsigned flags;
    // inputs
    const float *v, *c, *n;     // [T,3,3]
    const float *views;         // [nViews,16] or nullptr
    // scratch
    // per-(view,triangle) records (see enum ShadeRec)
    float4 *shrec;              // [nViews*T*8] shade records
    float4 *recE;               // [nViews*T]
    unsigned short *alive;      // [nViews*ceil(T/NT)] drawn triangles of the chunk (k_setup CTA): recE holds that many entries for it
    unsigned *chunks;           // band-sharded single view: [0] = number of 256-triangle chunks that may reach the band,
                                // [1..] their indices (k_band_chunks); nullptr = every chunk is visited (grid = chunks)
    unsigned *count;            // [nViews*nTiles] triangles per tile, accumulated by k_setup, returned to zero by k_alloc
    uint4 *busy;                // [nViews*nTiles] compacted busy tiles: (view:10 ty:11 tx:11, triangles, list offset, -); count in total[2]
    uint4 *busyH;               // [nViews*nTiles] the same for tiles with more than HEAVY_N triangles; count in total[4]
    unsigned gridHeavy;         // rasterizing CTA roles [0, gridHeavy) walk busyH, the others walk busy
    unsigned splitHeavy;        // k_alloc emits SPLIT_BANDS row-band records for tiles with more than SPLIT_N triangles
    unsigned *empty;            // [nViews*nTiles] compacted tiles without triangles (same packing); count in total[3]
    unsigned *offset;           // [nViews*nTiles] start of the tile's list
    unsigned *cursor;           // [nViews*nTiles] fill cursor
    float4 *ls;                 // [pairCap*4] staged triangle setups, tile by tile, ONE 64-byte entry (two whole 32-byte sectors, written
                                // by one thread) per (triangle, tile) pair: (x0 y0 x1 y1) (x2 y2 z0 z1) (z2 d1 d2 d3) (bbox x, bbox y,
                                // triangle index, flags) -- d = sign-normalised denominators; their reciprocals are formed when a tile
                                // stages the entry (rcp.rn: three instructions' worth per entry instead of 16 more bytes per pair)
    uint4 *wide;                // [wideCap] triangles that span more than WIDE_TILES tiles, handed by k_fill to k_fill_wide: (view, triangle,
                                // bbox x, bbox y); their number in total[5].  wideCap == 0: k_fill scatters them itself (no k_fill_wide launch)
    unsigned wideCap;
    unsigned long long *total;  // [0] pairs of this frame, [1] sticky max of overflowing totals, [2] busy tiles, [3] empty tiles
    unsigned long long *hstats; // mapped host word: (tiles of the launch << 32 | busy tiles), posted by k_raster for the next launch's grid size
    long long pairCap;
    // outputs (per view slab stride = rows*W (z) or rows*W*3)
    float *z, *color, *normals;
    unsigned char *color_u8;
    long long slabPixels;       // rows*W
    // row exchange of the uint8 image (crb_set_u8_exchange): u8xN > 0 = image row r of view k goes to row band d = r / u8xRows,
    // i.e. to u8x[d] + ((k * u8xRows + r - d * u8xRows) * W + x) * 3 -- u8x[d] is rank d's receive buffer (peer memory)
    unsigned char *u8x[CRB_MAX_EXCHANGE];
    int u8xN, u8xRows;
    float light[3];
    // per-pixel texturing (CRB_TEXTURE): packed texels B | G << 8 | R << 16, [texH, texW] (crb_pack_texture / crb_bind_texture);
    // `c` then holds (u, v, ignored) per corner (the record's colour slots: the same, or (u/z, v/z, 1/z) with CRB_TEX_PERSPECTIVE).
    // Kept last so that every other member keeps its offset.
    const uint32_t *tex;
    // With CRB_TEX_TRILINEAR `tex` is a whole mip chain (crb_bind_texture_mips) of the [texH, texW] texture: its layout follows
    // from the size alone (mip_step), so the Frame -- every kernel's parameter block -- does not grow.
    int texH, texW;
};

// ------------------------------------------------------------------------------------------------------------
// device arithmetic shared by every path.  Operation order restates the reference exactly.
// ------------------------------------------------------------------------------------------------------------

// pyx:116-130.  Source and destination alias in the reference (project_on_screen_multithread(triangles, triangles)),
// so column j sees the components columns < j already overwrote; restated literally (matters for inf/NaN inputs).
__device__ __forceinline__ void project_vertex(const ProjC &P, float &x, float &y, float &z)
{
    const float z0 = z;
    float X = ((x * P.p[0] + y * P.p[4]) + z * P.p[8]) + P.p[12];
    float Y = ((X * P.p[1] + y * P.p[5]) + z * P.p[9]) + P.p[13];
    float Z = ((X * P.p[2] + Y * P.p[6]) + z * P.p[10]) + P.p[14];
    X = X / z0;
    Y = Y / z0;
    Z = Z / z0;
    X = X + 1.0f;
    Y = Y + 1.0f;
    x = X * P.xs;
    y = Y * P.ys;
    z = Z;
}

// Batched views: v' = R (v - p) + q, evaluated ((r0*d0 + r1*d1) + r2*d2) + q   (crender_b200.h, crb_render_views)
__device__ __forceinline__ void view_point(const float *M, float &x, float &y, float &z)
{
    const float dx = x - M[9], dy = y - M[10], dz = z - M[11];
    x = ((M[0] * dx + M[1] * dy) + M[2] * dz) + M[12];
    y = ((M[3] * dx + M[4] * dy) + M[5] * dz) + M[13];
    z = ((M[6] * dx + M[7] * dy) + M[8] * dz) + M[14];
}
__device__ __forceinline__ void view_normal(const float *M, float &x, float &y, float &z)
{
    const float nx = x, ny = y, nz = z;
    x = (M[0] * nx + M[1] * ny) + M[2] * nz;
    y = (M[3] * nx + M[4] * ny) + M[5] * nz;
    z = (M[6] * nx + M[7] * ny) + M[8] * nz;
}

// (int)ceil(x) as the reference binary performs it (pyx:165-166): x86-64 cvttsd2si yields INT_MIN for anything
// outside int range (the C cast is undefined there); CUDA's cvt would saturate instead, so the range test is explicit.
__device__ __forceinline__ int ceil_to_int_ref(float x)
{
    const float c = ceilf(x);
    if (!(c >= -2147483648.0f && c < 2147483648.0f)) return INT_MIN;
    return (int)c;
}
__device__ __forceinline__ int clipi(int a, int lo, int hi) { return a < lo ? lo : (a > hi ? hi : a); }

// Depth -> 32-bit key whose unsigned order equals the float order the reference's `new_z > z_buffer` uses.
// -0.0 is folded onto +0.0 first (they compare equal in the reference, so the triangle index must break the tie).
__device__ __forceinline__ unsigned depth_key(float z)
{
    const unsigned b = __float_as_uint(__fadd_rn(z, 0.0f));        // -0.0 + 0.0 = +0.0, every other value unchanged (z is never NaN here)
    return b ^ ((unsigned)((int)b >> 31) | 0x80000000u);
}
__device__ __forceinline__ unsigned long long pack_key(float z, unsigned tri)
{
    return ((unsigned long long)depth_key(z) << 32) | (unsigned long long)(~tri);
}

// mu:5-34, all three coordinates of one pixel, plain restatement (used by shading and by the atomic path).
struct Tri9 {
    float x0, y0, x1, y1, x2, y2, z0, z1, z2;
};
__device__ __forceinline__ void barycentric(const Tri9 &t, float px, float py, float &b1, float &b2, float &b3)
{
    const float l01 = t.x1 - t.x2, l02 = t.y1 - t.y2;
    const float l03 = l01 * (t.y0 - t.y2) - l02 * (t.x0 - t.x2);
    const float l11 = t.x2 - t.x0, l12 = t.y2 - t.y0;
    const float l13 = l11 * (t.y1 - t.y0) - l12 * (t.x1 - t.x0);
    const float l21 = t.x0 - t.x1, l22 = t.y0 - t.y1;
    const float l23 = l21 * (t.y2 - t.y1) - l22 * (t.x2 - t.x1);
    b1 = (l01 * (py - t.y2) - l02 * (px - t.x2)) / l03;
    b2 = (l11 * (py - t.y0) - l12 * (px - t.x0)) / l13;
    b3 = (l21 * (py - t.y1) - l22 * (px - t.x1)) / l23;
}

__device__ __forceinline__ Tri9 load_tri9(const Frame &F, long long ridx)
{
    const float4 *R = F.shrec + ridx * SREC;
    const float4 a = R[S_A], b = R[S_B], c = R[S_C];
    Tri9 t;
    t.x0 = a.x; t.y0 = a.y; t.x1 = a.z; t.y1 = a.w;
    t.x2 = b.x; t.y2 = b.y; t.z0 = b.z; t.z1 = b.w;
    t.z2 = c.x;
    return t;
}

// flags of a triangle record / staged triangle
constexpr unsigned FL_NEG = 1u;      // bits 0..2: barycentric k is evaluated with negated edge vector and denominator
constexpr unsigned FL_REJ = 16u;     // bits 4..6: barycentric k may use the division-free rejection (denominator sane)
constexpr unsigned FL_SPAN = 256u;   // row spans may be bounded analytically (all three sane, coordinates <= 2^18)
constexpr unsigned FL_FDIV = 512u;   // all three denominators in [2^-40, 2^40]: div_rn_by() applies
constexpr float SPAN_COORD_MAX = 262144.0f;  // 2^18: beyond this the float span bounds lose sub-pixel accuracy
constexpr float FDIV_LO = 9.094947e-13f, FDIV_HI = 1.099511627776e12f;  // 2^-40, 2^40

// Correctly rounded a/d from r = rcp.rn(d), without the division routine: q0 = RN(a*r) is within 2 ulp of a/d; one
// residual step (e = a - d*q exactly via FMA, q += e*r) makes it faithful (<= 1 ulp), and Markstein's theorem then says
// a second step from a faithful quotient with a correctly rounded reciprocal returns RN(a/d) itself.  Preconditions
// (checked by the callers): |d| and |a| in [2^-40, 2^40], so no intermediate overflows, underflows or is subnormal.
// tests/test_gpu_parity.py::test_fast_division_is_ieee checks it against div.rn on ~4e9 operand pairs.
__device__ __forceinline__ float div_rn_by(float a, float d, float r)
{
    float q = a * r;
    float e = __fmaf_rn(-d, q, a);
    q = __fmaf_rn(e, r, q);
    e = __fmaf_rn(-d, q, a);
    return __fmaf_rn(e, r, q);
}
__device__ __forceinline__ bool fdiv_ok_lo(float n1, float n2, float n3)
{
    return fminf(fminf(fabsf(n1), fabsf(n2)), fabsf(n3)) >= FDIV_LO;   // NaN: false
}
__device__ __forceinline__ bool fdiv_ok(float n1, float n2, float n3)
{
    const float a1 = fabsf(n1), a2 = fabsf(n2), a3 = fabsf(n3);
    return fminf(fminf(a1, a2), a3) >= FDIV_LO && fmaxf(fmaxf(a1, a2), a3) <= FDIV_HI;   // NaN: false
}

// astype('int32') of a float32 on x86-64 (cvttss2si): INT32_MIN for NaN and out-of-range values -- the conversion of
// model.py:147-150's texel rule (ingest_b200.cu's k_vertex_colors states it the same way).
__device__ __forceinline__ int f32_to_i32_x86(float x)
{
    if (!(x > -2147483904.0f && x < 2147483648.0f)) return INT_MIN;
    return (int)x;
}

// Shading mode of shade_fragment / k_raster / k_shade_atomic: per-vertex colours (TEX_NONE), or per-pixel texturing
// (CRB_TEXTURE) with nearest (model.py:147-150's rule) or bilinear (CRB_TEX_BILINEAR) sampling, either of them with
// TEX_PERSP (CRB_TEX_PERSPECTIVE) added, and trilinear mip filtering (CRB_TEX_TRILINEAR) with or without it.  All are
// compile-time: a uniform branch on the divide costs the nearest instantiation of the large rasterizer shape a register.
enum TexMode { TEX_NONE = 0, TEX_NEAREST = 1, TEX_BILINEAR = 2, TEX_PERSP = 4, TEX_TRILINEAR = 8 };

// Texel (r, c) of a packed [th, tw] level as float B, G, R
__device__ __forceinline__ void texel_bgr(const uint32_t *tex, int tw, int r, int c, float t[3])
{
    const uint32_t p = __ldg(tex + (r * tw + c));     // th * tw < 2^31 (crb_bind_texture)
    t[0] = (float)(p & 255u); t[1] = (float)((p >> 8) & 255u); t[2] = (float)(p >> 16);
}

// CRB_TEX_BILINEAR (DESIGN 2): texel centres at (col + 0.5) / tw, (row + 0.5) / th -- those of the nearest rule -- clamped to
// the border texels.  float32, one rounding per operation, no FMA (the file is built with -fmad=false).
__device__ __forceinline__ void sample_bilinear(const uint32_t *tex, int H, int W, float u, float v, float c[3])
{
    const float tw = (float)W, th = (float)H;
    float sx = u * tw - 0.5f, sy = (1.0f - v) * th - 0.5f;
    sx = fminf(fmaxf(sx, -1.0f), tw);       // fmaxf(NaN, -1) = -1
    sy = fminf(fmaxf(sy, -1.0f), th);
    const float x0 = floorf(sx), y0 = floorf(sy);
    const float fx = sx - x0, fy = sy - y0, gx = 1.0f - fx, gy = 1.0f - fy;     // (sx - x0 is exact unless -1 < sx < 0)
    const long long ix = (long long)x0, iy = (long long)y0;                      // in [-1, 2^31]
    const int c0 = (int)min(max(ix, 0ll), (long long)W - 1), c1 = (int)min(max(ix + 1, 0ll), (long long)W - 1);
    const int r0 = (int)min(max(iy, 0ll), (long long)H - 1), r1 = (int)min(max(iy + 1, 0ll), (long long)H - 1);
    float t00[3], t01[3], t10[3], t11[3];
    texel_bgr(tex, W, r0, c0, t00); texel_bgr(tex, W, r0, c1, t01);
    texel_bgr(tex, W, r1, c0, t10); texel_bgr(tex, W, r1, c1, t11);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float top = t00[k] * gx + t01[k] * fx, bot = t10[k] * gx + t11[k] * fx;
        c[k] = top * gy + bot * fy;
    }
}

// CRB_TEX_TRILINEAR (DESIGN 2): level of detail of a pixel from the screen-space derivatives of (u, v) -- ux = du/dx etc. --
// clamped to the chain: lc = fmin(fmax(0.5 * L2(r2), 0), L-1), r2 = fmax(|(ux*tw, vx*th)|^2, |(uy*tw, vy*th)|^2), with the
// piecewise-linear log2 L2(f * 2^k) = (k - 1) + (2f - 1), f in [0.5, 1) (frexp; exact at powers of two).  r2 = 0, +inf and NaN
// give L2 = -2, +inf and NaN here, which clamp to the same lc as the definition's -inf, +inf and NaN.
__device__ __forceinline__ float mip_lod(const Frame &F, float ux, float vx, float uy, float vy)
{
    const float p = ux * (float)F.texW, q = vx * (float)F.texH, r = uy * (float)F.texW, s = vy * (float)F.texH;
    const float r2 = fmaxf(p * p + q * q, r * r + s * s);
    int k;
    const float f = frexpf(r2, &k);
    const float l2 = (float)(k - 1) + (2.0f * f - 1.0f);
    return fminf(fmaxf(0.5f * l2, 0.0f), (float)(31 - __clz(max(F.texH, F.texW))));    // L - 1; fmaxf(NaN, 0) = 0
}

// The next level of a chain from level (p, h, w): levels are stored back to back, each max(1, h >> 1) x max(1, w >> 1)
__device__ __forceinline__ const uint32_t *mip_step(const uint32_t *p, int &h, int &w)
{
    p += h * w;
    h = max(1, h >> 1); w = max(1, w >> 1);
    return p;
}

// CRB_TEX_TRILINEAR: bilinear samples of levels l0 = floor(lc) and l1 = min(l0 + 1, L-1), blended c0*(1 - fr) + c1*fr,
// fr = lc - l0.  With fr == 0 that is c0 bit for bit (texels are finite and >= 0), so the second level is not read.
__device__ __forceinline__ void sample_trilinear(const Frame &F, float lc, float u, float v, float c[3])
{
    const int l0 = (int)floorf(lc);
    const float fr = lc - (float)l0;
    int h = F.texH, w = F.texW;
    const uint32_t *p = F.tex;
    for (int l = 0; l < l0; ++l) p = mip_step(p, h, w);
    sample_bilinear(p, h, w, u, v, c);
    if (fr != 0.0f) {   // then lc < L-1, so l1 = l0 + 1
        p = mip_step(p, h, w);
        float c1[3];
        sample_bilinear(p, h, w, u, v, c1);
#pragma unroll
        for (int k = 0; k < 3; ++k) c[k] = c[k] * (1.0f - fr) + c1[k] * fr;
    }
}

// pyx:215-242 for the pixel's winning triangle: barycentrics (mu:5-34), depth, colour, normal (left-associated sums).
// Returns false if the fragment would not have been drawn (some barycentric < 0, NaN depth) -- cannot happen for a key
// that won, kept as a guard.  All operands come from the triangle's 128-byte shade record.
// TEX != TEX_NONE (per-pixel texturing, CRB_TEXTURE; an extension, DESIGN 2): the interpolated colour slots hold (u, v, -), or
// with CRB_TEX_PERSPECTIVE (U, V, W) = (u/z, v/z, 1/z), divided back to u = U/W, v = V/W; the texel they name (nearest) or
// the bilinear blend of the four around them replaces the colour before the fused Guro pass.  Compiled in only where asked
// for, so the per-vertex instantiations are the code they were.
template <int TEX = TEX_NONE>
__device__ __forceinline__ bool shade_fragment(const Frame &F, const float4 *R, float px, float py, float &z, float c[3], float n[3])
{
    const float4 A = R[S_A], B = R[S_B], C = R[S_C];
    // x0=A.x y0=A.y x1=A.z y1=A.w x2=B.x y2=B.y z0=B.z z1=B.w z2=C.x  l03=C.y l13=C.z l23=C.w
    const float n1 = (A.z - B.x) * (py - B.y) - (A.w - B.y) * (px - B.x);
    const float n2 = (B.x - A.x) * (py - A.y) - (B.y - A.y) * (px - A.x);
    const float n3 = (A.x - A.z) * (py - A.w) - (A.y - A.w) * (px - A.z);
    const float b1 = n1 / C.y, b2 = n2 / C.z, b3 = n3 / C.w;
    if (b1 < 0.0f || b2 < 0.0f || b3 < 0.0f) return false;
    z = (B.z * b1 + B.w * b2) + C.x * b3;
    if (z != z) return false;
    const float4 N0 = R[S_N0], N1 = R[S_N1], X = R[S_X], C1 = R[S_C1], C2 = R[S_C2];
    n[0] = (N0.x * b1 + N0.w * b2) + N1.z * b3;
    n[1] = (N0.y * b1 + N1.x * b2) + N1.w * b3;
    n[2] = (N0.z * b1 + N1.y * b2) + X.x * b3;
    c[0] = (X.y * b1 + C1.x * b2) + C1.w * b3;
    c[1] = (X.z * b1 + C1.y * b2) + C2.x * b3;
    c[2] = (X.w * b1 + C1.z * b2) + C2.y * b3;
    if (TEX != TEX_NONE) {
        float u = c[0], v = c[1];
        if (TEX & TEX_PERSP) { u = c[0] / c[2]; v = c[1] / c[2]; }    // correctly rounded (-prec-div=true)
        if (TEX & TEX_TRILINEAR) {
            // barycentric gradients: d(b1, b2, b3)/dx = ((y2-y1)/l03, (y0-y2)/l13, (y1-y0)/l23), d/dy = ((x1-x2)/l03, ...)
            const float gx0 = (B.y - A.w) / C.y, gx1 = (A.y - B.y) / C.z, gx2 = (A.w - A.y) / C.w;
            const float gy0 = (A.z - B.x) / C.y, gy1 = (B.x - A.x) / C.z, gy2 = (A.x - A.z) / C.w;
            float ux = (X.y * gx0 + C1.x * gx1) + C1.w * gx2, vx = (X.z * gx0 + C1.y * gx1) + C2.x * gx2;
            float uy = (X.y * gy0 + C1.x * gy1) + C1.w * gy2, vy = (X.z * gy0 + C1.y * gy1) + C2.x * gy2;
            if (TEX & TEX_PERSP) {   // d(U/W) = (dU - u dW) / W
                const float wx = (X.w * gx0 + C1.z * gx1) + C2.y * gx2, wy = (X.w * gy0 + C1.z * gy1) + C2.y * gy2;
                ux = (ux - u * wx) / c[2]; vx = (vx - v * wx) / c[2];
                uy = (uy - u * wy) / c[2]; vy = (vy - v * wy) / c[2];
            }
            sample_trilinear(F, mip_lod(F, ux, vx, uy, vy), u, v, c);
        } else if (TEX & TEX_BILINEAR) {
            sample_bilinear(F.tex, F.texH, F.texW, u, v, c);
        } else {   // row = clip(int32((1 - v) * th), 0, th-1), col = clip(int32(u * tw), 0, tw-1); BGR as cv2.imread gives it
            const int row = clipi(f32_to_i32_x86((1.0f - v) * (float)F.texH), 0, F.texH - 1);
            const int col = clipi(f32_to_i32_x86(u * (float)F.texW), 0, F.texW - 1);
            texel_bgr(F.tex, F.texW, row, col, c);
        }
    }
    if (F.flags & CRB_GURO) {  // guro_illumination.py:23-27 (float32, left-to-right sums)
        // np.sum accumulates from the identity +0.0 (all -0.0 products sum to +0.0, not -0.0)
        const float dot = (__fadd_rn(0.0f, n[0] * F.light[0]) + n[1] * F.light[1]) + n[2] * F.light[2];
        const float nrm = sqrtf((n[0] * n[0] + n[1] * n[1]) + n[2] * n[2]);
        float s = dot / (nrm + 1e-6f);
        if (s < 0.0f) s = 0.0f;
        if (s > 1.0f) s = 1.0f;
        c[0] *= s; c[1] *= s; c[2] *= s;
    }
    return true;
}

// Colour of a pixel no triangle covers.  Plain renders: 0 (pyx:66).  With the fused Guro pass the reference still runs
// draw_illumination over the whole buffer: normal (0,0,0) gives np.sum(...) = +0.0 whatever the signs of the light
// (the sum starts from the identity +0.0), shadow = clip(+0 / (0 + 1e-6)) = +0 and 0 * +0 = +0.
__device__ __forceinline__ float background_color(const Frame &)
{
    return 0.0f;
}

// run.py:26 .astype('uint8'): C truncation toward zero, then the low 8 bits.  NumPy on x86-64 truncates with cvttss2si, which
// yields INT_MIN (low byte 0) for NaN and for anything outside int range; CUDA's cvt.rzi saturates instead (3e9 and +inf would
// give 255), so the range test is explicit, as in ceil_to_int_ref.
__device__ __forceinline__ unsigned char to_u8(float c)
{
    return (unsigned char)(c >= -2147483648.0f && c < 2147483648.0f ? (int)c : INT_MIN);
}

// Address of pixel (x, image row yl of the band's buffers) of view `view` in the flipped uint8 image (run.py:26 image[::-1]):
// the caller's [views,rows,W,3] array, or -- row exchange -- the receive buffer of the rank that owns the image row.
__device__ __forceinline__ unsigned char *u8_pixel(const Frame &F, int view, int yl, int x)
{
    const int fr = F.row1 - F.row0 - 1 - yl;
    if (F.u8xN) {
        const int d = fr / F.u8xRows;
        return F.u8x[d] + (((long long)view * F.u8xRows + (fr - d * F.u8xRows)) * F.W + x) * 3;
    }
    return F.color_u8 + ((long long)view * F.slabPixels + (long long)fr * F.W + x) * 3;
}

// ------------------------------------------------------------------------------------------------------------
// K1+K2: vertex transform + projection, triangle setup, cull, bbox, per-tile counts
// ------------------------------------------------------------------------------------------------------------

// Coalesced, float4-vectorised staging of a CTA's contiguous run of [.,3,3] floats into shared memory.
__device__ __forceinline__ void stage_floats(const float *__restrict__ g, long long first, long long count, float *s)
{
    const float *src = g + first;
    if (count == (long long)NT * 9 && (reinterpret_cast<uintptr_t>(src) & 15u) == 0) {
        // a full chunk (the usual case): 576 float4, every thread's two or three loads in flight together, 32-bit indices
        const float4 *s4 = reinterpret_cast<const float4 *>(src);
        const unsigned t = threadIdx.x;
        const float4 a = __ldg(s4 + t), b = __ldg(s4 + t + NT);
        float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t < NT * 9 / 4 - 2 * NT) c = __ldg(s4 + t + 2 * NT);
        reinterpret_cast<float4 *>(s)[t] = a;
        reinterpret_cast<float4 *>(s)[t + NT] = b;
        if (t < NT * 9 / 4 - 2 * NT) reinterpret_cast<float4 *>(s)[t + 2 * NT] = c;
    } else if ((reinterpret_cast<uintptr_t>(src) & 15u) == 0) {
        const long long n4 = count >> 2;
        const float4 *s4 = reinterpret_cast<const float4 *>(src);
        for (long long i = threadIdx.x; i < n4; i += NT) reinterpret_cast<float4 *>(s)[i] = __ldg(s4 + i);
        for (long long i = (n4 << 2) + threadIdx.x; i < count; i += NT) s[i] = __ldg(src + i);
    } else {
        for (long long i = threadIdx.x; i < count; i += NT) s[i] = __ldg(src + i);
    }
}

__device__ __forceinline__ void tile_span(const Frame &F, unsigned bx, unsigned by, int &tx0, int &tx1, int &ty0, int &ty1)
{
    const int xl = bx & 0xFFFF, xr = bx >> 16, yt = by & 0xFFFF, yb = by >> 16;
    tx0 = xl / TW;
    tx1 = (xr - 1) / TW;
    ty0 = (yt - F.row0) / TH;
    ty1 = (yb - 1 - F.row0) / TH;
}

// ---- 1-D bulk copies global -> shared (TMA without a tensor map) and the mbarrier they complete on ----------------
constexpr int BC_STAGES = 4;
constexpr unsigned BC_BYTES = NT * 9 * 4;

__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned phase)
{
    const unsigned a = (unsigned)__cvta_generic_to_shared(bar);
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(a), "r"(phase) : "memory");
}
// one bulk copy global -> shared of `bytes` (16-byte multiple, both addresses 16-byte aligned), completion on `bar`
__device__ __forceinline__ void bulk_load(void *smem_dst, const void *gmem_src, unsigned bytes, unsigned long long *bar)
{
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst), m = (unsigned)__cvta_generic_to_shared(bar);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(m), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(d), "l"(gmem_src),
                 "r"(bytes), "r"(m) : "memory");
}

// Positions of the threads whose flag is set, in thread order (warp ballots + one shared-memory word per warp), and their number.
// Two block barriers; every thread of the CTA must call it.
__device__ __forceinline__ unsigned block_compact(const bool flag, unsigned *wsum, unsigned &total)
{
    const unsigned lane = threadIdx.x & 31u, wid = threadIdx.x >> 5;
    const unsigned b = __ballot_sync(0xFFFFFFFFu, flag);
    if (lane == 0) wsum[wid] = __popc(b);
    __syncthreads();
    unsigned base = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < NT / 32; ++w) {
        const unsigned c = wsum[w];
        if (w < (int)wid) base += c;
        tot += c;
    }
    total = tot;
    __syncthreads();
    return base + __popc(b & ((1u << lane) - 1u));
}

// One chunk of NT consecutive triangles of one view.  Every early exit below is taken by the whole CTA or lies behind
// the last barrier, so the function can be called in a loop (chunk-list mode).  PERSP: the colour slots of the record get
// the perspective-correct texture coordinates of CRB_TEX_PERSPECTIVE.
template <bool PERSP>
__device__ __forceinline__ void setup_chunk(const Frame &F, const int view, const long long chunk, const long long chunksPerView,
                                            float *sv, float *sn, float *sc, float *sM, unsigned char *slist, unsigned *wsum,
                                            const bool staged)
{
    const long long first = chunk * NT;
    const long long cnt = min((long long)NT, F.T - first);
    // A band-sharded filler (SURVEY 8e) sees every triangle of the frame but draws only those that reach its rows: there
    // the vertices are staged and tested first, and a CTA whose 256 triangles all miss the band stops before it has read
    // a normal or written a record (7 of 8 CTAs at N = 8).  A full-frame filler stages both arrays behind one barrier.
    const bool banded = F.row0 > 0 || F.row1 < F.H;
    unsigned short *alive = F.alive + (long long)view * chunksPerView + chunk;
    // `staged`: the chunk's vertices, normals and colours already lie in sv / sn / sc (k_setup's ring of bulk copies: the loads of
    // this chunk travelled while the previous one was being set up); anything else is staged here by the threads.
    if (!staged) {
        stage_floats(F.v, first * 9, cnt * 9, sv);
        if (!banded) stage_floats(F.n, first * 9, cnt * 9, sn);
    }
    if (F.views && threadIdx.x < 16) sM[threadIdx.x] = F.views[view * 16 + threadIdx.x];
    __syncthreads();
    // `me`: the triangle of the chunk this thread sets up (-1: none).  A full-frame filler culls first (pyx:202-204 needs only
    // the z of the three view-space normals) and hands the survivors to the first threads, so that the projection, the
    // denominators and the record stores below run in full warps for the ~half of a closed mesh that faces the camera
    // instead of in every warp at half occupancy.  (A band-sharded filler tests the rows first, see above.)
    int me = threadIdx.x < cnt ? (int)threadIdx.x : -1;
    unsigned kept = 0;
    if (!banded) {
        bool keep = false;
        if (me >= 0) {
            const float *q = sn + me * 9;
            float z0 = q[2], z1 = q[5], z2 = q[8];
            if (F.views) {   // view_normal, z row only
                z0 = (sM[6] * q[0] + sM[7] * q[1]) + sM[8] * q[2];
                z1 = (sM[6] * q[3] + sM[7] * q[4]) + sM[8] * q[5];
                z2 = (sM[6] * q[6] + sM[7] * q[7]) + sM[8] * q[8];
            }
            keep = !(((z0 + z1) + z2) >= 0.0f);
        }
        const unsigned pos = block_compact(keep, wsum, kept);
        if (kept == 0) {
            if (threadIdx.x == 0) *alive = 0;
            return;
        }
        if (keep) slist[pos] = (unsigned char)me;
        __syncthreads();
        me = threadIdx.x < kept ? (int)slist[threadIdx.x] : -1;
    }
    const bool valid = me >= 0;
    const int mi = valid ? me : 0;
    const long long tri = first + mi;
    const long long ridx = (long long)view * F.T + tri;
    float x[3], y[3], z[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        if (!valid) { x[k] = y[k] = z[k] = 1.0f; continue; }
        x[k] = sv[mi * 9 + k * 3 + 0];
        y[k] = sv[mi * 9 + k * 3 + 1];
        z[k] = sv[mi * 9 + k * 3 + 2];
        if (F.views) view_point(sM, x[k], y[k], z[k]);
        project_vertex(F.proj, x[k], y[k], z[k]);
    }

    // pyx:132-175: running min from (w,h), running max from 0; NaN never wins a comparison
    float fxl = (float)F.W, fxr = 0.0f, fyt = (float)F.H, fyb = 0.0f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        if (x[k] < fxl) fxl = x[k];
        if (x[k] > fxr) fxr = x[k];
        if (y[k] < fyt) fyt = y[k];
        if (y[k] > fyb) fyb = y[k];
    }
    int xl = clipi(ceil_to_int_ref(fxl), 0, F.W), xr = clipi(ceil_to_int_ref(fxr), 0, F.W);
    int yt = clipi(ceil_to_int_ref(fyt), 0, F.H), yb = clipi(ceil_to_int_ref(fyb), 0, F.H);
    yt = max(yt, F.row0);  // band sharding: rows outside [row0,row1) belong to another filler
    yb = min(yb, F.row1);
    bool drawn = valid && (xl < xr) && (yt < yb);  // pyx:209-211 and the empty range() cases
    if (banded) {
        if (!__syncthreads_or(drawn ? 1 : 0)) {
            if (threadIdx.x == 0) *alive = 0;
            return;
        }
        if (!staged) {
            stage_floats(F.n, first * 9, cnt * 9, sn);
            __syncthreads();
        }
    }
    // pyx:202-204: (n0z + n1z + n2z)/3 >= 0 in double -- only the sign of the float sum matters (NaN: not culled).  A full-frame
    // filler has culled already (every triangle that got this far faces the camera); the full view-space normals are formed
    // only where the record is written, so that their nine registers are not live across the projection and the denominators.
    if (banded && valid) {
        const float *q = sn + mi * 9;
        float z0 = q[2], z1 = q[5], z2 = q[8];
        if (F.views) {
            z0 = (sM[6] * q[0] + sM[7] * q[1]) + sM[8] * q[2];
            z1 = (sM[6] * q[3] + sM[7] * q[4]) + sM[8] * q[5];
            z2 = (sM[6] * q[6] + sM[7] * q[7]) + sM[8] * q[8];
        }
        drawn = drawn && !(((z0 + z1) + z2) >= 0.0f);
    }
    const unsigned bx = drawn ? ((unsigned)xl | ((unsigned)xr << 16)) : 0u;
    const unsigned by = drawn ? ((unsigned)yt | ((unsigned)yb << 16)) : 0u;

    float l03 = 0.f, l13 = 0.f, l23 = 0.f;
    unsigned fl = 0;
    if (drawn) {
    // denominators of mu:12-21 -- pure functions of the triangle, hoisted out of the per-pixel code (same bits)
    l03 = (x[1] - x[2]) * (y[0] - y[2]) - (y[1] - y[2]) * (x[0] - x[2]);
    l13 = (x[2] - x[0]) * (y[1] - y[0]) - (y[2] - y[0]) * (x[1] - x[0]);
    l23 = (x[0] - x[1]) * (y[2] - y[1]) - (y[0] - y[1]) * (x[2] - x[1]);
    // Division-free rejection (SURVEY 7, K3 obligation).  num/l3 is bit-identical to (-num)/(-l3), and negation commutes
    // with every rounding that produced num, so the rasterizer evaluates each coordinate with l3' = |l3| (edge vector
    // negated when l3 < 0, FL_NEG).  For L3_MIN <= l3' <= L3_MAX a numerator <= -REJ_EPS then gives a quotient that is a
    // negative NON-ZERO float (|q| >= 1e-36), i.e. exactly the reference's `bar < 0` -- no division needed (FL_REJ).
    // Everything else (denominator zero / tiny / huge / non-finite, numerator inside the guard band or NaN) takes the
    // exact division path.
    const float a03 = fabsf(l03), a13 = fabsf(l13), a23 = fabsf(l23);
    if (a03 >= L3_MIN && a03 <= L3_MAX) fl |= (FL_REJ << 0) | (l03 < 0.f ? (FL_NEG << 0) : 0u);
    if (a13 >= L3_MIN && a13 <= L3_MAX) fl |= (FL_REJ << 1) | (l13 < 0.f ? (FL_NEG << 1) : 0u);
    if (a23 >= L3_MIN && a23 <= L3_MAX) fl |= (FL_REJ << 2) | (l23 < 0.f ? (FL_NEG << 2) : 0u);
    float cmax = 0.0f;
#pragma unroll
    for (int k = 0; k < 3; ++k) cmax = fmaxf(cmax, fmaxf(fabsf(x[k]), fabsf(y[k])));
    const bool finite_xy = (x[0] - x[0] == 0.f) && (x[1] - x[1] == 0.f) && (x[2] - x[2] == 0.f) && (y[0] - y[0] == 0.f) &&
                           (y[1] - y[1] == 0.f) && (y[2] - y[2] == 0.f);
    if ((fl & (7u * FL_REJ)) == 7u * FL_REJ && finite_xy && cmax <= SPAN_COORD_MAX) fl |= FL_SPAN;
    if (fminf(fminf(a03, a13), a23) >= FDIV_LO && fmaxf(fmaxf(a03, a13), a23) <= FDIV_HI) fl |= FL_FDIV;
    }

    // the chunk's entries for k_fill and the atomic path, densely at the head of its recE block: the triangles that survived
    // the cull (a full-frame filler; the rare ones whose rectangle is empty carry bx = 0) or exactly the drawn ones (a
    // band-sharded filler, where most triangles of a visited chunk still miss the band)
    unsigned n_entries, dpos;
    bool entry;
    if (banded) {
        dpos = block_compact(drawn, wsum, n_entries);
        entry = drawn;
    } else {
        dpos = threadIdx.x; entry = valid;
        n_entries = __syncthreads_or(drawn ? 1 : 0) ? kept : 0u;
    }
    if (entry && n_entries) F.recE[(long long)view * F.T + first + dpos] = make_float4(__uint_as_float(bx), __uint_as_float(by), __uint_as_float((unsigned)mi), __uint_as_float(fl));
    if (threadIdx.x == 0) *alive = (unsigned short)n_entries;
    // the vertex colours are only needed for triangles that are drawn: a CTA without any (culled, off screen, or -- for a
    // band-sharded filler -- outside the band, which is 7 of 8 CTAs at N=8) never reads them
    if (n_entries == 0) return;
    if (!staged) {
        stage_floats(F.c, first * 9, cnt * 9, sc);
        __syncthreads();
    }
    if (drawn) {
    float4 *R = F.shrec + ridx * SREC;
    const float *q = sc + mi * 9;
    R[S_A] = make_float4(x[0], y[0], x[1], y[1]);
    R[S_B] = make_float4(x[2], y[2], z[0], z[1]);
    R[S_C] = make_float4(z[2], l03, l13, l23);
    float nx[3], ny[3], nz[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        nx[k] = sn[mi * 9 + k * 3 + 0];
        ny[k] = sn[mi * 9 + k * 3 + 1];
        nz[k] = sn[mi * 9 + k * 3 + 2];
        if (F.views) view_normal(sM, nx[k], ny[k], nz[k]);
    }
    R[S_N0] = make_float4(nx[0], ny[0], nz[0], nx[1]);
    R[S_N1] = make_float4(ny[1], nz[1], nx[2], ny[2]);
    if (PERSP) {
        // CRB_TEX_PERSPECTIVE (DESIGN 2): per corner (u*w, v*w, w), w = 1 / z with z the camera-space depth project_vertex
        // divides by -- still in sv; for batched views view_point's z row gives the same bits again
        float t[9];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float *p = sv + mi * 9 + k * 3;
            const float zc = F.views ? ((sM[6] * (p[0] - sM[9]) + sM[7] * (p[1] - sM[10])) + sM[8] * (p[2] - sM[11])) + sM[14] : p[2];
            const float w = 1.0f / zc;
            t[3 * k] = q[3 * k] * w; t[3 * k + 1] = q[3 * k + 1] * w; t[3 * k + 2] = w;
        }
        R[S_X] = make_float4(nz[2], t[0], t[1], t[2]);
        R[S_C1] = make_float4(t[3], t[4], t[5], t[6]);
        R[S_C2] = make_float4(t[7], t[8], __uint_as_float(fl), 0.0f);
    } else {
        R[S_X] = make_float4(nz[2], q[0], q[1], q[2]);
        R[S_C1] = make_float4(q[3], q[4], q[5], q[6]);
        R[S_C2] = make_float4(q[7], q[8], __uint_as_float(fl), 0.0f);
    }
    }
    if (F.flags & CRB_PATH_ATOMIC) return;

    // per-tile counts.  A triangle that touches a few tiles (the usual case) is counted by its own thread; one that spans many
    // (a quad of the 2048^2 basketball covers hundreds) is counted by its whole warp, a tile per lane -- left to one thread, a
    // screen-filling triangle alone kept the kernel busy for a millisecond
    int tx0 = 0, tx1 = -1, ty0 = 0, ty1 = -1;
    if (drawn) tile_span(F, bx, by, tx0, tx1, ty0, ty1);
    unsigned *cnt_view = F.count + (long long)view * F.nTiles;
    const int nt = drawn ? (tx1 - tx0 + 1) * (ty1 - ty0 + 1) : 0;
    // (counted with one fire-and-forget atomicAdd per (triangle, tile): aggregating the lanes of a warp that hit the same tile --
    // what k_fill does for its slot-returning atomics -- costs more in MATCH than the reductions it saves: 86 -> 96 us)
    if (nt <= WIDE_TILES)
        for (int ty = ty0; ty <= ty1; ++ty)
            for (int tx = tx0; tx <= tx1; ++tx) atomicAdd(cnt_view + ty * F.tilesX + tx, 1u);
    for (unsigned wide = __ballot_sync(0xFFFFFFFFu, nt > WIDE_TILES); wide; wide &= wide - 1u) {
        const int src = __ffs(wide) - 1;
        const int sx0 = __shfl_sync(0xFFFFFFFFu, tx0, src), sx1 = __shfl_sync(0xFFFFFFFFu, tx1, src);
        const int sy0 = __shfl_sync(0xFFFFFFFFu, ty0, src), n = __shfl_sync(0xFFFFFFFFu, nt, src);
        const int wx = sx1 - sx0 + 1;
        for (int i = (int)(threadIdx.x & 31u); i < n; i += 32) atomicAdd(cnt_view + (sy0 + i / wx) * F.tilesX + sx0 + i % wx, 1u);
    }
}

#ifndef CRB_SETUP_MIN_CTAS
#define CRB_SETUP_MIN_CTAS 3
#endif
// Persistent: a few CTAs per SM walk the (view, chunk) work items -- all chunks of all views, or the chunks k_band_chunks listed
// for a band-sharded filler -- through a ring of SETUP_STAGES shared-memory stages.  One thread issues the three 9 216-byte bulk
// copies (cp.async.bulk, completion counted on the stage's mbarrier) of the item two turns ahead as soon as the CTA is done
// with a stage, so a chunk's vertices, normals and colours arrive while the previous chunk is being projected: the memory
// round trip that headed every one-chunk CTA's life (load -> barrier -> work) is off the critical path.
constexpr int SETUP_STAGES = 2;
constexpr size_t SETUP_STAGE_FLOATS = 3 * (size_t)NT * 9;
constexpr size_t SETUP_DYN_SMEM = SETUP_STAGES * SETUP_STAGE_FLOATS * sizeof(float);
template <bool PERSP>
__global__ void __launch_bounds__(NT, CRB_SETUP_MIN_CTAS) k_setup(const Frame F)
{
    extern __shared__ __align__(128) float stg[];          // [SETUP_STAGES][3][NT * 9]
    __shared__ __align__(8) unsigned long long bar[SETUP_STAGES];
    __shared__ float sM[16];
    __shared__ unsigned char slist[NT];
    __shared__ unsigned wsum[NT / 32];
    if (blockIdx.x == 0 && threadIdx.x == 0) {  // k_alloc (next launch) accumulates
        F.total[0] = 0ull; F.total[2] = 0ull; F.total[3] = 0ull; F.total[4] = 0ull; F.total[5] = 0ull;
    }
    const long long chunksPerView = (F.T + NT - 1) / NT;
    const long long nItems = F.chunks ? (long long)F.chunks[0] : chunksPerView * F.nViews;
    const bool banded = F.row0 > 0 || F.row1 < F.H;
    // bulk copies want 16-byte aligned sources (a chunk is 9 216 bytes, so only the array bases matter) and whole chunks; a
    // band-sharded filler without a chunk list tests the vertices before it reads anything else (setup_chunk) and stages itself
    const bool bulk_ok = !((reinterpret_cast<uintptr_t>(F.v) | reinterpret_cast<uintptr_t>(F.n) | reinterpret_cast<uintptr_t>(F.c)) & 15u) &&
                         (!banded || F.chunks);
    auto item = [&](long long w, int &view) -> long long {
        if (F.chunks) { view = 0; return (long long)F.chunks[1 + w]; }
        view = (int)(w / chunksPerView);
        return w % chunksPerView;
    };
    auto issue = [&](long long w, int s) {            // one thread: the three bulk copies of item w into stage s (if it qualifies)
        int view;
        const long long chunk = item(w, view);
        if (!bulk_ok || (chunk + 1) * NT > F.T) return;
        float *d = stg + (size_t)s * SETUP_STAGE_FLOATS;
        bulk_load(d, F.v + chunk * NT * 9, BC_BYTES, &bar[s]);
        bulk_load(d + NT * 9, F.n + chunk * NT * 9, BC_BYTES, &bar[s]);
        bulk_load(d + 2 * NT * 9, F.c + chunk * NT * 9, BC_BYTES, &bar[s]);
    };
    if (threadIdx.x == 0) {
        for (int s = 0; s < SETUP_STAGES; ++s) mbar_init(&bar[s], 3u);      // three copies, one arrival each
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (int s = 0; s < SETUP_STAGES; ++s)
            if ((long long)blockIdx.x + (long long)s * gridDim.x < nItems) issue((long long)blockIdx.x + (long long)s * gridDim.x, s);
    }
    __syncthreads();
    unsigned uses = 0;                                  // bit s: parity of the bulk-loaded items stage s has delivered so far
    int i = 0;
    for (long long w = blockIdx.x; w < nItems; w += gridDim.x, ++i) {
        const int s = i % SETUP_STAGES;
        int view;
        const long long chunk = item(w, view);
        const bool staged = bulk_ok && (chunk + 1) * NT <= F.T;
        if (staged) {
            mbar_wait(&bar[s], (uses >> s) & 1u);
            uses ^= 1u << s;
        }
        float *d = stg + (size_t)s * SETUP_STAGE_FLOATS;
        setup_chunk<PERSP>(F, view, chunk, chunksPerView, d, d + NT * 9, d + 2 * NT * 9, sM, slist, wsum, staged);
        __syncthreads();                                // everybody is done with the stage (and with sM / slist / wsum)
        const long long w2 = w + (long long)SETUP_STAGES * gridDim.x;
        if (threadIdx.x == 0 && w2 < nItems) issue(w2, s);
    }
}

// Band-sharded fillers (SURVEY 8e) see every triangle of the frame but draw only those that reach their rows.  This
// pre-pass lists the 256-triangle chunks with at least one triangle whose pixel rectangle meets the band (same projection and
// rectangle code as k_setup, before the cull), so that k_setup and k_fill visit only those.  A few CTAs per SM stream the
// vertex array through a ring of BC_STAGES shared-memory buffers filled by 1-D bulk copies (cp.async.bulk, one 9 216-byte
// copy per chunk issued by one thread, completion counted on an mbarrier), i.e. at memory speed rather than at the rate at
// which 39 075 load -> barrier -> project -> exit CTAs can be launched and retired.
__global__ void __launch_bounds__(NT) k_band_chunks(const Frame F)
{
    __shared__ __align__(128) float sv[BC_STAGES][NT * 9];
    __shared__ __align__(8) unsigned long long bar[BC_STAGES];
    const long long nFull = F.T / NT;                 // a ragged last chunk is listed unconditionally (by CTA 0, below)
    if (blockIdx.x == 0 && threadIdx.x == 0 && nFull * NT < F.T) F.chunks[1 + atomicAdd(F.chunks, 1u)] = (unsigned)nFull;
    // this CTA's chunks: blockIdx.x + j * gridDim.x, j < nMine
    const long long nMine = nFull > blockIdx.x ? (nFull - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    if (threadIdx.x == 0) {
        for (int s = 0; s < BC_STAGES; ++s) mbar_init(&bar[s], 1u);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (int j = 0; j < BC_STAGES && j < nMine; ++j)
            bulk_load(sv[j], F.v + (blockIdx.x + (long long)j * gridDim.x) * (NT * 9), BC_BYTES, &bar[j]);
    }
    __syncthreads();
    for (long long j = 0; j < nMine; ++j) {
        const int s = (int)(j % BC_STAGES);
        mbar_wait(&bar[s], (unsigned)((j / BC_STAGES) & 1));
        // Conservative row test: a chunk listed without need costs a k_setup visit, a chunk missed would cost pixels.  The
        // screen y of each vertex is formed like project_vertex forms it, except that the division is a multiplication by
        // rcp.approx (relative difference < 3e-7, i.e. < 0.01 pixel on screen); the band is widened by far more than that,
        // and anything non-finite or beyond 1e9 (where the reference's (int)ceil wraps to INT_MIN) lists the chunk.
        // The x extent is not tested here (k_setup does that exactly).
        float ylo = 3.0e38f, yhi = -3.0e38f;
        bool odd = false;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float vx = sv[s][threadIdx.x * 9 + k * 3 + 0];
            const float vy = sv[s][threadIdx.x * 9 + k * 3 + 1];
            const float vz = sv[s][threadIdx.x * 9 + k * 3 + 2];
            const float X = ((vx * F.proj.p[0] + vy * F.proj.p[4]) + vz * F.proj.p[8]) + F.proj.p[12];
            const float Y = ((X * F.proj.p[1] + vy * F.proj.p[5]) + vz * F.proj.p[9]) + F.proj.p[13];
            float r;
            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(vz));
            const float ysc = (Y * r + 1.0f) * F.proj.ys;
            if (!(fabsf(ysc) < 1.0e9f)) odd = true;
            ylo = fminf(ylo, ysc);
            yhi = fmaxf(yhi, ysc);
        }
        // rows drawn are the integers r with ymin <= r < ymax inside [row0, row1)
        const bool reach = odd || ((ylo - (0.25f + 1.0e-5f * fabsf(ylo)) <= (float)(F.row1 - 1)) &&
                                   (yhi + (0.25f + 1.0e-5f * fabsf(yhi)) > (float)F.row0));
        const int any = __syncthreads_or(reach);   // also: everybody is done with sv[s]
        if (threadIdx.x == 0) {
            const long long chunk = blockIdx.x + j * gridDim.x;
            if (j + BC_STAGES < nMine) bulk_load(sv[s], F.v + (chunk + (long long)BC_STAGES * gridDim.x) * (NT * 9), BC_BYTES, &bar[s]);
            if (any) F.chunks[1 + atomicAdd(F.chunks, 1u)] = (unsigned)chunk;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// K2b: list space for every tile.  Block-wide exclusive scan (warp shuffles) of the tile counts, one bump
// allocation per CTA.  List order in memory is irrelevant: the packed key makes the result order-independent.
// ------------------------------------------------------------------------------------------------------------
template <int NTH = NT>
__device__ __forceinline__ unsigned block_exclusive_scan(unsigned v, unsigned *warp_sums, unsigned &block_total)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    unsigned inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned t = __shfl_up_sync(0xFFFFFFFFu, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) warp_sums[wid] = inc;
    __syncthreads();
    unsigned base = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < NTH / 32; ++w) {
        const unsigned s = warp_sums[w];
        if (w < wid) base += s;
        tot += s;
    }
    block_total = tot;
    __syncthreads();
    return base + inc - v;
}

__global__ void __launch_bounds__(NT) k_alloc(const Frame F)
{
    __shared__ unsigned warp_sums[NT / 32];
    __shared__ unsigned long long block_base;
    __shared__ unsigned busy_base, empty_base;
    const long long i = (long long)blockIdx.x * NT + threadIdx.x;
    const long long nAll = (long long)F.nViews * F.nTiles;
    const unsigned c = (i < nAll) ? F.count[i] : 0u;
    unsigned tot, nbusy, nheavy;
    const unsigned excl = block_exclusive_scan(c, warp_sums, tot);
    const unsigned brank = block_exclusive_scan(c ? 1u : 0u, warp_sums, nbusy);
    // a frame of one view is as slow as its heaviest tile: such tiles are cut into row bands (disjoint pixels, no merge)
    const bool cut = F.splitHeavy && c > SPLIT_N, heavy = cut || c > HEAVY_N;
    const unsigned hrecs = cut ? (unsigned)SPLIT_BANDS : (heavy ? 1u : 0u);
    const unsigned hrank = block_exclusive_scan(hrecs, warp_sums, nheavy);
    unsigned nheavyTiles;
    const unsigned htile = block_exclusive_scan(heavy ? 1u : 0u, warp_sums, nheavyTiles);
    __shared__ unsigned heavy_base;
    if (threadIdx.x == 0) {
        const unsigned valid = (unsigned)min((long long)NT, nAll - (long long)blockIdx.x * NT);
        block_base = tot ? atomicAdd(F.total, (unsigned long long)tot) : 0ull;
        busy_base = (unsigned)atomicAdd(F.total + 2, (unsigned long long)(nbusy - nheavyTiles));
        heavy_base = (unsigned)atomicAdd(F.total + 4, (unsigned long long)nheavy);
        empty_base = (unsigned)atomicAdd(F.total + 3, (unsigned long long)(valid - nbusy));
    }
    __syncthreads();
    if (i < nAll) {
        const unsigned long long o = block_base + excl;
        const unsigned o32 = (unsigned)(o > 0xFFFFFFFFull ? 0xFFFFFFFFull : o);
        F.offset[i] = o32;
        F.cursor[i] = 0u;
        F.count[i] = 0u;   // self-cleaning: the next frame's k_setup starts from zero
        const unsigned vw = (unsigned)(i / F.nTiles), tl = (unsigned)(i % F.nTiles);
        const unsigned packed = (vw << 22) | ((tl / (unsigned)F.tilesX) << 11) | (tl % (unsigned)F.tilesX);   // view:10 ty:11 tx:11
        constexpr unsigned FULL = (unsigned)TH << 8;                    // .w = first row | end row << 8 of the CTA's share of the tile
        if (cut)
            for (unsigned b = 0; b < (unsigned)SPLIT_BANDS; ++b)
                F.busyH[heavy_base + hrank + b] = make_uint4(packed, c, o32, (b * (TH / SPLIT_BANDS)) | (((b + 1) * (TH / SPLIT_BANDS)) << 8));
        else if (heavy) F.busyH[heavy_base + hrank] = make_uint4(packed, c, o32, FULL);
        else if (c) F.busy[busy_base + (brank - htile)] = make_uint4(packed, c, o32, FULL);
        else F.empty[empty_base + (threadIdx.x - brank)] = packed;
    }
}

// K2c: scatter the prepared setups into the tile lists (sign-normalised form the row loop wants).
constexpr int FT = 64;            // threads per k_fill CTA: four CTAs share a chunk, and one whose entries are used up leaves at once
__device__ __forceinline__ void fill_chunk(const Frame &F, const int view, const long long chunk, const long long chunksPerView, const bool skip,
                                           const unsigned tix /* position in the chunk, 0..NT-1 */)
{
    // the chunk's drawn triangles sit densely at the head of its recE block (setup_chunk): thread j takes entry j, so the warps
    // that have work are full and the others leave at once.  Speculative: the entry flies with the count that decides whether
    // it is looked at (recE is allocated for every (view, triangle); entries beyond the count are stale and not used)
    const long long slot = chunk * NT + tix;
    const float4 E = slot < F.T ? F.recE[(long long)view * F.T + slot] : make_float4(0.f, 0.f, 0.f, 0.f);
    const unsigned nd = F.alive[(long long)view * chunksPerView + chunk];
    if (skip || (tix & ~31u) >= nd) return;   // frame skipped / no entry for this warp (warp-uniform)
    const unsigned bx = tix < nd ? __float_as_uint(E.x) : 0u, by = tix < nd ? __float_as_uint(E.y) : 0u;
    const bool drawn = (bx >> 16) != 0;  // (x_right >= 1 for every drawn triangle)
    const long long tri = chunk * NT + (drawn ? (long long)(__float_as_uint(E.z) & 255u) : 0ll);
    const long long ridx = (long long)view * F.T + tri;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a, s2 = a, s3 = a;
    int tx0 = 0, tx1 = -1, ty0 = 0, ty1 = -1;
    if (drawn) {
        const float4 *R = F.shrec + ridx * SREC;
        const float4 c = R[S_C];
        a = R[S_A]; b = R[S_B];
        const unsigned fl = __float_as_uint(E.w);
        // |l3| where the coordinate is negated (flipping the sign bit is exact)
        s2 = make_float4(c.x, (fl & (FL_NEG << 0)) ? -c.y : c.y, (fl & (FL_NEG << 1)) ? -c.z : c.z, (fl & (FL_NEG << 2)) ? -c.w : c.w);
        s3 = make_float4(__uint_as_float(bx), __uint_as_float(by), __uint_as_float((unsigned)tri), __uint_as_float(fl));
        tile_span(F, bx, by, tx0, tx1, ty0, ty1);
    }
    const long long vb = (long long)view * F.nTiles;
    const int nt = drawn ? (tx1 - tx0 + 1) * (ty1 - ty0 + 1) : 0;
    {   // lanes of the warp that append to the same tile in the same turn take their slots with ONE atomicAdd (mesh neighbours
        // fall into the same tile: a warp's 32 triangles usually touch two or three tiles)
        const unsigned lane = tix & 31u;
        const int small = nt <= WIDE_TILES ? nt : 0;
        const int turns = __reduce_max_sync(0xFFFFFFFFu, small);
        int cx = tx0, cy = ty0;
        for (int k = 0; k < turns; ++k) {
            const bool act = k < small;
            const long long t = vb + cy * F.tilesX + cx;
            const unsigned tag = act ? (unsigned)t : 0xFFFFFFE0u + lane;      // inactive lanes match nobody
            const unsigned grp = __match_any_sync(0xFFFFFFFFu, tag);
            const int leader = __ffs(grp) - 1;
            unsigned base = 0;
            if (act && (int)lane == leader) base = F.offset[t] + atomicAdd(F.cursor + t, (unsigned)__popc(grp));
            base = __shfl_sync(0xFFFFFFFFu, base, leader);
            if (act) {
                float4 *o = F.ls + (size_t)(base + __popc(grp & ((1u << lane) - 1u))) * 4;     // one 64-byte entry = two whole sectors
                o[0] = a; o[1] = b; o[2] = s2; o[3] = s3;
                if (++cx > tx1) { cx = tx0; ++cy; }
            }
        }
    }
    // Triangles that span many tiles (a quad of the 2048^2 basketball covers hundreds).  With a k_fill_wide launch behind this
    // kernel they are only listed here and scattered there, a warp per triangle: done in place, one after the other by the warp
    // that owns them, a chunk of 256 such triangles kept two warps busy for the length of the whole kernel (basketball: 76 us of
    // k_fill on 128 warps).  Without that launch (or with the list full): in place, a tile per lane (see setup_chunk).
    unsigned widem = __ballot_sync(0xFFFFFFFFu, nt > WIDE_TILES);
    if (F.wideCap && widem) {
        const unsigned lane = tix & 31u;
        unsigned long long first = 0ull;
        if ((int)lane == __ffs(widem) - 1) first = atomicAdd(F.total + 5, (unsigned long long)__popc(widem));
        first = __shfl_sync(0xFFFFFFFFu, first, __ffs(widem) - 1);
        const unsigned long long at = first + __popc(widem & ((1u << lane) - 1u));
        const bool listed = nt > WIDE_TILES && at < (unsigned long long)F.wideCap;
        if (listed) F.wide[at] = make_uint4((unsigned)view, (unsigned)tri, bx, by);
        widem = __ballot_sync(0xFFFFFFFFu, nt > WIDE_TILES && !listed);
    }
    for (unsigned wide = widem; wide; wide &= wide - 1u) {
        const int src = __ffs(wide) - 1;
        auto bc = [src](float4 v) {
            return make_float4(__shfl_sync(0xFFFFFFFFu, v.x, src), __shfl_sync(0xFFFFFFFFu, v.y, src), __shfl_sync(0xFFFFFFFFu, v.z, src),
                               __shfl_sync(0xFFFFFFFFu, v.w, src));
        };
        const float4 wa = bc(a), wb = bc(b), w2 = bc(s2), w3 = bc(s3);
        const int sx0 = __shfl_sync(0xFFFFFFFFu, tx0, src), sx1 = __shfl_sync(0xFFFFFFFFu, tx1, src);
        const int sy0 = __shfl_sync(0xFFFFFFFFu, ty0, src), n = __shfl_sync(0xFFFFFFFFu, nt, src);
        const int wx = sx1 - sx0 + 1;
        for (int i = (int)(tix & 31u); i < n; i += 32) {
            const long long t = vb + (sy0 + i / wx) * F.tilesX + sx0 + i % wx;
            const unsigned at = F.offset[t] + atomicAdd(F.cursor + t, 1u);
            float4 *o = F.ls + (size_t)at * 4;
            o[0] = wa; o[1] = wb; o[2] = w2; o[3] = w3;
        }
    }
}

#ifndef CRB_FILL_MIN_CTAS
#define CRB_FILL_MIN_CTAS 16
#endif
__global__ void __launch_bounds__(FT, CRB_FILL_MIN_CTAS) k_fill(const Frame F)
{
    const long long chunksPerView = (F.T + NT - 1) / NT;
    const unsigned tix = (blockIdx.x & (NT / FT - 1)) * FT + threadIdx.x;
    if (!F.chunks) {
        // overflow: frame is skipped (host is told via crb_status); the test rides with the first loads instead of before them
        fill_chunk(F, blockIdx.y, blockIdx.x / (NT / FT), chunksPerView, *F.total > (unsigned long long)F.pairCap, tix);   // same chunk -> triangles mapping as k_setup
        return;
    }
    if (*F.total > (unsigned long long)F.pairCap) return;
    const unsigned n = F.chunks[0];
    for (unsigned i = blockIdx.x / (NT / FT); i < n; i += gridDim.x / (NT / FT)) fill_chunk(F, 0, F.chunks[1 + i], chunksPerView, false, tix);
}

// The triangles k_fill listed as spanning many tiles: a CTA per triangle (a screen-filling one covers thousands of tiles), a tile
// per thread and turn, four turns' slot atomics in flight before the first entry is stored.
constexpr int FWT = 256;
__global__ void __launch_bounds__(FWT) k_fill_wide(const Frame F)
{
    if (*F.total > (unsigned long long)F.pairCap) return;
    const unsigned long long listed = F.total[5];
    const unsigned n = (unsigned)(listed < (unsigned long long)F.wideCap ? listed : (unsigned long long)F.wideCap);
    for (unsigned e = blockIdx.x; e < n; e += gridDim.x) {
        const uint4 w = F.wide[e];
        const long long ridx = (long long)w.x * F.T + w.y;
        const float4 *R = F.shrec + ridx * SREC;
        const float4 a = R[S_A], b = R[S_B], c = R[S_C];
        const unsigned fl = __float_as_uint(R[S_C2].z);
        const float4 s2 = make_float4(c.x, (fl & (FL_NEG << 0)) ? -c.y : c.y, (fl & (FL_NEG << 1)) ? -c.z : c.z, (fl & (FL_NEG << 2)) ? -c.w : c.w);
        const float4 s3 = make_float4(__uint_as_float(w.z), __uint_as_float(w.w), __uint_as_float(w.y), __uint_as_float(fl));
        int tx0, tx1, ty0, ty1;
        tile_span(F, w.z, w.w, tx0, tx1, ty0, ty1);
        const int wx = tx1 - tx0 + 1, nt = wx * (ty1 - ty0 + 1);
        const long long vb = (long long)w.x * F.nTiles;
        for (int i0 = (int)threadIdx.x; i0 < nt; i0 += 4 * FWT) {
            unsigned at[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int i = i0 + FWT * j;
                at[j] = 0u;
                if (i < nt) {
                    const long long t = vb + (ty0 + i / wx) * F.tilesX + tx0 + i % wx;
                    at[j] = F.offset[t] + atomicAdd(F.cursor + t, 1u);
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (i0 + FWT * j < nt) {
                    float4 *o = F.ls + (size_t)at[j] * 4;
                    o[0] = a; o[1] = b; o[2] = s2; o[3] = s3;
                }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// K3+K4: tile rasterizer + deferred shading
// ------------------------------------------------------------------------------------------------------------

// shared-memory 64-bit min.  There is no native 64-bit ATOMS.MIN.  The first attempt is a CAS against the empty key: with a
// depth complexity of ~1.25 most fragments find their pixel still empty and are done with one shared-memory transaction
// (instead of a load and a CAS: bunny 4096^2 -2.8 %, T-Rex unchanged); the others continue from the value it returned --
// losers leave at once, winners retry only when two lanes hit the same pixel in the same instant.
__device__ __forceinline__ void smem_key_min(unsigned long long *p, unsigned long long key)
{
    unsigned long long cur = atomicCAS(p, KEY_EMPTY, key);
    if (cur == KEY_EMPTY) return;
    while (key < cur) {
        const unsigned long long old = atomicCAS(p, cur, key);
        if (old == cur) break;
        cur = old;
    }
}

// Tensor maps (TMA) of the three output arrays of one launch, as 3-D tensors [view][row][x] (x in floats: W for z,
// 3W for colour / normals) with boxes of BOX_ROWS rows x one tile width.  Built on the host per launch (the output
// pointers are per call).  `use` bit k = map k is valid (CRB_BUF_* order); 0 = the launch uses plain stores only.
struct __align__(64) TMaps {
    CUtensorMap z, c, n;        // boxes of BOX_ROWS rows: the shaded rows of a busy tile
    CUtensorMap zt, ct, nt;     // boxes of a whole tile (TH rows): the fused clear
    unsigned use;
};

__device__ __forceinline__ void tma_store_box(const CUtensorMap *m, const void *smem, int cx, int cy, int cv)
{
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];"
                 :: "l"((unsigned long long)m), "r"(cx), "r"(cy), "r"(cv), "r"((unsigned)__cvta_generic_to_shared(smem))
                 : "memory");
}
__device__ __forceinline__ void tma_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (TMA) once a barrier has ordered them
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Optional phase timing (build with -DCRB_PHASE_TIMING): lane 0 of every warp accumulates the cycles it spends in each
// phase of k_raster into g_phase[]; read with crb_phase_cycles().  Compiled out of the product build.
__device__ unsigned long long g_phase[16];
#ifdef CRB_PHASE_TIMING
#define PH_DECL long long ph_t = clock64();
#define PH(k)                                                                      \
    do {                                                                           \
        if ((threadIdx.x & 31) == 0) {                                             \
            const long long now_ = clock64();                                      \
            atomicAdd(&g_phase[k], (unsigned long long)(now_ - ph_t));             \
            ph_t = now_;                                                           \
        }                                                                          \
    } while (0)
#else
#define PH_DECL
#define PH(k) do { } while (0)
#endif

// Shape of the tile rasterizer: threads per CTA, triangles staged per pass, fragment queue per warp, rows per clear box, resident CTAs
// per SM the launch bounds ask for, and whether shaded colour / normal rows are staged in shared memory (TMA boxes / vector stores)
// or stored straight from registers.  Three shapes are instantiated, see RasterLarge / RasterSmall / RasterWide below.
template <int RT_, int CH_, int FQ_, int CLEAR_ROWS_, int MIN_CTAS_, bool OUT_STAGE_>
struct RasterShape {
    static constexpr int RT = RT_, CH = CH_, FQ = FQ_, CLEAR_ROWS = CLEAR_ROWS_, MIN_CTAS = MIN_CTAS_;
    static constexpr bool OUT_STAGE = OUT_STAGE_;
    static_assert(CH_ <= RT_ && CH_ <= 256 && RT_ % 32 == 0 && RT_ <= NT, "one staged triangle per thread, 8-bit owner index");
    static_assert(FQ_ % 32 == 0 && FQ_ >= 64 && TH % CLEAR_ROWS_ == 0, "queue rounds of FQ/32 - 1 pixels per row; whole clear boxes per tile");
};

template <class C>
struct __align__(128) TileSmem {
    static constexpr int RT = C::RT, CH = C::CH, FQ = C::FQ, CLEAR_ROWS = C::CLEAR_ROWS;
    // TMA source first (128-byte aligned): shaded colour / normal rows of the tile
    union {
        struct {
            // per staged triangle (written by its staging thread, see raster_tile): the three edges in the sign-normalised form
            // the row loop wants, each with the vertex its numerator is measured from -- mu:24-26 with l3' = |l3|
            float4 e0[CH];  // l01' y2 l02' x2      bar1 numerator = l01'*(py - y2) - l02'*(px - x2)
            float4 e1[CH];  // l11' y0 l12' x0      bar2
            float4 e2[CH];  // l21' y1 l22' x1      bar3
            float4 tz[CH];  // z0 z1 z2 | triangle index
            float4 td[CH];  // d1 d2 d3 (denominators, > 0 where sane) | PK_* flags and the tile-relative pixel rectangle
            float4 tr[CH];  // 1/d1 1/d2 1/d3 (correctly rounded) | first row work item of the triangle
            unsigned char owner[CH * TH];  // row work item -> staged triangle
            float4 slot[RT / 32][2][32];   // per warp, per trip parity: the trip's 32 rows (A1 A2 A3 | staged triangle, tile row)
            unsigned short fq[RT / 32][FQ];  // per warp: queue of fragments (row lane | x << 5 | trip parity << 10)
        } st;
        struct {                              // (without row staging: only the 3 KB the staged uint8 image of a tile needs)
            float col[C::OUT_STAGE ? TH * TW * 3 : TH * TW * 3 / 4];
            float nrm[C::OUT_STAGE ? TH * TW * 3 : 4];
        } out;
        struct {                              // clear CTAs only: the constant pattern their TMA boxes are stored from
            float z[CLEAR_ROWS * TW];         //   Z_INIT
            float c[CLEAR_ROWS * TW * 3];     //   background colour = 0 (background_color) = the cleared normals: one pattern serves both
        } pat;
    } u;
    unsigned long long keys[TH * KEY_STRIDE];
    unsigned warp_sums[RT / 32];
};

// Writes one tile of cleared pixels (fresh-filler values) with plain stores -- the path for images whose rows are not
// 16-byte multiples, launches without tensor maps, and the uint8 image.
template <int NTH>
__device__ __forceinline__ void write_clear_tile(const Frame &F, unsigned skip, int view, int x0, int yl0, int tw, int th)
{
    const long long slab = (long long)view * F.slabPixels;
    const bool vec = (tw == TW) && ((F.W & 3) == 0);
    const float bg = background_color(F);
    const bool wz = F.z && !(skip & CRB_BUF_Z), wc = F.color && !(skip & CRB_BUF_COLOR), wn = F.normals && !(skip & CRB_BUF_NORMALS);
    if (vec) {
        // thread -> (row = tid/8 (+32 per pass), 16-byte column q = tid%8 (+8, +16)): shifts only, 128-byte runs
        const int q = threadIdx.x & 7;
        for (int r = threadIdx.x >> 3; r < th; r += NTH / 8) {
            const long long rowpix = slab + (long long)(yl0 + r) * F.W + x0;
            if (wz) reinterpret_cast<float4 *>(F.z + rowpix)[q] = make_float4(Z_INIT, Z_INIT, Z_INIT, Z_INIT);
            if (wc) {
                float4 *o = reinterpret_cast<float4 *>(F.color + rowpix * 3);
                o[q] = make_float4(bg, bg, bg, bg); o[q + 8] = make_float4(bg, bg, bg, bg); o[q + 16] = make_float4(bg, bg, bg, bg);
            }
            if (wn) {
                float4 *o = reinterpret_cast<float4 *>(F.normals + rowpix * 3);
                o[q] = make_float4(0.f, 0.f, 0.f, 0.f); o[q + 8] = make_float4(0.f, 0.f, 0.f, 0.f); o[q + 16] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
    } else {
        for (int i = threadIdx.x; i < th * tw; i += NTH) {
            const int r = i / tw, xx = i % tw;
            const long long p = slab + (long long)(yl0 + r) * F.W + x0 + xx;
            if (wz) F.z[p] = Z_INIT;
            if (wc) { F.color[p * 3] = bg; F.color[p * 3 + 1] = bg; F.color[p * 3 + 2] = bg; }
            if (wn) { F.normals[p * 3] = 0.f; F.normals[p * 3 + 1] = 0.f; F.normals[p * 3 + 2] = 0.f; }
        }
    }
    if (F.color_u8 && tw == TW && !(F.W & 15) && !(reinterpret_cast<uintptr_t>(F.color_u8) & 15u)) {
        // a tile row of the uint8 image is 96 bytes = six 16-byte stores (rows are 16-byte multiples: W % 16 == 0; the receive
        // buffers of a row exchange are 256-byte aligned)
        const unsigned w4 = (unsigned)to_u8(bg) * 0x01010101u;
        const uint4 val = make_uint4(w4, w4, w4, w4);
        for (int i = threadIdx.x; i < th * 6; i += NTH) {
            const int r = i / 6, q = i - r * 6;
            reinterpret_cast<uint4 *>(u8_pixel(F, view, yl0 + r, x0))[q] = val;
        }
    } else if (F.color_u8) {
        const unsigned char b8 = to_u8(bg);
        for (int i = threadIdx.x; i < th * tw * 3; i += NTH) {
            const int r = i / (tw * 3), xx = i % (tw * 3);
            u8_pixel(F, view, yl0 + r, x0)[xx] = b8;
        }
    }
}

// Conservative bound of the pixels of one row that can pass `bar_k >= 0`, for one barycentric.
// Reference (mu:34): num = fl(fl(l1*fl(py-a)) - fl(l2*fl(px-b))), inside <=> !(num/l3 < 0).  With the sign-normalised
// (l1', l2', d' > 0) form, inside => num' >= -REJ_EPS (k_fill).  num' differs from the real-valued
// E(x) = A - l2'*(x-b) by at most 3*2^-24*(|A| + |l2'|*|x-b|); M below is > 16x that bound plus the guard band, so
// E(x) < -M proves the reference rejects the pixel.  E is linear in x: the admissible x form a half line whose end is
// e = b + (A+M)/l2'.  The end is computed with an approximate reciprocal (relative error < 2^-22) and widened by wd, which
// exceeds every rounding of that evaluation for coordinates up to 2^18 (FL_SPAN); no walk towards the exact end follows --
// a pixel admitted without need (1.4 % of the survivors) is rejected by the exact pass like any other.  An edge that is
// (nearly) horizontal, |l2'| < 1e-20, bounds nothing here: rows on its far side lie outside the triangle's pixel rectangle.
// tools/scratch/span_test.c checks the bound against the per-pixel test on 16 M random rows.
__device__ __forceinline__ void span_bound(float A, float l2, float b, float xc, float &lo, float &hi)
{
    const float w = fabsf(xc - b) + 16.0f;                                          // >= |x - b| for every x of the tile
    const float M = __fmaf_rn(__fmaf_rn(fabsf(l2), w, fabsf(A)), 3.814697e-6f, 1e-5f);   // 2^-18 * magnitude + guard
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(l2));
    const float d = (A + M) * r;
    const float e = d + b;
    const float wd = __fmaf_rn(fabsf(d), 9.5367431640625e-7f, 0.0078125f);         // 2^-20 |e - b| + 2^-7
    if (fabsf(l2) >= 1e-20f) {
        if (l2 > 0.0f) hi = fminf(hi, e + wd);     // x <= e   (fminf / fmaxf ignore a NaN: no tightening)
        else lo = fmaxf(lo, e - wd);               // x >= e
    }
}

// bits of a staged triangle's packed word (td[].w)
constexpr unsigned PK_REJ = 1u;      // bits 0..2: barycentric k may use the division-free rejection
constexpr unsigned PK_SPAN = 8u;     // FL_SPAN
constexpr unsigned PK_FAST = 16u;    // FL_SPAN and FL_FDIV: div_rn_by() applies whenever the numerators are >= 2^-40
constexpr int PK_XA = 8, PK_XB = 14, PK_YT = 20;   // tile-relative rectangle: first x (6 bits), end x (6 bits), first row (5 bits)

// Visibility + deferred shading of one busy tile (n triangles staged at list offset off).
template <class C, int TEX>
__device__ __forceinline__ void raster_tile(const Frame &F, const TMaps &M, TileSmem<C> &S_, const bool clear, const int view,
                                            const int tx, const int ty, const unsigned n, const unsigned off, const int rowLo, const int rowHi)
{
    constexpr int RT = C::RT, CH = C::CH, FQ = C::FQ;      // (shadow the defaults of the same names)
    constexpr bool OUT_STAGE = C::OUT_STAGE;
    typedef TileSmem<C> TS;
#ifndef CRB_NO_OPAQUE_SMEM
    // The address of the CTA's shared memory goes through an empty asm: under the 40-register cap the compiler otherwise re-derives
    // the shared-window base (S2R SR_CgaCtaId + LEA) inside the exact and the shading loops instead of keeping it; an opaque
    // value cannot be rematerialised, and __isShared keeps the accesses LDS / STS / ATOMS.
    TS *Sp = &S_;
    asm volatile("" : "+l"(Sp));
    __builtin_assume(__isShared(Sp));
    TS &S = *Sp;
#else
    TS &S = S_;
#endif
    const int x0 = tx * TW, yl0 = ty * TH;       // yl0: row inside the band's buffers
    const int y0 = F.row0 + yl0;                  // absolute image row
    const int tw = min(TW, F.W - x0), th = min(min(TH, F.row1 - y0), rowHi);   // this CTA's rows of the tile: [rowLo, th)
    // the thread index is read once, through an asm the compiler cannot re-issue: under the 40-register cap it otherwise
    // re-reads the special register (S2R + the lane / warp arithmetic) inside every loop -- 6 % of the kernel's instructions
    unsigned tid;
    asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tid));
    const unsigned lane = tid & 31u, wid = tid >> 5;
    PH_DECL
    for (int i = tid; i < TH * KEY_STRIDE / 2; i += RT) reinterpret_cast<ulonglong2 *>(S.keys)[i] = make_ulonglong2(KEY_EMPTY, KEY_EMPTY);

    // ---- visibility: every (triangle,row) of the tile is one work item -------------------------------------
    for (unsigned base = 0; base < n; base += CH) {
        const unsigned m = min((unsigned)CH, n - base);
        __syncthreads();  // keys initialised / previous pass finished with the staging area
        PH(2);
        unsigned rows = 0;
        float4 tr3 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (tid < m) {   // the setups k_fill prepared for this tile, brought into the form the row loop wants
            const unsigned at = off + base + tid;
            const float4 *en = F.ls + (size_t)at * 4;
            const float4 a = en[0], b = en[1], c = en[2], d4 = en[3];
            const uint4 d = make_uint4(__float_as_uint(d4.x), __float_as_uint(d4.y), __float_as_uint(d4.z), __float_as_uint(d4.w));
            // correctly rounded reciprocals of the (sign-normalised) denominators, for div_rn_by: RN(1/-x) = -RN(1/x), so these are
            // the bits k_setup's rcp.rn of the signed denominators would give after the same sign flip
            tr3 = make_float4(__frcp_rn(c.y), __frcp_rn(c.z), __frcp_rn(c.w), 0.0f);
#ifndef CRB_NO_REC_PREFETCH
            if (CH < 64) {   // the shading pass will want this triangle's 128-byte record: start pulling it into L1 now (T-Rex x128
                             // -2.6 %; tiles of ~150 triangles evict them again before they are shaded: the large shape goes without)
                const char *sr = reinterpret_cast<const char *>(F.shrec + ((long long)view * F.T + d.z) * SREC);
                asm volatile("prefetch.global.L1 [%0];" :: "l"(sr));
                asm volatile("prefetch.global.L1 [%0];" :: "l"(sr + 32));
                asm volatile("prefetch.global.L1 [%0];" :: "l"(sr + 64));
                asm volatile("prefetch.global.L1 [%0];" :: "l"(sr + 96));
            }
#endif
            // edge vectors, sign-normalised (exact negation: flip the sign bit)
            const unsigned s1 = (d.w & 1u) << 31, s2 = (d.w & 2u) << 30, s3 = (d.w & 4u) << 29;
            S.u.st.e0[tid] = make_float4(__uint_as_float(__float_as_uint(a.z - b.x) ^ s1), b.y,
                                                 __uint_as_float(__float_as_uint(a.w - b.y) ^ s1), b.x);
            S.u.st.e1[tid] = make_float4(__uint_as_float(__float_as_uint(b.x - a.x) ^ s2), a.y,
                                                 __uint_as_float(__float_as_uint(b.y - a.y) ^ s2), a.x);
            S.u.st.e2[tid] = make_float4(__uint_as_float(__float_as_uint(a.x - a.z) ^ s3), a.w,
                                                 __uint_as_float(__float_as_uint(a.y - a.w) ^ s3), a.z);
            S.u.st.tz[tid] = make_float4(b.z, b.w, c.x, __uint_as_float(d.z));
            const int yt = max((int)(d.y & 0xFFFF), y0 + rowLo), yb = min((int)(d.y >> 16), y0 + th);
            rows = (unsigned)max(yb - yt, 0);
            const int xa = max((int)(d.x & 0xFFFF), x0) - x0, xb = min((int)(d.x >> 16), x0 + tw) - x0;   // 0 <= xa < xb <= 32
            const unsigned pk = ((d.w >> 4) & 7u) | ((d.w & FL_SPAN) ? PK_SPAN : 0u) |
                                ((d.w & (FL_SPAN | FL_FDIV)) == (FL_SPAN | FL_FDIV) ? PK_FAST : 0u) |
                                ((unsigned)xa << PK_XA) | ((unsigned)max(xb, xa) << PK_XB) | ((unsigned)((yt - y0) & 31) << PK_YT);
            S.u.st.td[tid] = make_float4(c.y, c.z, c.w, __uint_as_float(pk));
        }
        if (base + CH < n) {     // the next pass's list entries (64 B each, contiguous): start pulling their lines in now (T-Rex x128: -1.3 %)
            const unsigned nm = min((unsigned)CH, n - base - CH);
            for (unsigned i = tid; i < (nm + 1u) / 2u; i += RT)
                asm volatile("prefetch.global.L1 [%0];" :: "l"(F.ls + (size_t)(off + base + CH + 2u * i) * 4));
        }
        unsigned totalRows;
        const unsigned start = block_exclusive_scan<RT>(rows, S.warp_sums, totalRows);
        if (tid < m) {
            S.u.st.tr[tid] = make_float4(tr3.x, tr3.y, tr3.z, __uint_as_float(start));
            for (unsigned j = 0; j < rows; ++j) S.u.st.owner[start + j] = (unsigned char)tid;
        }
        PH(3);
        __syncthreads();
        PH(4);

        // Row work items, 32 per warp per trip.  Trip counts are warp-uniform and the body is predicated, so the warp
        // stays converged (a per-thread `for (r = tid; ...)` with early `continue`s lets lanes drift apart under
        // independent thread scheduling: measured 7.5 active lanes per instruction).
        if (DBG(F, FLAG_DBG_NOROWS)) totalRows = 0;
        // Tiles of a few large triangles (on average 16+ rows of the tile each: long spans, a full queue round per row)
        // have too few rows to occupy eight warps 32 at a time: there a trip of fewer than NT rows is dealt out in equal
        // shares (bunny 4096^2: k_raster 343 -> 304 us).  Tiles of many small triangles keep whole warps: the span pass
        // costs a warp the same with 8 active lanes as with 32, and those tiles are bound by issue slots, not latency.
#ifndef CRB_DEAL_ROWS
#define CRB_DEAL_ROWS 16
#endif
        const bool deal = totalRows >= (unsigned)CRB_DEAL_ROWS * m;
        // Exact pass.  The surviving pixels of a trip's 32 rows are intervals (first x, count).  In rounds of at most FQ/32 - 1
        // pixels per row, the rows append one entry per fragment (row lane | x << 5 | trip parity << 10) to the warp's queue at
        // the positions an exclusive scan of the counts assigns, and the queue is evaluated 32 entries at a time -- whole
        // batches only: what is left (< 32 entries) moves to the front and heads the first batch of the warp's next trip,
        // whose rows go into the slot array of the other parity, so that all 32 lanes evaluate a fragment in every step but
        // the warp's last.  qn: entries in the queue (warp-uniform).
        unsigned qn = 0, trip = 0;
        bool finished = false;
        unsigned short *fq = S.u.st.fq[wid];
        float4 *slotw = &S.u.st.slot[wid][0][0];        // this warp's two slot arrays (trip parity 0 / 1)
        for (unsigned tb = 0; !finished; tb += RT) {
            const unsigned rem = tb < totalRows ? totalRows - tb : 0u;
            const unsigned share = (rem >= (unsigned)RT || !deal) ? 32u : (rem + RT / 32 - 1u) / (RT / 32);
            if (wid * share >= rem) {                        // no rows left for this warp (warp-uniform) ...
                if (qn == 0u) break;
                finished = true;                             // ... but fragments of its last trip: one more turn evaluates them
            }
            const unsigned r = tb + wid * share + lane;
            const bool active = !finished && lane < share && r < totalRows;
            const unsigned par = trip & 1u;
            ++trip;
            int xa = 0, cnt = 0;              // the row's candidate pixels: tile-relative [xa, xa + cnt)
            if (active) {
                const unsigned o = S.u.st.owner[r];
                const float4 E0 = S.u.st.e0[o], E1 = S.u.st.e1[o], E2 = S.u.st.e2[o];
                const unsigned pk = __float_as_uint(S.u.st.td[o].w);
                const unsigned yl = ((pk >> PK_YT) & 31u) + (r - __float_as_uint(S.u.st.tr[o].w));   // row inside the tile
                const float py = (float)(y0 + (int)yl);
                const float A1 = E0.x * (py - E0.y), A2 = E1.x * (py - E1.y), A3 = E2.x * (py - E2.y);
                xa = (int)((pk >> PK_XA) & 63u);
                int xb = (int)((pk >> PK_XB) & 63u);
                slotw[par * 32u + lane] = make_float4(A1, A2, A3, __uint_as_float(o | (yl << 8)));
                // pass 1: which pixels of the row need the exact path.  A pixel is certainly outside (bar_k < 0) when a
                // numerator is below its threshold; each numerator is a monotone function of x (every rounding in
                // A - l2*(px - b) is monotone), so the pixels that survive all three tests form ONE interval.
                if (pk & PK_SPAN) {
                    // analytic, conservative interval (span_bound)
                    float lo = (float)(x0 + xa), hi = (float)(x0 + xb - 1);
                    const float xc = (float)(x0 + TW / 2);
                    span_bound(A1, E0.z, E0.w, xc, lo, hi);
                    span_bound(A2, E1.z, E1.w, xc, lo, hi);
                    span_bound(A3, E2.z, E2.w, xc, lo, hi);
                    if (lo <= hi) {
                        xa = max(xa, (int)ceilf(lo) - x0);       // lo, hi lie within [x0 + xa - 1, x0 + xb]: the conversions are exact
                        xb = min(xb, (int)floorf(hi) + 1 - x0);
                    } else {
                        xb = xa;
                    }
                } else {
                    // triangles without the analytic bound (huge / non-finite coordinates or denominators): every pixel of
                    // the rectangle row is tested against the thresholds; the hull of the survivors is the interval
                    const float thr1 = (pk & (PK_REJ << 0)) ? -REJ_EPS : -INFINITY;
                    const float thr2 = (pk & (PK_REJ << 1)) ? -REJ_EPS : -INFINITY;
                    const float thr3 = (pk & (PK_REJ << 2)) ? -REJ_EPS : -INFINITY;
                    unsigned mask = 0;
#pragma unroll 1
                    for (int x = xa; x < xb; ++x) {
                        const float px = (float)(x0 + x);
                        const float n1 = A1 - E0.z * (px - E0.w);
                        const float n2 = A2 - E1.z * (px - E1.w);
                        const float n3 = A3 - E2.z * (px - E2.w);
                        if (!(n1 < thr1 || n2 < thr2 || n3 < thr3)) mask |= 1u << x;        // else: certainly bar < 0
                    }
                    xa = mask ? __ffs(mask) - 1 : 0;
                    xb = mask ? 32 - __clz(mask) : 0;
                }
                cnt = max(xb - xa, 0);
            }
            __syncwarp();                     // the slots are published
            const unsigned old = qn;          // entries of the previous trip still waiting (they sit at the front)
            unsigned done = 0;
            unsigned entry = lane | ((unsigned)xa << 5) | (par << 10);
            for (;;) {
                const bool more = __any_sync(0xFFFFFFFFu, cnt > 0);
                if (more) {
                    const int c = min(cnt, FQ / 32 - 1);
                    int inc = c;
#pragma unroll
                    for (int dd = 1; dd < 32; dd <<= 1) {
                        const int t = __shfl_up_sync(0xFFFFFFFFu, inc, dd);
                        if ((int)lane >= dd) inc += t;
                    }
                    unsigned short *at = fq + qn + (unsigned)(inc - c);
#pragma unroll
                    for (int j = 0; j < FQ / 32 - 1; ++j)
                        if (j < c) at[j] = (unsigned short)(entry + ((unsigned)j << 5));
                    entry += (unsigned)c << 5;
                    cnt -= c;
                    qn += (unsigned)__shfl_sync(0xFFFFFFFFu, inc, 31);
                    __syncwarp();
                }
                const bool flush = !more && (finished || done < old);     // the slots of the trip before last are about to be reused
                unsigned b = 0;
                for (; b + 32u <= qn || (flush && b < qn); b += 32u) {
                    if (b + lane < qn) {
                        const unsigned e = fq[b + lane];
                        const unsigned src = e & 31u, bit = (e >> 5) & 31u;
                        const float4 q = slotw[(e >> 10) * 32u + src];
                        const unsigned info = __float_as_uint(q.w), o2 = info & 255u;
                        const float2 h0 = *reinterpret_cast<const float2 *>(&S.u.st.e0[o2].z);
                        const float2 h1 = *reinterpret_cast<const float2 *>(&S.u.st.e1[o2].z);
                        const float2 h2 = *reinterpret_cast<const float2 *>(&S.u.st.e2[o2].z);
                        const float4 Z = S.u.st.tz[o2], D = S.u.st.td[o2], R = S.u.st.tr[o2];
                        const float px = (float)(x0 + (int)bit);
                        const float n1 = q.x - h0.x * (px - h0.y);
                        const float n2 = q.y - h1.x * (px - h1.y);
                        const float n3 = q.z - h2.x * (px - h2.y);
                        float b1, b2, b3;
                        // PK_FAST triangles have |numerator| < 2^40 by construction (coordinates <= 2^18): only the lower bound is tested
                        if ((__float_as_uint(D.w) & PK_FAST) && fdiv_ok_lo(n1, n2, n3)) {
                            b1 = div_rn_by(n1, D.x, R.x); b2 = div_rn_by(n2, D.y, R.y); b3 = div_rn_by(n3, D.z, R.z);
                        } else {
                            b1 = n1 / D.x; b2 = n2 / D.y; b3 = n3 / D.z;
                        }
                        if (!(b1 < 0.0f || b2 < 0.0f || b3 < 0.0f)) {                 // pyx:216
                            const float z = (Z.x * b1 + Z.y * b2) + Z.z * b3;             // pyx:219
                            if (z == z)                                                   // pyx:220 rejects NaN only
                                smem_key_min(S.keys + ((info >> 8) & 31u) * KEY_STRIDE + bit, pack_key(z, __float_as_uint(Z.w)));
                        }
                    }
                }
                if (b) {                      // what is left moves to the front
                    const unsigned left = qn > b ? qn - b : 0u;
                    unsigned short tmp = 0;
                    if (lane < left) tmp = fq[b + lane];
                    __syncwarp();
                    if (lane < left) fq[lane] = tmp;
                    done += min(b, qn);
                    qn = left;
                    __syncwarp();
                }
                if (!more) break;
            }
        }
        PH(5);
    }
    __syncthreads();
    PH(6);

    // ---- deferred shading of the winners, staged so that colour / normals leave as whole rows ---------------
    const long long slab = (long long)view * F.slabPixels;
    const bool tma = OUT_STAGE && clear && M.use != 0u && (F.flags & FLAG_OUT_TMA);     // colour / normal rows leave through TMA boxes
    const bool vec = OUT_STAGE && clear && !tma && (tw == TW) && ((F.W & 3) == 0) && !(F.flags & FLAG_OUT_DIRECT) &&
                     (F.color || F.normals);                                                            // ... or as 16-byte vector stores
    const bool stage = tma || vec;
    // The uint8 image of a fresh frame whose float32 rows need no staging (image-only frames: HostImagePipeline, the row exchange,
    // PeerImage) is staged instead: the shading loop writes its three bytes per pixel into shared memory and the tile's rows leave
    // as 16-byte vector stores, six per 96-byte row = three whole sectors -- what a row exchange sends over NVLink is sectors, and
    // three byte stores per pixel touch each of them partially (N = 8: 0.77 of the rendering rate delivered).
    const bool u8stage = !stage && clear && F.color_u8 && tw == TW && !(F.W & 15) && (!F.u8xN || F.u8xRows % TH == 0);
    const float bg = background_color(F);
    const long long tilebase = slab + (long long)yl0 * F.W + x0;          // first pixel of the tile in its slab
    const unsigned rowStep = (unsigned)(RT / TW) * (unsigned)F.W;
    long long pix = tilebase + (unsigned)((int)wid * F.W + (int)lane);    // this thread's pixels: column lane, rows wid, wid + 8, ...
    const float4 *recv = F.shrec + (long long)view * F.T * SREC;          // the view's shade records
    for (int p = tid; p < TH * TW; p += RT, pix += rowStep) {
        const int yy = p / TW, xx = (int)lane;
        if (yy < rowLo || yy >= th || xx >= tw) continue;
        const unsigned long long key = S.keys[yy * KEY_STRIDE + xx];
        float z = Z_INIT, c[3] = {bg, bg, bg}, nn[3] = {0.f, 0.f, 0.f};
        bool write = clear;
        if (key != KEY_EMPTY && !DBG(F, FLAG_DBG_NOSHADE)) {
            const unsigned tri = ~(unsigned)(key & 0xFFFFFFFFull);
            float fz, fc[3], fn[3];
            if (shade_fragment<TEX>(F, recv + (size_t)(DBG(F, FLAG_DBG_ONEREC) ? 0u : tri) * SREC, (float)(x0 + xx), (float)(y0 + yy), fz, fc, fn)) {
                const float zold = clear ? Z_INIT : F.z[pix];
                if (!(fz > zold)) {  // pyx:223: drawn unless new_z > z_buffer (equal depth overwrites)
                    z = fz; c[0] = fc[0]; c[1] = fc[1]; c[2] = fc[2]; nn[0] = fn[0]; nn[1] = fn[1]; nn[2] = fn[2];
                    write = true;
                }
            }
        }
        if (OUT_STAGE && stage) {
            S.u.out.col[p * 3] = c[0]; S.u.out.col[p * 3 + 1] = c[1]; S.u.out.col[p * 3 + 2] = c[2];
            S.u.out.nrm[p * 3] = nn[0]; S.u.out.nrm[p * 3 + 1] = nn[1]; S.u.out.nrm[p * 3 + 2] = nn[2];
            if (F.z && !DBG(F, FLAG_DBG_NOOUT)) F.z[pix] = z;
        } else if (write) {
            if (F.z) F.z[pix] = z;
            if (F.color) { F.color[pix * 3] = c[0]; F.color[pix * 3 + 1] = c[1]; F.color[pix * 3 + 2] = c[2]; }
            if (F.normals) { F.normals[pix * 3] = nn[0]; F.normals[pix * 3 + 1] = nn[1]; F.normals[pix * 3 + 2] = nn[2]; }
        }
        if (F.color_u8 && write) {       // (one test on the float32-only path, as before the staging)
            unsigned char *o = u8stage ? reinterpret_cast<unsigned char *>(S.u.out.col) + p * 3 : u8_pixel(F, view, yl0 + yy, x0 + xx);
            o[0] = to_u8(c[0]); o[1] = to_u8(c[1]); o[2] = to_u8(c[2]);
        }
    }
    PH(7);
    if (u8stage) {
        __syncthreads();
        const unsigned char *sb = reinterpret_cast<const unsigned char *>(S.u.out.col);
        for (int i = tid; i < (th - rowLo) * 6; i += RT) {
            const int r = rowLo + i / 6, q = i - (i / 6) * 6;
            reinterpret_cast<uint4 *>(u8_pixel(F, view, yl0 + r, x0))[q] = reinterpret_cast<const uint4 *>(sb + r * (TW * 3))[q];
        }
    }
    if (DBG(F, FLAG_DBG_NOOUT)) return;
    if (OUT_STAGE && tma) {
        fence_async_smem();
        __syncthreads();
        PH(8);
        if (lane == 0) {   // box job j: array j/4 (colour, normals), row block j%4; one job per warp with eight warps
            for (unsigned job = wid; job < 8u; job += RT / 32) {
                const int r = (int)(job & 3u) * BOX_ROWS;
                if (r >= rowLo && r < th) {       // row bands are multiples of BOX_ROWS
                    if (job < 4u) { if (M.use & CRB_BUF_COLOR) tma_store_box(&M.c, S.u.out.col + r * TW * 3, x0 * 3, yl0 + r, view); }
                    else if (M.use & CRB_BUF_NORMALS) tma_store_box(&M.n, S.u.out.nrm + r * TW * 3, x0 * 3, yl0 + r, view);
                }
            }
            tma_commit();
        }
    } else if (OUT_STAGE && vec) {
        __syncthreads();
        const int q = tid & 7;
        for (int r = rowLo + (tid >> 3); r < th; r += RT / 8) {
            const long long o = (slab + (long long)(yl0 + r) * F.W + x0) * 3;
            if (F.color) {
                float4 *g = reinterpret_cast<float4 *>(F.color + o);
                const float4 *sc = reinterpret_cast<const float4 *>(S.u.out.col + r * TW * 3);
                g[q] = sc[q]; g[q + 8] = sc[q + 8]; g[q + 16] = sc[q + 16];
            }
            if (F.normals) {
                float4 *g = reinterpret_cast<float4 *>(F.normals + o);
                const float4 *sn = reinterpret_cast<const float4 *>(S.u.out.nrm + r * TW * 3);
                g[q] = sn[q]; g[q + 8] = sn[q + 8]; g[q + 16] = sn[q + 16];
            }
        }
    }
    PH(9);
}

// The fused clear through TMA: one tile = three whole-tile boxes (z, colour, normals) stored from the constant pattern in
// shared memory; the hardware clips boxes at the image edge.  Called by one lane.
template <class C>
__device__ __forceinline__ void tma_clear_tile(const TMaps &M, const TileSmem<C> &S, unsigned t)
{
    constexpr int CLEAR_ROWS = C::CLEAR_ROWS;
    const int view = (int)(t >> 22), yl0 = (int)((t >> 11) & 2047u) * TH, x0 = (int)(t & 2047u) * TW;
#pragma unroll
    for (int r = 0; r < TH; r += CLEAR_ROWS) {
        if (M.use & CRB_BUF_Z) tma_store_box(&M.zt, S.u.pat.z, x0, yl0 + r, view);
        if (M.use & CRB_BUF_COLOR) tma_store_box(&M.ct, S.u.pat.c, x0 * 3, yl0 + r, view);
        if (M.use & CRB_BUF_NORMALS) tma_store_box(&M.nt, S.u.pat.c, x0 * 3, yl0 + r, view);
    }
}

// Grid roles.  Busy tiles: one CTA each when the grid is large enough (it is sized from the busy-tile count the host
// last saw, see run_tiled), a strided walk otherwise.  The frame's clear is fused: with tensor maps every fourth CTA
// (blockIdx % 4 == 3) is a "clear CTA" that only issues the TMA boxes of the tiles without triangles (70 % of a T-Rex
// frame) -- a few thousand cycles of queueing, no arithmetic -- so those stores drain beside the rasterizing CTAs that
// share its SM for the whole length of the kernel.  Launches without tensor maps clear with plain stores up front,
// every CTA adopting its share of the empty tiles.
// Resident CTAs per SM follow the shape (RasterSmall 12 at 40 registers, RasterLarge 8 at 62, RasterWide 6 at 40); the
// static_assert in k_raster ties each shape's shared memory to the residency its launch bounds ask for.
#ifndef CRB_RASTER_MIN_CTAS
#define CRB_RASTER_MIN_CTAS 8
#endif
template <class C, int TEX>
__global__ void __launch_bounds__(C::RT, C::MIN_CTAS) k_raster(const Frame F, const __grid_constant__ TMaps M)
{
    constexpr int RT = C::RT, CLEAR_ROWS = C::CLEAR_ROWS;
    static_assert(sizeof(TileSmem<C>) + 1024 <= 233472 / C::MIN_CTAS, "k_raster: shared memory per CTA exceeds the residency its launch bounds assume");
    __shared__ TileSmem<C> S;
    PH_DECL
    const bool clear = (F.flags & CRB_CLEAR_FIRST) != 0;
    const bool split = clear && M.use != 0u;
    const unsigned nAll = (unsigned)F.nTiles * (unsigned)F.nViews;
    unsigned bidx = blockIdx.x, Gb = gridDim.x;
    if (split) {
        const unsigned Gc = gridDim.x / CE, ci = blockIdx.x / CE;
        Gb = gridDim.x - Gc;
        if ((blockIdx.x & (CE - 1u)) == CE - 1u) {
            // ---- clear CTA: warp w issues the tiles e = ci + (w + k * warps) * Gc
            const unsigned stride = Gc * (RT / 32);
            unsigned e = ci + (threadIdx.x >> 5) * Gc;
            unsigned t = e < nAll ? F.empty[e] : 0u;              // speculative: flies with the totals
            const unsigned long long pairs = F.total[0];
            const unsigned ne = (unsigned)F.total[3];
            if (pairs > (unsigned long long)F.pairCap || DBG(F, FLAG_DBG_NOCLEAR)) return;     // frame skipped: buffers stay untouched
            const float bg = background_color(F);
            for (int i = threadIdx.x; i < CLEAR_ROWS * TW * 3 / 4; i += RT) {
                reinterpret_cast<float4 *>(S.u.pat.c)[i] = make_float4(bg, bg, bg, bg);       // (bg is 0.0f: also the normals' pattern)
                if (i < CLEAR_ROWS * TW / 4) reinterpret_cast<float4 *>(S.u.pat.z)[i] = make_float4(Z_INIT, Z_INIT, Z_INIT, Z_INIT);
            }
            fence_async_smem();
            __syncthreads();
            if ((threadIdx.x & 31) == 0) {
                while (e < ne) {
                    const unsigned en = e + stride;
                    const unsigned tn = en < ne ? F.empty[en] : 0u;
                    tma_clear_tile(M, S, t);
                    e = en; t = tn;
                }
                tma_commit();
                tma_wait_read();
            }
            return;
        }
        bidx = ci * (CE - 1u) + (blockIdx.x & (CE - 1u));
    }
    // the first gridHeavy roles take the tiles with many triangles, in blockIdx (= dispatch) order before everything else
    const unsigned GH = F.gridHeavy;
    const bool heavyRole = bidx < GH;
    const uint4 *lst = heavyRole ? F.busyH : F.busy;
    const unsigned first = heavyRole ? bidx : bidx - GH, stride = heavyRole ? GH : Gb - GH;
    const unsigned cap = heavyRole ? nAll * (unsigned)SPLIT_BANDS : nAll;      // entries the list has room for
    uint4 rec = first < cap ? lst[first] : make_uint4(0u, 0u, 0u, 0u);     // speculative: flies with the totals
    const unsigned long long pairs = F.total[0];
    const unsigned nLight = (unsigned)F.total[2], nHeavy = (unsigned)F.total[4];
    const unsigned nb = heavyRole ? nHeavy : nLight;
    if (pairs > (unsigned long long)F.pairCap) {   // frame skipped; the host is told via crb_status
        if (bidx == 0 && threadIdx.x == 0) atomicMax(F.total + 1, pairs);
        return;
    }
    if (bidx == 0 && threadIdx.x == 0 && F.hstats) {
        volatile unsigned long long *hs = reinterpret_cast<volatile unsigned long long *>(F.hstats);
        hs[0] = ((unsigned long long)nAll << 32) | nLight;
        hs[1] = (unsigned long long)nHeavy | ((F.total[5] > 0xFFFFFFFFull ? 0xFFFFFFFFull : F.total[5]) << 32);     // + triangles that span many tiles
        hs[2] = pairs;                                                                                                  // (triangle, tile) pairs: the next launch's shape
    }
    if (clear && !split && !DBG(F, FLAG_DBG_NOCLEAR)) {
        const unsigned ne = (unsigned)F.total[3];
        for (unsigned e = bidx; e < ne; e += Gb) {
            const unsigned t = F.empty[e];
            const int view = (int)(t >> 22), ty = (int)((t >> 11) & 2047u), tx = (int)(t & 2047u);
            write_clear_tile<RT>(F, 0u, view, tx * TW, ty * TH, min(TW, F.W - tx * TW), min(TH, F.row1 - F.row0 - ty * TH));
        }
    }
    PH(0);
    for (unsigned cta = first; cta < nb; cta += stride) {
        const uint4 cur = rec;
        if (cta != first) {
            if ((threadIdx.x & 31) == 0) tma_wait_read();   // the previous tile's rows have left shared memory
            __syncthreads();
        }
        if (cta + stride < nb) rec = lst[cta + stride];     // the next tile's record arrives while this one is rasterized
        raster_tile<C, TEX>(F, M, S, clear, (int)(cur.x >> 22), (int)(cur.x & 2047u), (int)((cur.x >> 11) & 2047u), cur.y, cur.z,
                    (int)(cur.w & 255u), (int)(cur.w >> 8));
    }
#ifdef CRB_PHASE_TIMING
    ph_t = clock64();
#endif
    if ((threadIdx.x & 31) == 0) tma_wait_read();           // shared memory must outlive the bulk reads
    PH(10);
}

// The two throughput shapes of the tile rasterizer, both CTAs of 128 threads that store shaded pixels straight from registers
// (the third, RasterWide, follows them).
// Round 1 / early round 2 ran ONE shape: 256 threads, 128 triangles staged per pass, shaded rows staged in shared memory for TMA
// boxes, 6 CTAs per SM at 40 registers.  ncu showed 28 % of all stall samples at block barriers -- the eight warps of a CTA waiting
// for each other before shading, while most tiles hold 20-40 triangles, i.e. fewer (triangle, row) items than eight warps take
// 32 at a time.  Four warps per tile idle less, run the per-warp prologue half as often, and without the 24 KB of row staging
// twice as many tiles are in flight per SM (measured, k_raster per 128 T-Rex views / bunny 4096^2 / 10 M-triangle sphere 8192^2):
//     256 threads, CH 128, rows staged, 6 CTAs/SM, 40 registers      1003 / 286 / 1193 us
//     192 threads, CH  64,              8 CTAs/SM, 40 registers       929 / 265 / 1193
//     160 threads, CH  56,              9 CTAs/SM, 40 registers       895 / 253 / 1239
//     128 threads, CH  32, FQ 128,     12 CTAs/SM, 40 registers       883 / 246 / 1492
//     128 threads, CH  24, FQ 256,     12 CTAs/SM, 40 registers       868 / 232 / 1680    <- RasterSmall
//     128 threads, CH  96, FQ 256,      8 CTAs/SM, 62 registers       911 / 252 / 1107    <- RasterLarge
//     128 threads, CH 128, FQ 256,      7 CTAs/SM, 66 registers       965 / 270 / 1133
// Tiles of ~150 triangles (the sphere) want many triangles per staging pass and registers instead of warps; ordinary frames want
// many small CTAs.  run_raster picks the shape per launch from the triangles per busy tile the previous launch posted.
#ifdef CRB_LARGE_OUT_STAGE       // (shaded rows staged for TMA boxes: 24 KB more shared memory per CTA, needs CRB_RASTER_MIN_CTAS <= 6)
constexpr bool LARGE_OUT_STAGE = true;
#else
constexpr bool LARGE_OUT_STAGE = false;
#endif
typedef RasterShape<CRB_RT, CRB_CH, CRB_FQ, CRB_CLEAR_ROWS, CRB_RASTER_MIN_CTAS, LARGE_OUT_STAGE> RasterLarge;
#ifndef CRB_SMALL_RT
#define CRB_SMALL_RT 128
#endif
#ifndef CRB_SMALL_CH
#define CRB_SMALL_CH 24
#endif
#ifndef CRB_SMALL_FQ
#define CRB_SMALL_FQ 256
#endif
#ifndef CRB_SMALL_CLEAR_ROWS
#define CRB_SMALL_CLEAR_ROWS 8
#endif
#ifndef CRB_SMALL_MIN_CTAS
#define CRB_SMALL_MIN_CTAS 12
#endif
typedef RasterShape<CRB_SMALL_RT, CRB_SMALL_CH, CRB_SMALL_FQ, CRB_SMALL_CLEAR_ROWS, CRB_SMALL_MIN_CTAS, false> RasterSmall;
// ... and a third for frames of so few busy tiles that they do not fill the machine once (a single 1024^2 frame): eight warps per
// tile, 128 triangles per pass -- such a frame takes as long as its slowest CTA, and idle warps cost nothing there
typedef RasterShape<256, 128, 256, 16, 6, false> RasterWide;
#ifndef CRB_SHAPE_LARGE_FROM
#define CRB_SHAPE_LARGE_FROM 64      // triangles per busy tile from which the large shape is launched
#endif

// ------------------------------------------------------------------------------------------------------------
// Differential path (CRB_PATH_ATOMIC): one warp per triangle, global 64-bit atomicMin, then a per-pixel shade.
// Same records, same arithmetic, no binning, no shared memory -- an independent check of the tiled path.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT) k_raster_atomic(const Frame F, unsigned long long *keybuf)
{
    const long long slot = ((long long)blockIdx.x * NT + threadIdx.x) >> 5;     // entry of a chunk's dense list of drawn triangles
    const int lane = threadIdx.x & 31;
    if (slot >= F.T || (unsigned)(slot % NT) >= F.alive[slot / NT]) return;
    const float4 r2 = F.recE[slot];
    const unsigned bx = __float_as_uint(r2.x), by = __float_as_uint(r2.y);
    if ((bx >> 16) == 0) return;       // an entry whose pixel rectangle is empty
    const long long tri = slot / NT * NT + (__float_as_uint(r2.z) & 255u);
    const Tri9 t = load_tri9(F, tri);
    const int xl = bx & 0xFFFF, xr = bx >> 16, yt = by & 0xFFFF, yb = by >> 16;
    const int bw = xr - xl;
    const long long area = (long long)bw * (yb - yt);
    for (long long i = lane; i < area; i += 32) {
        const int x = xl + (int)(i % bw), y = yt + (int)(i / bw);
        float b1, b2, b3;
        barycentric(t, (float)x, (float)y, b1, b2, b3);
        if (b1 < 0.0f || b2 < 0.0f || b3 < 0.0f) continue;
        const float z = (t.z0 * b1 + t.z1 * b2) + t.z2 * b3;
        if (z != z) continue;
        atomicMin(keybuf + (long long)(y - F.row0) * F.W + x, pack_key(z, (unsigned)tri));
    }
}

template <int TEX>
__global__ void __launch_bounds__(NT) k_shade_atomic(const Frame F, unsigned long long *keybuf)
{
    const long long pix = (long long)blockIdx.x * NT + threadIdx.x;
    if (pix >= F.slabPixels) return;
    const unsigned long long key = keybuf[pix];
    const bool clear = (F.flags & CRB_CLEAR_FIRST) != 0;
    float z = Z_INIT, c[3] = {0.f, 0.f, 0.f}, nn[3] = {0.f, 0.f, 0.f};
    bool write = clear;
    if (key != KEY_EMPTY) {
        keybuf[pix] = KEY_EMPTY;
        const unsigned tri = ~(unsigned)(key & 0xFFFFFFFFull);
        const int y = F.row0 + (int)(pix / F.W), x = (int)(pix % F.W);
        float fz, fc[3], fn[3];
        if (shade_fragment<TEX>(F, F.shrec + (size_t)tri * SREC, (float)x, (float)y, fz, fc, fn)) {
            const float zold = clear ? Z_INIT : F.z[pix];
            if (!(fz > zold)) {
                z = fz; c[0] = fc[0]; c[1] = fc[1]; c[2] = fc[2]; nn[0] = fn[0]; nn[1] = fn[1]; nn[2] = fn[2];
                write = true;
            }
        }
    }
    if (!write) return;
    F.z[pix] = z;
    F.color[pix * 3] = c[0]; F.color[pix * 3 + 1] = c[1]; F.color[pix * 3 + 2] = c[2];
    F.normals[pix * 3] = nn[0]; F.normals[pix * 3 + 1] = nn[1]; F.normals[pix * 3 + 2] = nn[2];
}

// ------------------------------------------------------------------------------------------------------------
// small kernels: fills, post-passes, view export
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT) k_fill_u64(unsigned long long *p, long long n, unsigned long long v)
{
    for (long long i = (long long)blockIdx.x * NT + threadIdx.x; i < n; i += (long long)gridDim.x * NT) p[i] = v;
}

// crb_pack_texture: uint8 [texels,3] (BGR) -> uint32 B | G << 8 | R << 16, so that a textured pixel reads its texel with one
// aligned 4-byte load instead of three byte loads
__global__ void __launch_bounds__(NT) k_pack_texture(const uint8_t *__restrict__ bgr, long long texels, uint32_t *__restrict__ out)
{
    const long long stride = (long long)gridDim.x * NT;
    for (long long i = (long long)blockIdx.x * NT + threadIdx.x; i < texels; i += stride)
        out[i] = (uint32_t)bgr[3 * i] | ((uint32_t)bgr[3 * i + 1] << 8) | ((uint32_t)bgr[3 * i + 2] << 16);
}

// crb_pack_texture_mips: level k+1 of a mip chain from level k (DESIGN 2), one thread per destination texel, per channel
// (t[r0][c0] + t[r0][c1] + t[r1][c0] + t[r1][c1] + 2) >> 2 with r0 = min(2r, sh-1), r1 = min(2r+1, sh-1), columns alike
__global__ void __launch_bounds__(NT) k_mip_level(const uint32_t *__restrict__ src, int sh, int sw, uint32_t *__restrict__ dst, int dh, int dw)
{
    const long long n = (long long)dh * dw, stride = (long long)gridDim.x * NT;
    for (long long i = (long long)blockIdx.x * NT + threadIdx.x; i < n; i += stride) {
        const int r = (int)(i / dw), c = (int)(i - (long long)r * dw);
        const int r0 = min(2 * r, sh - 1), r1 = min(2 * r + 1, sh - 1), c0 = min(2 * c, sw - 1), c1 = min(2 * c + 1, sw - 1);
        const uint32_t a = __ldg(src + r0 * sw + c0), b = __ldg(src + r0 * sw + c1);
        const uint32_t d = __ldg(src + r1 * sw + c0), e = __ldg(src + r1 * sw + c1);
        uint32_t out = 0;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int sh8 = 8 * k;
            const uint32_t s = ((a >> sh8) & 255u) + ((b >> sh8) & 255u) + ((d >> sh8) & 255u) + ((e >> sh8) & 255u) + 2u;
            out |= (s >> 2) << sh8;
        }
        dst[i] = out;
    }
}

// pyx:65-67
__global__ void __launch_bounds__(NT) k_init_buffers(float *z, float *color, float *normals, long long pixels)
{
    const long long stride = (long long)gridDim.x * NT;
    for (long long i = (long long)blockIdx.x * NT + threadIdx.x; i < pixels * 3; i += stride) {
        color[i] = 0.0f;
        normals[i] = 0.0f;
        if (i < pixels) z[i] = Z_INIT;
    }
}

// One tile of the sparse read-back, by one warp; returns the tile rows it copied.
__device__ __forceinline__ unsigned readback_tile(const Frame &F, const unsigned t, unsigned *shown_rows, float *hz, float *hc, float *hn)
{
    const bool busy = F.cursor[t] != 0u;                          // k_fill left the tile's pair count here
    const unsigned before = shown_rows[t];
    const int tx = (int)(t % (unsigned)F.tilesX), ty = (int)(t / (unsigned)F.tilesX);
    const int x0 = tx * TW, yl0 = ty * TH;
    const int tw = min(TW, F.W - x0), th = min(TH, F.row1 - F.row0 - yl0);
    const unsigned lane = threadIdx.x & 31u;
    unsigned now = 0u, copied = 0u;
    if (tw == TW && !(F.W & 3)) {
        // a tile row is 56 float4: 8 of z, 24 of colour, 24 of normals; lane l takes float4 l and l + 32 of the row.
        // Four rows are read before any is written, so that a few warps keep the link busy.
        constexpr int RB = 4;
        const float f0 = lane < 8u ? Z_INIT : background_color(F);   // fresh value of the lane's first float4 (z | colour)
        for (int r0 = 0; r0 < th; r0 += RB) {
            float4 a[RB], b[RB];
#pragma unroll
            for (int j = 0; j < RB; ++j) {
                a[j] = b[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (r0 + j < th) {
                    const long long rowpix = (long long)(yl0 + r0 + j) * F.W + x0;
                    a[j] = lane < 8u ? reinterpret_cast<const float4 *>(F.z + rowpix)[lane]
                                     : reinterpret_cast<const float4 *>(F.color + rowpix * 3)[lane - 8u];
                    if (lane < 24u) b[j] = reinterpret_cast<const float4 *>(F.normals + rowpix * 3)[lane];   // float4 32..55: the normals
                }
            }
#pragma unroll
            for (int j = 0; j < RB; ++j) {
                const int r = r0 + j;
                if (r >= th) break;
                const long long rowpix = (long long)(yl0 + r) * F.W + x0;
                // bit comparison: -0.0 or NaN in a written pixel is not "fresh"
                const bool differs = __float_as_uint(a[j].x) != __float_as_uint(f0) || __float_as_uint(a[j].y) != __float_as_uint(f0) ||
                                     __float_as_uint(a[j].z) != __float_as_uint(f0) || __float_as_uint(a[j].w) != __float_as_uint(f0) ||
                                     (__float_as_uint(b[j].x) | __float_as_uint(b[j].y) | __float_as_uint(b[j].z) | __float_as_uint(b[j].w)) != 0u;
                const bool holds = __any_sync(0xFFFFFFFFu, differs);
                if (holds) now |= 1u << r;
                if (holds || ((before >> r) & 1u)) {
                    if (lane < 8u) { if (hz) reinterpret_cast<float4 *>(hz + rowpix)[lane] = a[j]; }
                    else if (hc) reinterpret_cast<float4 *>(hc + rowpix * 3)[lane - 8u] = a[j];
                    if (lane < 24u && hn) reinterpret_cast<float4 *>(hn + rowpix * 3)[lane] = b[j];
                    ++copied;
                }
            }
        }
    } else {
        // ragged tiles (image edge, widths that are not a multiple of 4): whole tile, element by element
        for (int i = (int)lane; i < th * tw; i += 32) {
            const int r = i / tw, xx = i % tw;
            const long long p = (long long)(yl0 + r) * F.W + x0 + xx;
            if (hz) hz[p] = F.z[p];
            if (hc) { hc[p * 3] = F.color[p * 3]; hc[p * 3 + 1] = F.color[p * 3 + 1]; hc[p * 3 + 2] = F.color[p * 3 + 2]; }
            if (hn) { hn[p * 3] = F.normals[p * 3]; hn[p * 3 + 1] = F.normals[p * 3 + 1]; hn[p * 3 + 2] = F.normals[p * 3 + 2]; }
        }
        now = busy ? 0xFFFFFFFFu : 0u;
        copied = (unsigned)th;
    }
    if (lane == 0u) shown_rows[t] = now;
    return copied;
}

// Sparse read-back (crb_render_host + CRB_DL_SPARSE).  The host copy of the three buffers persists between calls, every
// call renders a FRESH frame, and a pixel row no fragment was written to holds fresh-filler values both before and after --
// so only the 32-pixel tile rows that hold something now, or held something in the frame the host copy currently shows,
// need to cross PCIe.  A SMALL grid does it (READBACK_CTAS): the copy is bound by the link, a few dozen warps saturate it,
// and a larger grid only deepens the queue of posted writes that the next frame's upload and kernel launches (whose read
// requests share the upstream link) have to wait behind -- measured on the T-Rex orbit, three frames in flight: 1 024
// CTAs 5 170, 8 CTAs 5 450 frames/s (colour only: 8 200 -> 9 800).  CTA b looks at the tiles b, b + G, b + 2G, ... (busy
// tiles cluster in space; the interleave spreads them over the CTAs), lists those that are busy now or have rows to take
// back, and its warps take one listed tile each: a warp compares the tile's rows with the fresh pattern (z 1e6, colour /
// normals 0) as it reads them, copies the rows that differ now or differed before straight into the mapped pinned host
// arrays (16-byte stores, 128 / 384-byte runs), and keeps the tile's new row mask for the next call.  The host arrays end
// up bit-identical to a full download (tests/test_gpu_parity.py::test_sparse_readback_*).  `rows_copied` counts tile
// rows (32 pixels x 28 bytes when all three buffers are wanted).
constexpr int READBACK_CTAS = 8;

__global__ void __launch_bounds__(NT) k_readback(const Frame F, unsigned *shown_rows, float *hz, float *hc, float *hn,
                                                  unsigned long long *rows_copied)
{
    __shared__ unsigned s_list[NT];
    __shared__ unsigned s_n;
    if (F.total[0] > (unsigned long long)F.pairCap) return;      // frame skipped: the host copy stays as it is
    const unsigned G = gridDim.x, nT = (unsigned)F.nTiles, perCta = (nT + G - 1u) / G;
    unsigned copied = 0u;
    for (unsigned k0 = 0; k0 < perCta; k0 += NT) {
        if (threadIdx.x == 0) s_n = 0u;
        __syncthreads();
        const unsigned k = k0 + threadIdx.x;
        const unsigned long long t = (unsigned long long)k * G + blockIdx.x;
        if (k < perCta && t < nT && (F.cursor[t] != 0u || shown_rows[t] != 0u)) s_list[atomicAdd(&s_n, 1u)] = (unsigned)t;
        __syncthreads();
        const unsigned n = s_n;
        for (unsigned i = threadIdx.x >> 5; i < n; i += NT / 32) copied += readback_tile(F, s_list[i], shown_rows, hz, hc, hn);
        __syncthreads();
    }
    if ((threadIdx.x & 31) == 0 && copied) atomicAdd(rows_copied, (unsigned long long)copied);
}

// guro_illumination.py:20-27 over the whole buffer, in place
__global__ void __launch_bounds__(NT) k_guro(float *color, const float *normals, long long pixels, float l0, float l1, float l2)
{
    const long long stride = (long long)gridDim.x * NT;
    for (long long i = (long long)blockIdx.x * NT + threadIdx.x; i < pixels; i += stride) {
        const float n0 = normals[i * 3], n1 = normals[i * 3 + 1], n2 = normals[i * 3 + 2];
        const float dot = (__fadd_rn(0.0f, n0 * l0) + n1 * l1) + n2 * l2;   // np.sum accumulates from +0.0
        const float nrm = sqrtf((n0 * n0 + n1 * n1) + n2 * n2);
        float s = dot / (nrm + 1e-6f);
        if (s < 0.0f) s = 0.0f;
        if (s > 1.0f) s = 1.0f;
        color[i * 3] *= s; color[i * 3 + 1] *= s; color[i * 3 + 2] *= s;
    }
}

// run.py:26
__global__ void __launch_bounds__(NT) k_color_u8_flipped(const float *color, unsigned char *out, int rows, int W)
{
    const long long n = (long long)rows * W * 3, stride = (long long)gridDim.x * NT;
    const long long rowElems = (long long)W * 3;
    for (long long i = (long long)blockIdx.x * NT + threadIdx.x; i < n; i += stride) {
        const long long r = i / rowElems, e = i % rowElems;
        out[(rows - 1 - r) * rowElems + e] = to_u8(color[i]);
    }
}

__global__ void __launch_bounds__(NT) k_transform_view(const float *v, const float *n, long long nVerts, const float *view,
                                                       float *vo, float *no)
{
    __shared__ float M[16];
    if (threadIdx.x < 16) M[threadIdx.x] = view[threadIdx.x];
    __syncthreads();
    const long long i = (long long)blockIdx.x * NT + threadIdx.x;
    if (i >= nVerts) return;
    float x = v[i * 3], y = v[i * 3 + 1], z = v[i * 3 + 2];
    view_point(M, x, y, z);
    vo[i * 3] = x; vo[i * 3 + 1] = y; vo[i * 3 + 2] = z;
    x = n[i * 3]; y = n[i * 3 + 1]; z = n[i * 3 + 2];
    view_normal(M, x, y, z);
    no[i * 3] = x; no[i * 3 + 1] = y; no[i * 3 + 2] = z;
}

// Self-test of div_rn_by against the IEEE division instruction sequence: pseudo-random and adversarial operands
// (all-ones / all-zeros significands, neighbours of powers of two) with exponents spanning the admitted range.
__device__ __forceinline__ unsigned mix32(unsigned x)
{
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}
__device__ __forceinline__ float selftest_operand(unsigned h, unsigned h2)
{
    unsigned mant = h & 0x7FFFFFu;
    const unsigned kind = (h2 >> 8) & 15u;
    if (kind == 0) mant = 0x7FFFFFu;              // 1.11...1
    else if (kind == 1) mant = 0u;                // power of two
    else if (kind == 2) mant = 1u;
    else if (kind == 3) mant = 0x7FFFFEu;
    else if (kind == 4) mant = 0x400000u;         // 1.5
    else if (kind == 5) mant &= 0x7FF000u;        // short significands (screen coordinates are often like this)
    const unsigned expo = 127u - 40u + (h2 % 81u);   // 2^-40 .. 2^40
    return __uint_as_float(((h2 >> 31) << 31) | (expo << 23) | mant);
}
__global__ void __launch_bounds__(NT) k_selftest_fdiv(unsigned long long samples, unsigned seed, unsigned long long *out)
{
    unsigned long long bad = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * NT + threadIdx.x; i < samples; i += (unsigned long long)gridDim.x * NT) {
        const unsigned h0 = mix32((unsigned)i ^ seed), h1 = mix32(h0 + (unsigned)(i >> 32) + 0x9e3779b9u);
        const unsigned h2 = mix32(h1 ^ 0x85ebca6bu), h3 = mix32(h2 + 0xc2b2ae35u);
        const float a = selftest_operand(h0, h1), d = selftest_operand(h2, h3);
        const float fast = div_rn_by(a, d, __frcp_rn(d)), ref = __fdiv_rn(a, d);
        if (__float_as_uint(fast) != __float_as_uint(ref)) {
            if (!bad) { out[1] = __float_as_uint(a); out[2] = __float_as_uint(d); }
            ++bad;
        }
    }
    if (bad) atomicAdd(out, bad);
}

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
thread_local char g_err[512] = "";

int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess) return fail(CRB_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_));     \
    } while (0)

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace

// for the library's other translation unit (ingest_b200.cu); not exported
int crb_internal_fail(int code, const char *msg) { return fail(code, "%s", msg); }

struct crb_filler {
    int h, w, device;
    int row0, row1;
    float fov, z_near, z_far;
    ProjC proj;
    // outputs
    float *z, *color, *normals;
    bool own_buffers;
    // workspace
    void *ws;
    size_t ws_bytes;
    bool own_ws;
    long long maxT;
    int maxViews;
    long long pairCap;
    float4 *shrec, *recE;
    unsigned short *alive;
    unsigned *chunks;
    unsigned *count, *offset, *cursor, *empty;
    uint4 *busy, *busyH;
    float4 *ls;
    uint4 *wide;
    long long wideCap;
    unsigned long long *total;
    float *stage_v, *stage_c, *stage_n;  // device staging for host-pointer calls
    // differential path scratch (library-owned, lazily allocated)
    unsigned long long *keybuf;
    long long keybuf_pixels;
    long long launches;
    // optional timing of the dominant kernel (k_raster) with CUDA events on the launching stream
    int raster_ctas;       // experiments: fixed k_raster grid (0 = automatic)
    int raster_shape;      // CRB_OPT_RASTER_SHAPE: 0 = per launch from the posted statistics, 1 = RasterLarge, 2 = RasterSmall, 3 = RasterWide
    int sm_count;
    int use_tma;           // tensor maps are built where the layout allows (CRB_NO_TMA=1 disables): k_clear stores TMA boxes
    unsigned *shown_busy;        // sparse read-back: per tile, mask of the 32 rows that hold something in the frame the caller's host arrays show
    long long shown_tiles;
    unsigned long long *tiles_copied;   // device counter behind crb_readback_stats
    const void *map_host[3];     // host pointers already resolved to device-visible addresses
    void *map_dev[3];
    size_t set_bytes;      // size of one workspace set
    cudaStream_t s_prep, s_raster;      // batched views: setup/binning of launch i+1 runs beside the rasterizer of launch i
    cudaEvent_t ev_start, ev_fill[2], ev_raster[2];
    int chunk_pipeline;    // CRB_CHUNK_PIPELINE=0 disables
    unsigned launch_seq;   // launches issued through the two-stream pipeline (parity = workspace set)
    int set_used[2];       // the set has a rasterizer launch whose completion is recorded in ev_raster[set]
    int pending_join;      // 1 + set of the last pipelined launch the caller's stream has not been made to wait for (CRB_DEFER_JOIN)
    int split_heavy;       // single-view launches cut heavy tiles into row bands (CRB_SPLIT_HEAVY=0 disables)
    int band_prepass;      // band-sharded fillers list the chunks that reach the band first (CRB_OPT_BAND_PREPASS)
    int tiles_per_cta;     // k_raster grid = estimated busy tiles / this (CRB_TILES_PER_CTA)
    unsigned dbg_flags;    // ablation switches (CRB_DEBUG_SKIP), never set in production
    int out_tma;           // ... and so does k_raster for the shaded colour / normal rows (CRB_OUT_TMA=0 disables)
    unsigned long long *hstats;      // pinned + mapped: busy-tile statistics of the most recent k_raster launch
    unsigned long long *hstats_dev;
    bool prof_on;
    int prof_n;
    cudaEvent_t *prof_ev;  // 2 * PROF_MAX events, created on first use
    int wide_kernel;       // triangles that span many tiles are scattered by k_fill_wide (CRB_OPT_WIDE_KERNEL = 0: by k_fill itself)
    unsigned char *u8x[CRB_MAX_EXCHANGE];   // crb_set_u8_exchange: receive buffer of every row band (u8x_n == 0: off)
    int u8x_n, u8x_rows;
    const uint32_t *tex;   // crb_bind_texture: packed texels (caller-owned device memory), NULL = none
    int tex_h, tex_w;
    int tex_levels;        // crb_bind_texture_mips: levels of the bound chain; 0 = a single level (crb_bind_texture)
};

namespace {

struct WsLayout {
    size_t shrec, recE, alive, chunks, count, offset, cursor, busy, busyH, empty, ls, wide, total, set_bytes, sv, sc, sn, bytes;
};

long long default_pair_cap(const crb_filler *f, long long T, int views)
{
    const long long tiles = (long long)((f->w + TW - 1) / TW) * ((f->row1 - f->row0 + TH - 1) / TH);
    long long cap = 4 * T * views + tiles * views + 65536;
    return cap;
}

long long wide_capacity(long long T, int views) { return (T > 0 ? T : 1) * views / 8 + 1024; }

WsLayout ws_layout(const crb_filler *f, long long T, int views, long long pairCap)
{
    WsLayout L;
    const long long tiles = (long long)((f->w + TW - 1) / TW) * ((f->row1 - f->row0 + TH - 1) / TH);
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o = align_up(o + bytes, 256); return at; };
    const size_t recs = (size_t)(T > 0 ? T : 1) * views;
    L.shrec = take(recs * SREC * sizeof(float4));
    L.recE = take(recs * sizeof(float4));
    L.alive = take((size_t)((T > 0 ? T : 1) + NT - 1) / NT * views * sizeof(unsigned short));
    L.chunks = take(4 * ((size_t)((T > 0 ? T : 1) + NT - 1) / NT + 2));
    L.count = take((size_t)tiles * views * 4);
    L.offset = take((size_t)tiles * views * 4);
    L.cursor = take((size_t)tiles * views * 4);
    L.busy = take((size_t)tiles * views * 16);
    L.busyH = take((size_t)tiles * views * 16 * SPLIT_BANDS);
    L.empty = take((size_t)tiles * views * 4);
    L.ls = take((size_t)pairCap * 64);
    L.wide = take((size_t)wide_capacity(T, views) * 16);
    L.total = take(64);
    L.set_bytes = o;            // everything above exists twice (two launches of a batch in flight, see crb_render_views)
    o = 2 * L.set_bytes;
    L.sv = take((size_t)(T > 0 ? T : 1) * 36);
    L.sc = take((size_t)(T > 0 ? T : 1) * 36);
    L.sn = take((size_t)(T > 0 ? T : 1) * 36);
    L.bytes = o;
    return L;
}

int check_filler(const crb_filler *f)
{
    if (!f) return fail(CRB_ERR_INVALID, "filler is NULL");
    return CRB_OK;
}

// Shared by every render entry point: triangle indices are packed into 32 bits (the ~tri half of the visibility key, the
// staged triangle's index word), so a larger T would silently alias winners.
int check_triangles(const crb_filler *f, int64_t T, const float *v, const float *c, const float *n)
{
    if (T < 0) return fail(CRB_ERR_INVALID, "T < 0");
    if (T > 0 && (!v || !c || !n)) return fail(CRB_ERR_INVALID, "NULL triangle array");
    if (!f->ws) return fail(CRB_ERR_STATE, "workspace not bound");
    if (T > f->maxT) return fail(CRB_ERR_STATE, "T=%lld exceeds the workspace's max_triangles=%lld", (long long)T, f->maxT);
    if (T > 0xFFFFFFF0ll) return fail(CRB_ERR_INVALID, "T exceeds 32-bit triangle indices");
    return CRB_OK;
}

int host_projection(int h, int w, float fov, float z_near, float z_far, ProjC *P)
{
    if (w == 0) return fail(CRB_ERR_ZERODIV, "division by zero");  // pyx:59 h / w
    const float a = (float)((double)h / (double)w);
    const double ang = (((double)fov / 2.0) / 180.0) * 3.141592653589793;  // pyx:55, np.pi
    const float fl = (float)(1.0 / tan(ang));
    const float d = z_far - z_near;
    if (d == 0.0f || a == 0.0f) return fail(CRB_ERR_ZERODIV, "float division");  // pyx:84, pyx:86
    const float q = z_far / d;
    memset(P->p, 0, sizeof(P->p));
    P->p[0] = fl / a;
    P->p[5] = fl;
    P->p[10] = q;
    P->p[11] = 1.0f;
    P->p[14] = (-z_near) * q;
    P->xs = (float)((double)w / 2.0);
    P->ys = (float)((double)h / 2.0);
    return CRB_OK;
}

void fill_frame(const crb_filler *f, Frame *F, int set = 0)
{
    memset(F, 0, sizeof(*F));
    F->proj = f->proj;
    F->W = f->w;
    F->H = f->h;
    F->row0 = f->row0;
    F->row1 = f->row1;
    F->tilesX = (f->w + TW - 1) / TW;
    F->tilesY = (f->row1 - f->row0 + TH - 1) / TH;
    F->nTiles = F->tilesX * F->tilesY;
    const size_t so = set ? f->set_bytes : 0;     // the second workspace set lies set_bytes behind the first
    auto at = [so](auto *p) { return reinterpret_cast<decltype(p)>(reinterpret_cast<char *>(p) + so); };
    F->shrec = at(f->shrec); F->recE = at(f->recE); F->alive = at(f->alive);
    F->count = at(f->count); F->offset = at(f->offset); F->cursor = at(f->cursor);
    F->busy = at(f->busy); F->busyH = at(f->busyH); F->empty = at(f->empty);
    F->ls = at(f->ls);
    F->wide = at(f->wide);
    F->wideCap = 0;          // run_prep decides per launch whether k_fill_wide follows k_fill
    F->total = at(f->total);
    F->hstats = f->hstats_dev;
    F->pairCap = f->pairCap;
    F->slabPixels = (long long)(f->row1 - f->row0) * f->w;
    F->tex = f->tex;
    F->texH = f->tex_h;
    F->texW = f->tex_w;
}

// CRB_TEX_PERSPECTIVE, CRB_TEX_BILINEAR and CRB_TEX_TRILINEAR are modes of CRB_TEXTURE, which needs a bound texture;
// CRB_TEX_TRILINEAR needs a bound mip chain and excludes CRB_TEX_BILINEAR
int check_texture(const crb_filler *f, unsigned flags)
{
    if ((flags & (CRB_TEX_PERSPECTIVE | CRB_TEX_BILINEAR | CRB_TEX_TRILINEAR)) && !(flags & CRB_TEXTURE))
        return fail(CRB_ERR_INVALID, "CRB_TEX_PERSPECTIVE / CRB_TEX_BILINEAR / CRB_TEX_TRILINEAR need CRB_TEXTURE");
    if ((flags & CRB_TEX_BILINEAR) && (flags & CRB_TEX_TRILINEAR))
        return fail(CRB_ERR_INVALID, "CRB_TEX_BILINEAR and CRB_TEX_TRILINEAR exclude each other");
    if ((flags & CRB_TEXTURE) && !f->tex) return fail(CRB_ERR_STATE, "CRB_TEXTURE: no texture bound (crb_bind_texture)");
    if ((flags & CRB_TEX_TRILINEAR) && !f->tex_levels)
        return fail(CRB_ERR_STATE, "CRB_TEX_TRILINEAR: no mip chain bound (crb_bind_texture_mips)");
    return CRB_OK;
}

int launch_check(crb_filler *f, const char *name)
{
    f->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(CRB_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(e));
    return CRB_OK;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda).
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn()
{
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
        else
            cudaGetLastError();
    }
    return fn;
}

// [views][rows][W*comps] float32, boxes of BOX_ROWS x (TW*comps).  Returns false if the layout cannot be described.
bool encode_map(CUtensorMap *m, float *base, int comps, const Frame &F, int box_rows)
{
    EncodeTiledFn fn = encode_tiled_fn();
    const long long rows = F.row1 - F.row0;
    if (!fn || !base || rows <= 0 || (reinterpret_cast<uintptr_t>(base) & 15u)) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)F.W * comps, (cuuint64_t)rows, (cuuint64_t)F.nViews};
    const cuuint64_t strides[2] = {(cuuint64_t)F.W * comps * 4, (cuuint64_t)rows * F.W * comps * 4};
    const cuuint32_t box[3] = {(cuuint32_t)(TW * comps), (cuuint32_t)box_rows, 1u};
    const cuuint32_t es[3] = {1u, 1u, 1u};
    return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// All or nothing: every non-NULL output array gets a map, or the launch uses plain stores.
unsigned encode_maps(TMaps *M, const Frame &F, int clear_rows)
{
    unsigned use = 0;
    if (F.z) { if (!encode_map(&M->z, F.z, 1, F, BOX_ROWS) || !encode_map(&M->zt, F.z, 1, F, clear_rows)) return 0u; use |= CRB_BUF_Z; }
    if (F.color) { if (!encode_map(&M->c, F.color, 3, F, BOX_ROWS) || !encode_map(&M->ct, F.color, 3, F, clear_rows)) return 0u; use |= CRB_BUF_COLOR; }
    if (F.normals) { if (!encode_map(&M->n, F.normals, 3, F, BOX_ROWS) || !encode_map(&M->nt, F.normals, 3, F, clear_rows)) return 0u; use |= CRB_BUF_NORMALS; }
    return use;
}

// project/setup/count -> alloc -> fill -> raster+shade for up to maxViews views
// k_setup's ring of stages needs more than the 48 KB of shared memory a kernel gets by default: opt in once per device
int setup_smem_attr(int device)
{
    static bool done[64] = {};
    if (device >= 0 && device < 64 && done[device]) return CRB_OK;
    CU(cudaFuncSetAttribute(k_setup<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SETUP_DYN_SMEM));
    CU(cudaFuncSetAttribute(k_setup<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SETUP_DYN_SMEM));
    if (device >= 0 && device < 64) done[device] = true;
    return CRB_OK;
}

// k_setup with `grid` CTAs; CRB_TEX_PERSPECTIVE frames write the perspective-correct texture coordinates into the records
void launch_setup(const Frame &F, unsigned grid, cudaStream_t st)
{
    if (F.flags & CRB_TEX_PERSPECTIVE) k_setup<true><<<grid, NT, SETUP_DYN_SMEM, st>>>(F);
    else k_setup<false><<<grid, NT, SETUP_DYN_SMEM, st>>>(F);
}

#ifndef CRB_PREPASS_EIGHTHS
#define CRB_PREPASS_EIGHTHS 5  // the band pre-pass runs for bands of at most this many eighths of the frame (half-frame bands gain
                               // 7 %; a cut balanced by measurement lands a few strips off the middle, which must not switch it off)
#endif
// project/setup/count -> alloc -> fill for up to maxViews views
int run_prep(crb_filler *f, Frame &F, cudaStream_t st, int slot = 0)
{
    int rc;
    // Triangles that span many tiles get a kernel of their own (k_fill_wide) -- but only where there are any: the launch is
    // issued when the previous frame at this position of the batch posted two dozen or more per view (k_raster reports their
    // number with the busy-tile statistics) or has not reported yet; otherwise k_fill scatters the odd one itself, as it does when the list is full.
    bool wide_kernel = false;
    if (f->hstats && f->wide_kernel) {
        const unsigned long long hs = *reinterpret_cast<volatile unsigned long long *>(f->hstats + HSTAT_WORDS * (slot & 7));
        const unsigned long long hw = *reinterpret_cast<volatile unsigned long long *>(f->hstats + HSTAT_WORDS * (slot & 7) + 1) >> 32;
        wide_kernel = hs == 0ull || hw >= 24ull * (unsigned long long)F.nViews;      // (a handful per view is quicker done in place than launched for)
    }
    F.wideCap = wide_kernel && !(F.flags & CRB_PATH_ATOMIC) ? (unsigned)(f->wideCap > 0xFFFFFFF0ll ? 0xFFFFFFF0ll : f->wideCap) : 0u;
    unsigned gT = (unsigned)((F.T + NT - 1) / NT);
    // band-sharded single view: list the chunks that can reach the band first, then walk only those (persistent grids)
    const bool banded = F.row0 > 0 || F.row1 < F.H;
    F.chunks = nullptr;
    // (it reads the vertex array once more than k_setup alone would: it pays when many chunks miss the band -- measured on the
    // 10 M-triangle sphere with the persistent k_setup that walks the listed chunks through its bulk-copy ring: half-frame bands
    // 1.14 -> 1.06 ms; round 1, with one-chunk CTAs: half 1.16 -> 1.22 ms, quarter 0.84 -> 0.82, eighth 0.59 -> 0.51)
    if (banded && f->band_prepass && 8ll * (F.row1 - F.row0) <= (long long)CRB_PREPASS_EIGHTHS * F.H && F.nViews == 1 && !F.views && F.T >= 8 * NT && !(F.flags & CRB_PATH_ATOMIC) &&
        !(reinterpret_cast<uintptr_t>(F.v) & 15u)) {
        const size_t so = (size_t)(reinterpret_cast<const char *>(F.alive) - reinterpret_cast<const char *>(f->alive));   // workspace set in use
        F.chunks = reinterpret_cast<unsigned *>(reinterpret_cast<char *>(f->chunks) + so);
        CU(cudaMemsetAsync(F.chunks, 0, 4, st));
        constexpr int bcPerSm = 4;   // 4 x 36 KB rings per SM
        const unsigned gP = (unsigned)min((long long)gT, (long long)f->sm_count * bcPerSm);
        k_band_chunks<<<gP, NT, 0, st>>>(F);
        if ((rc = launch_check(f, "k_band_chunks"))) return rc;
        gT = (unsigned)min((long long)gT, (long long)f->sm_count * 6);
    }
    if (F.T > 0) {
        if ((rc = setup_smem_attr(f->device))) return rc;
        const long long items = F.chunks ? (long long)gT : (long long)gT * F.nViews;
        launch_setup(F, (unsigned)min(items, (long long)f->sm_count * CRB_SETUP_MIN_CTAS), st);
        if ((rc = launch_check(f, "k_setup"))) return rc;
    } else {
        CU(cudaMemsetAsync(F.total, 0, 8, st));
        CU(cudaMemsetAsync(F.total + 2, 0, 24, st));
    }
    // cutting heavy tiles only pays while the frame is latency-bound, i.e. while its tiles do not fill the machine several
    // times over (T-Rex 1024^2: 56 -> 38 us; the 8192^2 sphere with 75 triangles in every tile would lose 25 %)
    F.splitHeavy = (F.nViews == 1 && f->split_heavy && F.nTiles <= 4 * f->sm_count * 6) ? 1u : 0u;
    const long long nAllTiles = (long long)F.nViews * F.nTiles;
    k_alloc<<<(unsigned)((nAllTiles + NT - 1) / NT), NT, 0, st>>>(F);
    if ((rc = launch_check(f, "k_alloc"))) return rc;
    if (F.T > 0) {
        k_fill<<<dim3(gT * (NT / FT), F.nViews), FT, 0, st>>>(F);
        if ((rc = launch_check(f, "k_fill"))) return rc;
        if (F.wideCap) {
            k_fill_wide<<<(unsigned)f->sm_count * 6, FWT, 0, st>>>(F);
            if ((rc = launch_check(f, "k_fill_wide"))) return rc;
        }
    }
    return CRB_OK;
}

// raster + shade (+ fused clear) of the frame run_prep binned
// shading instantiation of a frame: per-vertex colours, or per-pixel texturing with its filter and interpolation
int tex_mode(const Frame &F)
{
    if (!(F.flags & CRB_TEXTURE)) return TEX_NONE;
    const int filter = (F.flags & CRB_TEX_TRILINEAR) ? TEX_TRILINEAR : (F.flags & CRB_TEX_BILINEAR) ? TEX_BILINEAR : TEX_NEAREST;
    return filter | ((F.flags & CRB_TEX_PERSPECTIVE) ? TEX_PERSP : 0);
}

template <class C>
void launch_raster(const Frame &F, const TMaps &M, unsigned grid, cudaStream_t st)
{
    switch (tex_mode(F)) {
    case TEX_NEAREST: k_raster<C, TEX_NEAREST><<<grid, C::RT, 0, st>>>(F, M); break;
    case TEX_NEAREST | TEX_PERSP: k_raster<C, TEX_NEAREST | TEX_PERSP><<<grid, C::RT, 0, st>>>(F, M); break;
    case TEX_BILINEAR: k_raster<C, TEX_BILINEAR><<<grid, C::RT, 0, st>>>(F, M); break;
    case TEX_BILINEAR | TEX_PERSP: k_raster<C, TEX_BILINEAR | TEX_PERSP><<<grid, C::RT, 0, st>>>(F, M); break;
    case TEX_TRILINEAR: k_raster<C, TEX_TRILINEAR><<<grid, C::RT, 0, st>>>(F, M); break;
    case TEX_TRILINEAR | TEX_PERSP: k_raster<C, TEX_TRILINEAR | TEX_PERSP><<<grid, C::RT, 0, st>>>(F, M); break;
    default: k_raster<C, TEX_NONE><<<grid, C::RT, 0, st>>>(F, M);
    }
}

int run_raster(crb_filler *f, Frame &F, cudaStream_t st, int slot)
{
    int rc;
    slot &= 7;                                   // busy-tile statistics are kept per position in a batch of launches
    if (F.hstats) F.hstats += HSTAT_WORDS * slot;
    const long long nAllTiles = (long long)F.nViews * F.nTiles;
    const bool prof = f->prof_on && f->prof_n < PROF_MAX;
    // Shape of the rasterizer's CTAs (RasterSmall / RasterLarge / RasterWide, see there).  A frame whose busy tiles do not even
    // fill the machine once is as slow as its slowest CTA: the most threads per tile win (single T-Rex frame 1024^2: wide 36 us,
    // large 41, small 60); up to a few waves the large shape (T-Rex 2048^2: 67 vs 80 us); beyond that throughput counts and the
    // triangles per busy tile decide (bunny 4096^2, one frame: small 262 us, large 286, wide 315).  Busy tiles and pairs are those
    // the previous launch at this position of the batch posted; before any launch has reported, the frame's tiles and triangles.
    int shape = f->raster_shape;
    if (shape == 0) {
        const long long wave = (long long)f->sm_count * RasterWide::MIN_CTAS;
        double busy = (double)nAllTiles, per_tile = (double)F.T * 2.0 / (double)F.nTiles;
        if (f->hstats) {
            const unsigned long long hs = *reinterpret_cast<volatile unsigned long long *>(f->hstats + HSTAT_WORDS * slot);
            const unsigned long long hh = *reinterpret_cast<volatile unsigned long long *>(f->hstats + HSTAT_WORDS * slot + 1) & 0xFFFFFFFFull;
            const unsigned long long hp = *reinterpret_cast<volatile unsigned long long *>(f->hstats + HSTAT_WORDS * slot + 2);
            const double records = (double)((hs & 0xFFFFFFFFull) + hh);
            if ((hs >> 32) > 0 && records > 0) {
                busy = records * (double)nAllTiles / (double)(hs >> 32);
                per_tile = (double)hp / records;
            }
        }
        shape = busy <= (double)wave ? 3 : (busy <= 4.0 * (double)wave || per_tile >= (double)CRB_SHAPE_LARGE_FROM) ? 1 : 2;
    }
    const int clear_rows = shape == 2 ? RasterSmall::CLEAR_ROWS : shape == 3 ? RasterWide::CLEAR_ROWS : RasterLarge::CLEAR_ROWS;
    const int min_ctas = shape == 2 ? RasterSmall::MIN_CTAS : shape == 3 ? RasterWide::MIN_CTAS : RasterLarge::MIN_CTAS;
    TMaps M;
    memset(&M, 0, sizeof(M));
    const bool clear = (F.flags & CRB_CLEAR_FIRST) != 0;
    if (f->use_tma && clear && !(F.W & 3) && !F.color_u8) M.use = encode_maps(&M, F, clear_rows);
    if (M.use && f->out_tma == 1) F.flags |= FLAG_OUT_TMA;
    if (f->out_tma == 2) F.flags |= FLAG_OUT_DIRECT;
    F.flags |= f->dbg_flags;
    // Grid: one CTA per busy tile.  The busy count is only known on the device, so the grid is sized from the busy
    // FRACTION the previous launch posted (+12 % and a floor of one wave); k_raster walks with stride gridDim when the
    // estimate was low, and an all-tiles grid is used until a first launch has reported.
    long long gL = nAllTiles, gH = nAllTiles / 16 + 1;     // light / heavy rasterizing roles
    if (f->raster_ctas > 0) { gL = f->raster_ctas; gH = f->raster_ctas / 8 + 1; }
    else if (f->hstats && f->raster_ctas == 0) {
        const unsigned long long hs = *reinterpret_cast<volatile unsigned long long *>(f->hstats + HSTAT_WORDS * slot);
        const unsigned long long hh = *reinterpret_cast<volatile unsigned long long *>(f->hstats + HSTAT_WORDS * slot + 1) & 0xFFFFFFFFull;
        const double tiles = (double)(hs >> 32), light = (double)(hs & 0xFFFFFFFFull), heavy = (double)hh;
        if (tiles > 0) {
            gL = (long long)(light / tiles * 1.125 * (double)nAllTiles / (double)f->tiles_per_cta) + 56;
            gH = (long long)(heavy / tiles * 1.125 * (double)nAllTiles) + 8;
            const long long wave = (long long)f->sm_count * min_ctas;
            if (gL + gH < wave) gL = wave - gH;
        }
    }
    if (gH > nAllTiles) gH = nAllTiles;
    if (gL > nAllTiles) gL = nAllTiles;
    if (gH < 1) gH = 1;
    if (gL < 1) gL = 1;
    F.gridHeavy = (unsigned)gH;
    long long gR = gL + gH;
    if (M.use) gR = (long long)CE * ((gR + CE - 2) / (CE - 1));     // CE - 1 rasterizing CTAs + one clear CTA per group of CE (see k_raster)
    if (prof) CU(cudaEventRecord(f->prof_ev[2 * f->prof_n], st));
    // per-pixel texturing: the instantiation of the same shape with the frame's texture filter
    if (shape == 2) launch_raster<RasterSmall>(F, M, (unsigned)gR, st);
    else if (shape == 3) launch_raster<RasterWide>(F, M, (unsigned)gR, st);
    else launch_raster<RasterLarge>(F, M, (unsigned)gR, st);
    if ((rc = launch_check(f, "k_raster"))) return rc;
    if (prof) {
        CU(cudaEventRecord(f->prof_ev[2 * f->prof_n + 1], st));
        f->prof_n++;
    }
    return CRB_OK;
}

int run_tiled(crb_filler *f, Frame &F, cudaStream_t st, int slot = 0)
{
    int rc = run_prep(f, F, st, slot);
    return rc ? rc : run_raster(f, F, st, slot);
}

int run_atomic(crb_filler *f, Frame &F, cudaStream_t st)
{
    int rc;
    if (F.nViews != 1 || F.views) return fail(CRB_ERR_INVALID, "CRB_PATH_ATOMIC supports single-view renders only");
    if (!F.z || !F.color || !F.normals) return fail(CRB_ERR_STATE, "CRB_PATH_ATOMIC needs all three buffers");
    if (f->keybuf_pixels < F.slabPixels) {
        if (f->keybuf) cudaFree(f->keybuf);
        f->keybuf = nullptr;
        CU(cudaMalloc(&f->keybuf, (size_t)F.slabPixels * 8));
        f->keybuf_pixels = F.slabPixels;
        k_fill_u64<<<1184, NT, 0, st>>>(f->keybuf, F.slabPixels, KEY_EMPTY);
        if ((rc = launch_check(f, "k_fill_u64"))) return rc;
    }
    if (F.T > 0) {
        if ((rc = setup_smem_attr(f->device))) return rc;
        launch_setup(F, (unsigned)min((F.T + NT - 1) / NT, (long long)f->sm_count * CRB_SETUP_MIN_CTAS), st);
        if ((rc = launch_check(f, "k_setup"))) return rc;
        k_raster_atomic<<<(unsigned)((F.T * 32 + NT - 1) / NT), NT, 0, st>>>(F, f->keybuf);
        if ((rc = launch_check(f, "k_raster_atomic"))) return rc;
    }
    const unsigned gS = (unsigned)((F.slabPixels + NT - 1) / NT);
    switch (tex_mode(F)) {
    case TEX_NEAREST: k_shade_atomic<TEX_NEAREST><<<gS, NT, 0, st>>>(F, f->keybuf); break;
    case TEX_NEAREST | TEX_PERSP: k_shade_atomic<TEX_NEAREST | TEX_PERSP><<<gS, NT, 0, st>>>(F, f->keybuf); break;
    case TEX_BILINEAR: k_shade_atomic<TEX_BILINEAR><<<gS, NT, 0, st>>>(F, f->keybuf); break;
    case TEX_BILINEAR | TEX_PERSP: k_shade_atomic<TEX_BILINEAR | TEX_PERSP><<<gS, NT, 0, st>>>(F, f->keybuf); break;
    case TEX_TRILINEAR: k_shade_atomic<TEX_TRILINEAR><<<gS, NT, 0, st>>>(F, f->keybuf); break;
    case TEX_TRILINEAR | TEX_PERSP: k_shade_atomic<TEX_TRILINEAR | TEX_PERSP><<<gS, NT, 0, st>>>(F, f->keybuf); break;
    default: k_shade_atomic<TEX_NONE><<<gS, NT, 0, st>>>(F, f->keybuf);
    }
    return launch_check(f, "k_shade_atomic");
}

// CRB_DEFER_JOIN left rasterizer work in flight that the caller's stream does not know about: order `st` behind it.
int join_pending(crb_filler *f, cudaStream_t st)
{
    if (f->pending_join) {
        CU(cudaStreamWaitEvent(st, f->ev_raster[f->pending_join - 1], 0));
        f->pending_join = 0;
    }
    return CRB_OK;
}

int bind_ws_pointers(crb_filler *f, void *ws, size_t bytes, long long T, int views, long long pairCap, cudaStream_t st)
{
    if (views < 1) views = 1;
    if (views > 1024) return fail(CRB_ERR_INVALID, "max_views > 1024 (views per launch; crb_render_views chunks longer batches itself)");
    if (T < 0) return fail(CRB_ERR_INVALID, "max_triangles < 0");
    if (pairCap <= 0) pairCap = default_pair_cap(f, T, views);
    if (pairCap > 0xFFFFFFF0ll) return fail(CRB_ERR_INVALID, "pair capacity exceeds 32-bit list offsets");
    const WsLayout L = ws_layout(f, T, views, pairCap);
    if (!ws || bytes < L.bytes) return fail(CRB_ERR_INVALID, "workspace too small: %zu < %zu", bytes, L.bytes);
    if (reinterpret_cast<uintptr_t>(ws) & 255u) return fail(CRB_ERR_INVALID, "workspace must be 256-byte aligned");
    char *b = (char *)ws;
    f->ws = ws; f->ws_bytes = bytes;
    f->maxT = T; f->maxViews = views; f->pairCap = pairCap;
    f->shrec = (float4 *)(b + L.shrec); f->recE = (float4 *)(b + L.recE);
    f->alive = (unsigned short *)(b + L.alive);
    f->chunks = (unsigned *)(b + L.chunks);
    f->count = (unsigned *)(b + L.count); f->offset = (unsigned *)(b + L.offset); f->cursor = (unsigned *)(b + L.cursor);
    f->busy = (uint4 *)(b + L.busy); f->busyH = (uint4 *)(b + L.busyH); f->empty = (unsigned *)(b + L.empty);
    f->ls = (float4 *)(b + L.ls);
    f->wide = (uint4 *)(b + L.wide);
    f->wideCap = wide_capacity(T, views);
    f->total = (unsigned long long *)(b + L.total);
    f->stage_v = (float *)(b + L.sv); f->stage_c = (float *)(b + L.sc); f->stage_n = (float *)(b + L.sn);
    f->set_bytes = L.set_bytes;
    for (int k = 0; k < 2; ++k) {
        CU(cudaMemsetAsync(b + k * L.set_bytes + L.count, 0, L.offset - L.count, st));  // tile counts start at zero, k_alloc keeps them so
        CU(cudaMemsetAsync(b + k * L.set_bytes + L.total, 0, 64, st));
    }
    return CRB_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------------------
// The expensive, size-independent part of a filler -- two streams, five events and a mapped page-locked statistics block
// (cudaHostAlloc / cudaFreeHost alone cost milliseconds and synchronise the device) -- is recycled through a process-wide
// free list: the reference's only idiom is a NEW filler per frame (run.py:21), so crb_create / crb_destroy must be cheap.
// ------------------------------------------------------------------------------------------------------------
#include <mutex>
namespace {
struct Shell {
    int device;
    cudaStream_t s_prep, s_raster;
    cudaEvent_t ev_start, ev_fill[2], ev_raster[2];
    unsigned long long *hstats, *hstats_dev;
};
std::mutex g_shell_mu;
std::vector<Shell> g_shells;
constexpr size_t SHELL_POOL_MAX = 64;

int shell_acquire(int device, Shell *out)
{
    {
        std::lock_guard<std::mutex> lk(g_shell_mu);
        for (size_t i = 0; i < g_shells.size(); ++i)
            if (g_shells[i].device == device) {
                *out = g_shells[i];
                g_shells.erase(g_shells.begin() + (long)i);
                if (out->hstats) memset(out->hstats, 0, HSTAT_BYTES);
                return CRB_OK;
            }
    }
    Shell sh;
    memset(&sh, 0, sizeof(sh));
    sh.device = device;
    int lo = 0, hi = 0;
    CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    // equal priorities measured best (a high-priority front end costs the rasterizer more than it gains: -1 % on the headline,
    // with the 256-thread rasterizer and again with the 128-thread shapes)
    CU(cudaStreamCreateWithPriority(&sh.s_prep, cudaStreamNonBlocking, lo));
    CU(cudaStreamCreateWithPriority(&sh.s_raster, cudaStreamNonBlocking, lo));
    CU(cudaEventCreateWithFlags(&sh.ev_start, cudaEventDisableTiming));
    for (int k = 0; k < 2; ++k) {
        CU(cudaEventCreateWithFlags(&sh.ev_fill[k], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&sh.ev_raster[k], cudaEventDisableTiming));
    }
    void *hp = nullptr, *dp = nullptr;
    if (cudaHostAlloc(&hp, HSTAT_BYTES, cudaHostAllocMapped) == cudaSuccess && cudaHostGetDevicePointer(&dp, hp, 0) == cudaSuccess) {
        memset(hp, 0, HSTAT_BYTES);
        sh.hstats = (unsigned long long *)hp;
        sh.hstats_dev = (unsigned long long *)dp;
    } else {
        if (hp) cudaFreeHost(hp);
        cudaGetLastError();
    }
    *out = sh;
    return CRB_OK;
}

void shell_destroy(Shell &sh)
{
    if (sh.hstats) cudaFreeHost(sh.hstats);
    if (sh.s_prep) cudaStreamDestroy(sh.s_prep);
    if (sh.s_raster) cudaStreamDestroy(sh.s_raster);
    if (sh.ev_start) cudaEventDestroy(sh.ev_start);
    for (int k = 0; k < 2; ++k) {
        if (sh.ev_fill[k]) cudaEventDestroy(sh.ev_fill[k]);
        if (sh.ev_raster[k]) cudaEventDestroy(sh.ev_raster[k]);
    }
}

void shell_release(Shell &sh)
{
    {
        std::lock_guard<std::mutex> lk(g_shell_mu);
        if (g_shells.size() < SHELL_POOL_MAX) {
            g_shells.push_back(sh);
            return;
        }
    }
    shell_destroy(sh);
}
}  // namespace

// ------------------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------------------
extern "C" {

int crb_version(void) { return CRB_VERSION; }
const char *crb_last_error(void) { return g_err; }

int crb_device_count(int *count)
{
    if (!count) return fail(CRB_ERR_INVALID, "count is NULL");
    CU(cudaGetDeviceCount(count));
    return CRB_OK;
}

// ---- frame memory shared between the ranks of one node (SURVEY 8e: band-sharded fillers write their rows straight into the
// destination rank's frame over NVLink; the "gather" is the rasterizer's own stores) --------------------------------
static_assert(sizeof(cudaIpcMemHandle_t) == CRB_SHARED_HANDLE_BYTES, "handle size");

int crb_shared_alloc(int device, size_t bytes, void **ptr, unsigned char handle[CRB_SHARED_HANDLE_BYTES])
{
    if (!ptr || !handle || bytes == 0) return fail(CRB_ERR_INVALID, "NULL argument or zero size");
    CU(cudaSetDevice(device));
    CU(cudaMalloc(ptr, bytes));
    cudaIpcMemHandle_t h;
    const cudaError_t e = cudaIpcGetMemHandle(&h, *ptr);
    if (e != cudaSuccess) {
        cudaFree(*ptr);
        *ptr = nullptr;
        return fail(CRB_ERR_CUDA, "cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
    }
    memcpy(handle, &h, sizeof(h));
    return CRB_OK;
}

int crb_shared_open(int device, const unsigned char handle[CRB_SHARED_HANDLE_BYTES], void **ptr)
{
    if (!ptr || !handle) return fail(CRB_ERR_INVALID, "NULL argument");
    CU(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    CU(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return CRB_OK;
}

int crb_shared_close(int device, void *ptr)
{
    if (!ptr) return CRB_OK;
    CU(cudaSetDevice(device));
    CU(cudaIpcCloseMemHandle(ptr));
    return CRB_OK;
}

int crb_shared_free(int device, void *ptr)
{
    if (!ptr) return CRB_OK;
    CU(cudaSetDevice(device));
    CU(cudaFree(ptr));
    return CRB_OK;
}

int crb_projection(int h, int w, float fov, float z_near, float z_far, float proj[16])
{
    if (!proj) return fail(CRB_ERR_INVALID, "proj is NULL");
    ProjC P;
    int rc = host_projection(h, w, fov, z_near, z_far, &P);
    if (rc) return rc;
    memcpy(proj, P.p, sizeof(P.p));
    return CRB_OK;
}

int crb_create(int h, int w, float fov, float z_near, float z_far, int device, crb_filler **out)
{
    if (!out) return fail(CRB_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (h < 0 || w < 0 || h > MAX_DIM || w > MAX_DIM) return fail(CRB_ERR_INVALID, "resolution %dx%d outside [0,%d]", h, w, MAX_DIM);
    ProjC P;
    int rc = host_projection(h, w, fov, z_near, z_far, &P);
    if (rc) return rc;
    int ndev = 0;
    CU(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(CRB_ERR_INVALID, "device %d not in [0,%d)", device, ndev);
    crb_filler *f = new (std::nothrow) crb_filler();
    if (!f) return fail(CRB_ERR_INVALID, "out of host memory");
    memset(f, 0, sizeof(*f));
    f->h = h; f->w = w; f->device = device;
    f->row0 = 0; f->row1 = h;
    f->fov = fov; f->z_near = z_near; f->z_far = z_far;
    f->proj = P;
    {
        int sms = 0;
        CU(cudaSetDevice(device));
        CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
        f->sm_count = sms > 0 ? sms : 148;
        f->raster_ctas = 0;
        f->raster_shape = 0;
        f->use_tma = 1;
        f->split_heavy = 1;
        f->band_prepass = 1;
        f->chunk_pipeline = 1;
        f->wide_kernel = 1;
        {
            Shell sh;
            int src = shell_acquire(device, &sh);
            if (src) { delete f; return src; }
            f->s_prep = sh.s_prep; f->s_raster = sh.s_raster; f->ev_start = sh.ev_start;
            for (int k = 0; k < 2; ++k) { f->ev_fill[k] = sh.ev_fill[k]; f->ev_raster[k] = sh.ev_raster[k]; }
            f->hstats = sh.hstats; f->hstats_dev = sh.hstats_dev;
        }
        f->tiles_per_cta = 1;
        f->out_tma = 1;
#ifdef CRB_ABLATION     // development builds only (make variants): switches read from the environment
        if (const char *e = getenv("CRB_RASTER_CTAS")) f->raster_ctas = atoi(e);
        if (const char *e = getenv("CRB_TILES_PER_CTA")) { int k = atoi(e); if (k >= 1 && k <= 64) f->tiles_per_cta = k; }
        if (const char *e = getenv("CRB_NO_TMA")) f->use_tma = atoi(e) ? 0 : 1;
        if (const char *e = getenv("CRB_OUT_TMA")) f->out_tma = atoi(e);
        if (const char *e = getenv("CRB_DEBUG_SKIP")) f->dbg_flags = ((unsigned)atoi(e) & 31u) << 16;
#endif
    }
    *out = f;
    return CRB_OK;
}

void crb_destroy(crb_filler *f)
{
    if (!f) return;
    cudaSetDevice(f->device);
    if (f->own_buffers) { cudaFree(f->z); cudaFree(f->color); cudaFree(f->normals); }
    if (f->own_ws) cudaFree(f->ws);
    if (f->keybuf) cudaFree(f->keybuf);
    if (f->s_prep) cudaStreamSynchronize(f->s_prep);        // nothing of ours may still be running when the caller frees memory
    if (f->s_raster) cudaStreamSynchronize(f->s_raster);
    {
        Shell sh;
        memset(&sh, 0, sizeof(sh));
        sh.device = f->device;
        sh.s_prep = f->s_prep; sh.s_raster = f->s_raster; sh.ev_start = f->ev_start;
        for (int k = 0; k < 2; ++k) { sh.ev_fill[k] = f->ev_fill[k]; sh.ev_raster[k] = f->ev_raster[k]; }
        sh.hstats = f->hstats; sh.hstats_dev = f->hstats_dev;
        shell_release(sh);
    }
    if (f->shown_busy) cudaFree(f->shown_busy);
    if (f->tiles_copied) cudaFree(f->tiles_copied);
    if (f->prof_ev) {
        for (int i = 0; i < 2 * PROF_MAX; ++i) cudaEventDestroy(f->prof_ev[i]);
        delete[] f->prof_ev;
    }
    delete f;
}

int crb_get_size(const crb_filler *f, int *h, int *w)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    if (h) *h = f->h;
    if (w) *w = f->w;
    return CRB_OK;
}

int crb_get_projection(const crb_filler *f, float proj[16])
{
    if (check_filler(f) || !proj) return fail(CRB_ERR_INVALID, "NULL argument");
    memcpy(proj, f->proj.p, sizeof(f->proj.p));
    return CRB_OK;
}

int crb_set_band(crb_filler *f, int row0, int row1)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    if (row0 < 0 || row1 > f->h || row0 > row1) return fail(CRB_ERR_INVALID, "band [%d,%d) outside [0,%d)", row0, row1, f->h);
    if (f->ws || f->z) return fail(CRB_ERR_STATE, "set the band before binding buffers / workspace");
    f->row0 = row0; f->row1 = row1;
    return CRB_OK;
}

int crb_bind_buffers(crb_filler *f, float *z, float *color, float *normals)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    if (f->own_buffers) return fail(CRB_ERR_STATE, "buffers are library-owned");
    if ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(color) | reinterpret_cast<uintptr_t>(normals)) & 15u)
        return fail(CRB_ERR_INVALID, "buffers must be 16-byte aligned");
    f->z = z; f->color = color; f->normals = normals;
    return CRB_OK;
}

size_t crb_workspace_bytes(const crb_filler *f, int64_t max_triangles, int max_views, int64_t pair_capacity)
{
    if (!f || max_triangles < 0) return 0;
    if (max_views < 1) max_views = 1;
    if (pair_capacity <= 0) pair_capacity = default_pair_cap(f, max_triangles, max_views);
    return ws_layout(f, max_triangles, max_views, pair_capacity).bytes;
}

int crb_bind_workspace(crb_filler *f, void *workspace, size_t bytes, int64_t max_triangles, int max_views,
                       int64_t pair_capacity, void *stream)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    if (f->own_ws) return fail(CRB_ERR_STATE, "workspace is library-owned");
    CU(cudaSetDevice(f->device));
    { int jrc = join_pending(f, (cudaStream_t)stream); if (jrc) return jrc; }
    return bind_ws_pointers(f, workspace, bytes, max_triangles, max_views, pair_capacity, (cudaStream_t)stream);
}

int crb_alloc_owned(crb_filler *f, int64_t max_triangles, int max_views, int64_t pair_capacity)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    CU(cudaSetDevice(f->device));
    const size_t px = (size_t)(f->row1 - f->row0) * f->w;
    if (!f->z && !f->own_buffers) {
        CU(cudaMalloc(&f->z, (px ? px : 1) * 4));
        CU(cudaMalloc(&f->color, (px ? px : 1) * 12));
        CU(cudaMalloc(&f->normals, (px ? px : 1) * 12));
        f->own_buffers = true;
        int rc = crb_init_buffers(f, nullptr);
        if (rc) return rc;
    }
    if (f->own_ws) { cudaFree(f->ws); f->ws = nullptr; f->own_ws = false; }
    if (max_views < 1) max_views = 1;
    if (pair_capacity <= 0) pair_capacity = default_pair_cap(f, max_triangles, max_views);
    const size_t bytes = ws_layout(f, max_triangles, max_views, pair_capacity).bytes;
    void *ws = nullptr;
    CU(cudaMalloc(&ws, bytes));
    int rc = bind_ws_pointers(f, ws, bytes, max_triangles, max_views, pair_capacity, nullptr);
    if (rc) { cudaFree(ws); f->ws = nullptr; return rc; }
    f->own_ws = true;
    return CRB_OK;
}

int crb_device_buffers(const crb_filler *f, float **z, float **color, float **normals)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    if (z) *z = f->z;
    if (color) *color = f->color;
    if (normals) *normals = f->normals;
    return CRB_OK;
}

int crb_init_buffers(crb_filler *f, void *stream)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    if (!f->z || !f->color || !f->normals) return fail(CRB_ERR_STATE, "buffers not bound");
    CU(cudaSetDevice(f->device));
    { int jrc = join_pending(f, (cudaStream_t)stream); if (jrc) return jrc; }
    const long long px = (long long)(f->row1 - f->row0) * f->w;
    if (px == 0) return CRB_OK;
    k_init_buffers<<<1184, NT, 0, (cudaStream_t)stream>>>(f->z, f->color, f->normals, px);
    return launch_check(f, "k_init_buffers");
}

int crb_render(crb_filler *f, const float *v, const float *c, const float *n, int64_t T, unsigned flags, void *stream)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    if (!f->z || !f->color || !f->normals) return fail(CRB_ERR_STATE, "buffers not bound");
    { int trc = check_triangles(f, T, v, c, n); if (trc) return trc; }
    { int xrc = check_texture(f, flags); if (xrc) return xrc; }
    CU(cudaSetDevice(f->device));
    { int jrc = join_pending(f, (cudaStream_t)stream); if (jrc) return jrc; }
    if ((long long)(f->row1 - f->row0) * f->w == 0) return CRB_OK;
    Frame F;
    fill_frame(f, &F);
    F.T = T; F.nViews = 1; F.flags = flags & (CRB_CLEAR_FIRST | CRB_PATH_ATOMIC | CRB_TEX_FLAGS);
    F.v = v; F.c = c; F.n = n;
    F.z = f->z; F.color = f->color; F.normals = f->normals;
    return (flags & CRB_PATH_ATOMIC) ? run_atomic(f, F, (cudaStream_t)stream) : run_tiled(f, F, (cudaStream_t)stream);
}

int crb_pack_texture(const uint8_t *bgr, int th, int tw, uint32_t *out, void *stream)
{
    if (!bgr || !out || th < 1 || tw < 1 || (long long)th * tw >= (1ll << 31))
        return fail(CRB_ERR_INVALID, "crb_pack_texture: bad argument (NULL pointer, or th, tw < 1, or th * tw >= 2^31)");
    const long long texels = (long long)th * tw;
    k_pack_texture<<<(unsigned)min((texels + NT - 1) / NT, 4096ll), NT, 0, (cudaStream_t)stream>>>(bgr, texels, out);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(CRB_ERR_CUDA, "launch of k_pack_texture failed: %s", cudaGetErrorString(e));
    return CRB_OK;
}

int crb_bind_texture(crb_filler *f, const uint32_t *texels, int th, int tw)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    if (!texels) { f->tex = nullptr; f->tex_h = f->tex_w = f->tex_levels = 0; return CRB_OK; }
    if (th < 1 || tw < 1 || (long long)th * tw >= (1ll << 31))
        return fail(CRB_ERR_INVALID, "crb_bind_texture: th, tw must be >= 1 with th * tw < 2^31 (got %d x %d)", th, tw);
    if (reinterpret_cast<uintptr_t>(texels) & 3u) return fail(CRB_ERR_INVALID, "crb_bind_texture: texels must be 4-byte aligned");
    f->tex = texels; f->tex_h = th; f->tex_w = tw; f->tex_levels = 0;
    return CRB_OK;
}

int crb_mip_layout(int th, int tw, int *levels, long long *texels)
{
    if (th < 1 || tw < 1 || (long long)th * tw >= (1ll << 31))
        return fail(CRB_ERR_INVALID, "crb_mip_layout: th, tw must be >= 1 with th * tw < 2^31 (got %d x %d)", th, tw);
    int L = 1;
    long long n = (long long)th * tw;
    for (int h = th, w = tw; h > 1 || w > 1; ++L) {
        h = max(1, h >> 1); w = max(1, w >> 1);
        n += (long long)h * w;
    }
    if (n >= (1ll << 31)) return fail(CRB_ERR_INVALID, "crb_mip_layout: a %d x %d chain has %lld >= 2^31 texels", th, tw, n);
    if (levels) *levels = L;
    if (texels) *texels = n;
    return CRB_OK;
}

int crb_pack_texture_mips(const uint8_t *bgr, int th, int tw, uint32_t *out, void *stream)
{
    int L;
    { int rc = crb_mip_layout(th, tw, &L, nullptr); if (rc) return rc; }
    { int rc = crb_pack_texture(bgr, th, tw, out, stream); if (rc) return rc; }
    uint32_t *src = out;
    for (int l = 1, h = th, w = tw; l < L; ++l) {
        const int dh = max(1, h >> 1), dw = max(1, w >> 1);
        uint32_t *dst = src + (long long)h * w;
        const long long n = (long long)dh * dw;
        k_mip_level<<<(unsigned)min((n + NT - 1) / NT, 4096ll), NT, 0, (cudaStream_t)stream>>>(src, h, w, dst, dh, dw);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return fail(CRB_ERR_CUDA, "launch of k_mip_level failed: %s", cudaGetErrorString(e));
        src = dst; h = dh; w = dw;
    }
    return CRB_OK;
}

int crb_bind_texture_mips(crb_filler *f, const uint32_t *chain, int th, int tw)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    if (!chain) return crb_bind_texture(f, nullptr, 0, 0);
    int L;
    { int rc = crb_mip_layout(th, tw, &L, nullptr); if (rc) return rc; }
    { int rc = crb_bind_texture(f, chain, th, tw); if (rc) return rc; }
    f->tex_levels = L;
    return CRB_OK;
}

// H2D of the three [T,3,3] arrays into the filler's staging area.
static int upload_inputs(crb_filler *f, const float *v, const float *c, const float *n, int64_t T, cudaStream_t st)
{
    if (T > 0) {
        // Equally spaced host arrays (the rows of one [3,T,3,3] block, the usual case) go up as ONE strided copy: under a
        // pipeline the link is saturated by the read-back of earlier frames and every separate transfer queues behind it.
        const ptrdiff_t sp = (const char *)c - (const char *)v, dp = (char *)f->stage_c - (char *)f->stage_v;
        bool one = false;
        if (sp >= (ptrdiff_t)((size_t)T * 36) && sp == (const char *)n - (const char *)c && sp < (1ll << 30) &&
            dp == (char *)f->stage_n - (char *)f->stage_c && dp >= (ptrdiff_t)((size_t)T * 36) && dp < (1ll << 30)) {
            // (rows that lie in separate host allocations are refused by the runtime: three copies then)
            one = cudaMemcpy2DAsync(f->stage_v, (size_t)dp, v, (size_t)sp, (size_t)T * 36, 3, cudaMemcpyHostToDevice, st) == cudaSuccess;
            if (!one) cudaGetLastError();
        }
        if (!one) {
            CU(cudaMemcpyAsync(f->stage_v, v, (size_t)T * 36, cudaMemcpyHostToDevice, st));
            CU(cudaMemcpyAsync(f->stage_c, c, (size_t)T * 36, cudaMemcpyHostToDevice, st));
            CU(cudaMemcpyAsync(f->stage_n, n, (size_t)T * 36, cudaMemcpyHostToDevice, st));
        }
    }
    return CRB_OK;
}

// Pageable host arrays -> device (CRB_HOST_PAGEABLE).  cudaMemcpyAsync from pageable memory is staged by the driver on the
// calling thread at a few GB/s; a reference Model's NumPy arrays are pageable, and for the 10 M-triangle frame (1.08 GB) that
// copy was 75 ms of a 130 ms frame.  Here `nth` worker threads each own two 8 MB slots of a process-wide pinned ring: copy a
// chunk into a slot (memcpy), queue its cudaMemcpyAsync, go on with the next chunk while that one travels; a slot is reused
// once the event recorded behind its copy has fired.  All source bytes have been read when the function returns.
namespace {
constexpr size_t PG_CHUNK = 8u << 20;
constexpr int PG_MAX_THREADS = 8, PG_SLOTS_PER_THREAD = 2;
struct PageRing {
    std::mutex mu;                     // one pageable upload at a time
    int device = -1;
    char *base = nullptr;
    cudaEvent_t ev[PG_MAX_THREADS * PG_SLOTS_PER_THREAD] = {};
    bool used[PG_MAX_THREADS * PG_SLOTS_PER_THREAD] = {};     // the slot's last copy may still be in flight (its event tells)
};
PageRing g_ring;
struct PgSeg { char *dst; const char *src; size_t len; };
}  // namespace

static int upload_pageable(crb_filler *f, const float *v, const float *c, const float *n, int64_t T, cudaStream_t st)
{
    if (T <= 0) return CRB_OK;
    const size_t bytes = (size_t)T * 36;
    std::lock_guard<std::mutex> lock(g_ring.mu);
    if (!g_ring.base || g_ring.device != f->device) {      // first use, or a filler on another device (events belong to a device)
        if (g_ring.base) {
            cudaSetDevice(g_ring.device);
            for (int sl = 0; sl < PG_MAX_THREADS * PG_SLOTS_PER_THREAD; ++sl) {
                if (g_ring.used[sl]) cudaEventSynchronize(g_ring.ev[sl]);
                cudaEventDestroy(g_ring.ev[sl]);
                g_ring.ev[sl] = nullptr; g_ring.used[sl] = false;
            }
            cudaFreeHost(g_ring.base);
            g_ring.base = nullptr;
            CU(cudaSetDevice(f->device));
        }
        CU(cudaHostAlloc((void **)&g_ring.base, PG_CHUNK * PG_MAX_THREADS * PG_SLOTS_PER_THREAD, cudaHostAllocPortable));
        for (auto &e : g_ring.ev) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        g_ring.device = f->device;
    }
    std::vector<PgSeg> segs;
    const float *src[3] = {v, c, n};
    float *dst[3] = {f->stage_v, f->stage_c, f->stage_n};
    for (int a = 0; a < 3; ++a)
        for (size_t o = 0; o < bytes; o += PG_CHUNK)
            segs.push_back({(char *)dst[a] + o, (const char *)src[a] + o, bytes - o < PG_CHUNK ? bytes - o : PG_CHUNK});
    unsigned hw = std::thread::hardware_concurrency();
    int nth = (int)(hw ? hw / 2 : 4);
    nth = nth < 1 ? 1 : (nth > PG_MAX_THREADS ? PG_MAX_THREADS : nth);
    if ((size_t)nth > segs.size()) nth = (int)segs.size();
    std::atomic<int> err{0};
    auto work = [&](int t) {
        if (cudaSetDevice(f->device) != cudaSuccess) { err = 1; return; }
        int k = 0;
        for (size_t i = (size_t)t; i < segs.size(); i += (size_t)nth, ++k) {
            const int sl = t * PG_SLOTS_PER_THREAD + (k % PG_SLOTS_PER_THREAD);
            if (g_ring.used[sl] && cudaEventSynchronize(g_ring.ev[sl]) != cudaSuccess) { err = 1; return; }
            char *slot = g_ring.base + (size_t)sl * PG_CHUNK;
            memcpy(slot, segs[i].src, segs[i].len);
            if (cudaMemcpyAsync(segs[i].dst, slot, segs[i].len, cudaMemcpyHostToDevice, st) != cudaSuccess ||
                cudaEventRecord(g_ring.ev[sl], st) != cudaSuccess) { err = 1; return; }
            g_ring.used[sl] = true;
        }
    };
    if (nth == 1) work(0);
    else {
        std::vector<std::thread> team;
        for (int t = 1; t < nth; ++t) team.emplace_back(work, t);
        work(0);
        for (auto &th : team) th.join();
    }
    if (err) { cudaGetLastError(); return fail(CRB_ERR_CUDA, "staged upload of pageable host arrays failed"); }
    return CRB_OK;     // (copies still in flight keep their slots: the next call waits on the slot's event before it reuses one)
}

// Development aid (CRB_TRACE=1 in the environment): CUDA events at the stage boundaries of crb_render_host, dumped as
// microseconds since the first one by crb_trace_dump -- the only timeline tool on a box without nsys.
namespace {
struct TraceRec { cudaEvent_t e[4]; const void *who; };
std::vector<TraceRec> g_trace;
const bool g_trace_on = getenv("CRB_TRACE") && atoi(getenv("CRB_TRACE"));
inline void trace_mark(TraceRec *r, int k, cudaStream_t st)
{
    if (!r) return;
    cudaEventCreate(&r->e[k]);
    cudaEventRecord(r->e[k], st);
}
}  // namespace

static int render_host_once(crb_filler *f, const float *v, const float *c, const float *n, int64_t T, unsigned flags,
                            unsigned download_mask, float *z_out, float *color_out, float *normals_out, void *stream)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    { int trc = check_triangles(f, T, v, c, n); if (trc) return trc; }
    { int xrc = check_texture(f, flags); if (xrc) return xrc; }
    CU(cudaSetDevice(f->device));
    { int jrc = join_pending(f, (cudaStream_t)stream); if (jrc) return jrc; }
    cudaStream_t st = (cudaStream_t)stream;
    TraceRec trec{}, *tr = (g_trace_on && g_trace.size() < 4096) ? &trec : nullptr;
    trec.who = f;
    trace_mark(tr, 0, st);
    { int urc = (flags & CRB_HOST_PAGEABLE) ? upload_pageable(f, v, c, n, T, st) : upload_inputs(f, v, c, n, T, st); if (urc) return urc; }
    const bool sync_upload = (flags & CRB_SYNC_UPLOAD) && (flags & CRB_NO_SYNC) && !(flags & CRB_HOST_PAGEABLE) && T > 0;
    if (sync_upload) CU(cudaEventRecord(f->ev_start, st));      // (ev_start: free between crb_render_views calls)
    trace_mark(tr, 1, st);
    int rc = crb_render(f, f->stage_v, f->stage_c, f->stage_n, T, flags & ~(CRB_HOST_PAGEABLE | CRB_SYNC_UPLOAD), stream);
    if (rc) return rc;
    trace_mark(tr, 2, st);
    const bool sparse = (flags & CRB_DL_SPARSE) && (flags & CRB_CLEAR_FIRST) && !(flags & CRB_PATH_ATOMIC);
    float *hp[3] = {(download_mask & CRB_BUF_Z) ? z_out : nullptr, (download_mask & CRB_BUF_COLOR) ? color_out : nullptr,
                    (download_mask & CRB_BUF_NORMALS) ? normals_out : nullptr};
    bool mapped = sparse;
    for (int k = 0; k < 3 && mapped; ++k) {     // the host arrays must be pinned + device-visible for the tile copies
        if (!hp[k]) continue;
        if (f->map_host[k] != hp[k]) {
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, hp[k]) != cudaSuccess || at.type != cudaMemoryTypeHost || !at.devicePointer) {
                cudaGetLastError();
                mapped = false;
                break;
            }
            f->map_host[k] = hp[k];
            f->map_dev[k] = at.devicePointer;
        }
        hp[k] = (float *)f->map_dev[k];
    }
    if (sparse && !mapped) return fail(CRB_ERR_INVALID, "CRB_DL_SPARSE needs pinned (cudaHostAlloc / cudaHostRegister'ed, mapped) output arrays");
    if (sparse) {
        Frame F;
        fill_frame(f, &F);
        F.z = f->z; F.color = f->color; F.normals = f->normals;
        if (f->shown_tiles != F.nTiles) {
            if (f->shown_busy) cudaFree(f->shown_busy);
            f->shown_busy = nullptr;
            CU(cudaMalloc(&f->shown_busy, 4 * (size_t)(F.nTiles > 0 ? F.nTiles : 1)));
            CU(cudaMemsetAsync(f->shown_busy, 0, 4 * (size_t)(F.nTiles > 0 ? F.nTiles : 1), st));
            f->shown_tiles = F.nTiles;
        }
        if (!f->tiles_copied) {
            CU(cudaMalloc(&f->tiles_copied, 8));
            CU(cudaMemsetAsync(f->tiles_copied, 0, 8, st));
        }
        if (F.nTiles > 0) {
            const int want = READBACK_CTAS;
            k_readback<<<(unsigned)(F.nTiles < want ? F.nTiles : want), NT, 0, st>>>(F, f->shown_busy, hp[0], hp[1], hp[2], f->tiles_copied);
            if ((rc = launch_check(f, "k_readback"))) return rc;
        }
    } else {
        rc = crb_download(f, download_mask, z_out, color_out, normals_out, stream);
        if (rc) return rc;
    }
    trace_mark(tr, 3, st);
    if (tr) g_trace.push_back(trec);
    if (!(flags & CRB_NO_SYNC)) CU(cudaStreamSynchronize(st));
    else if (sync_upload) CU(cudaEventSynchronize(f->ev_start));      // the inputs have left host memory; the frame is still in flight
    return CRB_OK;
}

int crb_host_register(void *ptr, size_t bytes)
{
    if (!ptr || !bytes) return fail(CRB_ERR_INVALID, "NULL argument or zero size");
    const cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(CRB_ERR_CUDA, "cudaHostRegister failed: %s", cudaGetErrorString(e));
    }
    return CRB_OK;
}

int crb_host_unregister(void *ptr)
{
    if (!ptr) return CRB_OK;
    const cudaError_t e = cudaHostUnregister(ptr);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(CRB_ERR_CUDA, "cudaHostUnregister failed: %s", cudaGetErrorString(e));
    }
    return CRB_OK;
}

int crb_trace_dump(const char *path)
{
    if (!path) return fail(CRB_ERR_INVALID, "NULL path");
    FILE *fp = fopen(path, "w");
    if (!fp) return fail(CRB_ERR_INVALID, "cannot open %s", path);
    CU(cudaDeviceSynchronize());
    for (size_t i = 0; i < g_trace.size(); ++i) {
        float ms[4] = {0, 0, 0, 0};
        for (int k = 0; k < 4; ++k) cudaEventElapsedTime(&ms[k], g_trace[0].e[0], g_trace[i].e[k]);
        fprintf(fp, "%zu %p %.1f %.1f %.1f %.1f\n", i, g_trace[i].who, ms[0] * 1e3, ms[1] * 1e3, ms[2] * 1e3, ms[3] * 1e3);
    }
    fclose(fp);
    for (auto &r : g_trace) for (int k = 0; k < 4; ++k) cudaEventDestroy(r.e[k]);
    g_trace.clear();
    return CRB_OK;
}

int crb_render_host(crb_filler *f, const float *v, const float *c, const float *n, int64_t T, unsigned flags,
                    unsigned download_mask, float *z_out, float *color_out, float *normals_out, void *stream)
{
    for (int attempt = 0;; ++attempt) {
        int rc = render_host_once(f, v, c, n, T, flags, download_mask, z_out, color_out, normals_out, stream);
        if (rc || (flags & CRB_NO_SYNC) || (flags & CRB_PATH_ATOMIC)) return rc;   // asynchronous callers check crb_status themselves
        // the call is synchronous: a frame the pair list could not hold must not pass silently
        int64_t need = 0, cap = 0;
        rc = crb_status(f, &need, &cap, stream);
        if (rc != CRB_ERR_OVERFLOW) return rc;
        if (!f->own_ws || attempt >= 3) return rc;          // caller-owned workspace: report, the caller re-binds a larger one
        const long long maxT = f->maxT;
        const int maxViews = f->maxViews;
        rc = crb_alloc_owned(f, maxT, maxViews, need + need / 4 + 1024);   // library-owned: grow and draw the frame again
        if (rc) return rc;
    }
}

int crb_render_views(crb_filler *f, const float *v, const float *c, const float *n, int64_t T, const float *views,
                     int n_views, float *z_out, float *color_out, float *normals_out, uint8_t *color_u8_out,
                     unsigned flags, const float light[3], void *stream)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    if (n_views < 0) return fail(CRB_ERR_INVALID, "negative size");
    { int trc = check_triangles(f, T, v, c, n); if (trc) return trc; }
    if (n_views > 0 && !views && n_views != 1) return fail(CRB_ERR_INVALID, "views is NULL (allowed for one untransformed view only)");
    if (flags & CRB_PATH_ATOMIC) return fail(CRB_ERR_INVALID, "CRB_PATH_ATOMIC supports single-view renders only");
    if ((flags & CRB_GURO) && !light) return fail(CRB_ERR_INVALID, "CRB_GURO needs a light direction");
    { int xrc = check_texture(f, flags); if (xrc) return xrc; }
    if ((reinterpret_cast<uintptr_t>(z_out) | reinterpret_cast<uintptr_t>(color_out) | reinterpret_cast<uintptr_t>(normals_out)) & 15u)
        return fail(CRB_ERR_INVALID, "output slabs must be 16-byte aligned");
    if (f->u8x_n && color_u8_out) return fail(CRB_ERR_INVALID, "color_u8_out must be NULL while a row exchange is set (crb_set_u8_exchange)");
    if (f->u8x_n && f->u8x_n * f->u8x_rows != f->row1 - f->row0) return fail(CRB_ERR_STATE, "row exchange bands do not cover the filler's rows");
    CU(cudaSetDevice(f->device));
    const long long slab = (long long)(f->row1 - f->row0) * f->w;
    if (slab == 0) return CRB_OK;
    // Launches of maxViews views each.  With more than one launch, launch i+1's setup / binning kernels run on a second
    // stream beside launch i's rasterizer (two workspace sets): the memory-bound front end hides behind the issue-bound
    // rasterizer.  Rasterizer launches themselves stay serialised (they would only share the SMs).
    cudaStream_t user = (cudaStream_t)stream;
    const int launches = (n_views + f->maxViews - 1) / f->maxViews;
    const bool defer = (flags & CRB_DEFER_JOIN) != 0;
    const bool pipe = f->chunk_pipeline && (launches > 1 || defer) && launches > 0;
    if (!pipe) {
        int rc = join_pending(f, user);
        if (rc) return rc;
    } else {
        // everything the caller queued so far (inputs produced, earlier results consumed) comes first
        CU(cudaEventRecord(f->ev_start, user));
        CU(cudaStreamWaitEvent(f->s_prep, f->ev_start, 0));
        CU(cudaStreamWaitEvent(f->s_raster, f->ev_start, 0));
    }
    int i = 0, last_set = 0;
    for (int v0 = 0; v0 < n_views; v0 += f->maxViews, ++i) {
        const int set = pipe ? (int)(f->launch_seq++ & 1u) : 0;
        Frame F;
        fill_frame(f, &F, set);
        F.T = T; F.nViews = (n_views - v0 < f->maxViews) ? n_views - v0 : f->maxViews;
        F.flags = (flags & (CRB_GURO | CRB_TEX_FLAGS)) | CRB_CLEAR_FIRST;
        F.v = v; F.c = c; F.n = n;
        F.views = views ? views + (size_t)v0 * 16 : nullptr;
        F.z = z_out ? z_out + (size_t)v0 * slab : nullptr;
        F.color = color_out ? color_out + (size_t)v0 * slab * 3 : nullptr;
        F.normals = normals_out ? normals_out + (size_t)v0 * slab * 3 : nullptr;
        F.color_u8 = color_u8_out ? color_u8_out + (size_t)v0 * slab * 3 : nullptr;
        if (f->u8x_n) {      // row exchange: the uint8 image leaves through the receive buffers of the row bands
            F.u8xN = f->u8x_n; F.u8xRows = f->u8x_rows;
            for (int d = 0; d < f->u8x_n; ++d) F.u8x[d] = f->u8x[d] + (size_t)v0 * f->u8x_rows * f->w * 3;
            F.color_u8 = F.u8x[0];
        }
        if (light) { F.light[0] = light[0]; F.light[1] = light[1]; F.light[2] = light[2]; }
        int rc;
        if (!pipe) {
            rc = run_tiled(f, F, user, i);
            if (rc) return rc;
            continue;
        }
        if (f->set_used[set]) CU(cudaStreamWaitEvent(f->s_prep, f->ev_raster[set], 0));   // the set's previous frame has been rasterized
        if ((rc = run_prep(f, F, f->s_prep, i))) return rc;
        CU(cudaEventRecord(f->ev_fill[set], f->s_prep));
        CU(cudaStreamWaitEvent(f->s_raster, f->ev_fill[set], 0));
        if ((rc = run_raster(f, F, f->s_raster, i))) return rc;
        CU(cudaEventRecord(f->ev_raster[set], f->s_raster));
        f->set_used[set] = 1;
        last_set = set;
    }
    if (pipe) {
        f->pending_join = 1 + last_set;
        if (!defer) return join_pending(f, user);
    }
    return CRB_OK;
}

int crb_set_u8_exchange(crb_filler *f, int n_bands, int rows_per_band, void *const *band_base)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    if (n_bands == 0) { f->u8x_n = 0; return CRB_OK; }
    if (n_bands < 0 || n_bands > CRB_MAX_EXCHANGE || rows_per_band <= 0 || !band_base) return fail(CRB_ERR_INVALID, "bad row exchange");
    if ((long long)n_bands * rows_per_band != f->row1 - f->row0) return fail(CRB_ERR_INVALID, "n_bands * rows_per_band must equal the filler's rows");
    for (int d = 0; d < n_bands; ++d)
        if (!band_base[d] || (reinterpret_cast<uintptr_t>(band_base[d]) & 15u)) return fail(CRB_ERR_INVALID, "band_base must be non-NULL and 16-byte aligned");
    for (int d = 0; d < n_bands; ++d) f->u8x[d] = static_cast<unsigned char *>(band_base[d]);
    f->u8x_n = n_bands; f->u8x_rows = rows_per_band;
    return CRB_OK;
}

int crb_join(crb_filler *f, void *stream)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    CU(cudaSetDevice(f->device));
    return join_pending(f, (cudaStream_t)stream);
}

int crb_render_image_host(crb_filler *f, const float *v, const float *c, const float *n, int64_t T, unsigned flags,
                          const float light[3], uint8_t *image_dev, uint8_t *image_host, uint64_t status_pinned[4], void *stream)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    { int trc = check_triangles(f, T, v, c, n); if (trc) return trc; }
    if (!image_dev || !image_host) return fail(CRB_ERR_INVALID, "NULL image buffer");
    { int xrc = check_texture(f, flags); if (xrc) return xrc; }
    CU(cudaSetDevice(f->device));
    cudaStream_t st = (cudaStream_t)stream;
    { int jrc = join_pending(f, st); if (jrc) return jrc; }
    int rc = upload_inputs(f, v, c, n, T, st);
    if (rc) return rc;
    // one untransformed view, no float32 output: the rasterizer writes the flipped uint8 image itself
    rc = crb_render_views(f, f->stage_v, f->stage_c, f->stage_n, T, nullptr, 1, nullptr, nullptr, nullptr, image_dev,
                          flags & (CRB_GURO | CRB_TEX_FLAGS), light, stream);
    if (rc) return rc;
    const size_t bytes = (size_t)(f->row1 - f->row0) * f->w * 3;
    if (bytes) CU(cudaMemcpyAsync(image_host, image_dev, bytes, cudaMemcpyDeviceToHost, st));
    if (status_pinned) {
        rc = crb_status_async(f, status_pinned, stream);
        if (rc) return rc;
    }
    if (!(flags & CRB_NO_SYNC)) CU(cudaStreamSynchronize(st));
    return CRB_OK;
}

int crb_transform_view(crb_filler *f, const float *v, const float *n, int64_t T, const float *view, float *v_out,
                       float *n_out, void *stream)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    if (T < 0 || !view || (T > 0 && (!v || !n || !v_out || !n_out))) return fail(CRB_ERR_INVALID, "bad argument");
    CU(cudaSetDevice(f->device));
    if (T == 0) return CRB_OK;
    k_transform_view<<<(unsigned)((T * 3 + NT - 1) / NT), NT, 0, (cudaStream_t)stream>>>(v, n, T * 3, view, v_out, n_out);
    return launch_check(f, "k_transform_view");
}

int crb_guro(crb_filler *f, const float light[3], void *stream)
{
    if (check_filler(f) || !light) return fail(CRB_ERR_INVALID, "NULL argument");
    if (!f->color || !f->normals) return fail(CRB_ERR_STATE, "buffers not bound");
    CU(cudaSetDevice(f->device));
    { int jrc = join_pending(f, (cudaStream_t)stream); if (jrc) return jrc; }
    const long long px = (long long)(f->row1 - f->row0) * f->w;
    if (px == 0) return CRB_OK;
    k_guro<<<1184, NT, 0, (cudaStream_t)stream>>>(f->color, f->normals, px, light[0], light[1], light[2]);
    return launch_check(f, "k_guro");
}

int crb_color_u8_flipped(crb_filler *f, uint8_t *out_u8, void *stream)
{
    if (check_filler(f) || !out_u8) return fail(CRB_ERR_INVALID, "NULL argument");
    if (!f->color) return fail(CRB_ERR_STATE, "buffers not bound");
    CU(cudaSetDevice(f->device));
    { int jrc = join_pending(f, (cudaStream_t)stream); if (jrc) return jrc; }
    if ((long long)(f->row1 - f->row0) * f->w == 0) return CRB_OK;
    k_color_u8_flipped<<<1184, NT, 0, (cudaStream_t)stream>>>(f->color, out_u8, f->row1 - f->row0, f->w);
    return launch_check(f, "k_color_u8_flipped");
}

int crb_download(crb_filler *f, unsigned mask, float *z_host, float *color_host, float *normals_host, void *stream)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    if (!f->z || !f->color || !f->normals) return fail(CRB_ERR_STATE, "buffers not bound");
    CU(cudaSetDevice(f->device));
    { int jrc = join_pending(f, (cudaStream_t)stream); if (jrc) return jrc; }
    const size_t px = (size_t)(f->row1 - f->row0) * f->w;
    cudaStream_t st = (cudaStream_t)stream;
    if (px == 0) return CRB_OK;
    if ((mask & CRB_BUF_Z) && z_host) CU(cudaMemcpyAsync(z_host, f->z, px * 4, cudaMemcpyDeviceToHost, st));
    if ((mask & CRB_BUF_COLOR) && color_host) CU(cudaMemcpyAsync(color_host, f->color, px * 12, cudaMemcpyDeviceToHost, st));
    if ((mask & CRB_BUF_NORMALS) && normals_host) CU(cudaMemcpyAsync(normals_host, f->normals, px * 12, cudaMemcpyDeviceToHost, st));
    return CRB_OK;
}

int crb_upload(crb_filler *f, unsigned mask, const float *z_host, const float *color_host, const float *normals_host,
               void *stream)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    if (!f->z || !f->color || !f->normals) return fail(CRB_ERR_STATE, "buffers not bound");
    CU(cudaSetDevice(f->device));
    { int jrc = join_pending(f, (cudaStream_t)stream); if (jrc) return jrc; }
    const size_t px = (size_t)(f->row1 - f->row0) * f->w;
    cudaStream_t st = (cudaStream_t)stream;
    if (px == 0) return CRB_OK;
    if ((mask & CRB_BUF_Z) && z_host) CU(cudaMemcpyAsync(f->z, z_host, px * 4, cudaMemcpyHostToDevice, st));
    if ((mask & CRB_BUF_COLOR) && color_host) CU(cudaMemcpyAsync(f->color, color_host, px * 12, cudaMemcpyHostToDevice, st));
    if ((mask & CRB_BUF_NORMALS) && normals_host) CU(cudaMemcpyAsync(f->normals, normals_host, px * 12, cudaMemcpyHostToDevice, st));
    return CRB_OK;
}

int crb_status(crb_filler *f, int64_t *pairs_needed, int64_t *pair_capacity, void *stream)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    if (!f->ws) return fail(CRB_ERR_STATE, "workspace not bound");
    CU(cudaSetDevice(f->device));
    { int jrc = join_pending(f, (cudaStream_t)stream); if (jrc) return jrc; }
    unsigned long long t[2] = {0, 0}, u[2] = {0, 0};
    unsigned long long *total1 = reinterpret_cast<unsigned long long *>(reinterpret_cast<char *>(f->total) + f->set_bytes);
    CU(cudaMemcpyAsync(t, f->total, 16, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CU(cudaMemcpyAsync(u, total1, 16, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    if (u[0] > t[0]) t[0] = u[0];
    if (u[1] > t[1]) t[1] = u[1];
    if (pair_capacity) *pair_capacity = f->pairCap;
    if (t[1] > (unsigned long long)f->pairCap) {
        if (pairs_needed) *pairs_needed = (int64_t)t[1];
        CU(cudaMemsetAsync(f->total + 1, 0, 8, (cudaStream_t)stream));
        CU(cudaMemsetAsync(total1 + 1, 0, 8, (cudaStream_t)stream));
        return fail(CRB_ERR_OVERFLOW, "frame needs %llu (triangle,tile) pairs, workspace holds %lld; frame not drawn", t[1],
                    f->pairCap);
    }
    if (pairs_needed) *pairs_needed = (int64_t)t[0];
    return CRB_OK;
}

int64_t crb_pair_capacity(const crb_filler *f) { return (f && f->ws) ? (int64_t)f->pairCap : 0; }

int crb_status_async(crb_filler *f, uint64_t pinned[4], void *stream)
{
    if (check_filler(f) || !pinned) return fail(CRB_ERR_INVALID, "NULL argument");
    if (!f->ws) return fail(CRB_ERR_STATE, "workspace not bound");
    CU(cudaSetDevice(f->device));
    { int jrc = join_pending(f, (cudaStream_t)stream); if (jrc) return jrc; }
    unsigned long long *total1 = reinterpret_cast<unsigned long long *>(reinterpret_cast<char *>(f->total) + f->set_bytes);
    CU(cudaMemcpyAsync(pinned, f->total, 16, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CU(cudaMemcpyAsync(pinned + 2, total1, 16, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return CRB_OK;
}

int crb_set_option(crb_filler *f, int option, int value)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    switch (option) {
    case CRB_OPT_CHUNK_PIPELINE: f->chunk_pipeline = value ? 1 : 0; return CRB_OK;
    case CRB_OPT_TMA: f->use_tma = value ? 1 : 0; return CRB_OK;
    case CRB_OPT_TMA_ROWS: f->out_tma = (value == 2) ? 2 : (value ? 1 : 0); return CRB_OK;
    case CRB_OPT_RASTER_CTAS: f->raster_ctas = value > 0 ? value : 0; return CRB_OK;
    case CRB_OPT_SPLIT_HEAVY: f->split_heavy = value ? 1 : 0; return CRB_OK;
    case CRB_OPT_WIDE_KERNEL: f->wide_kernel = value ? 1 : 0; return CRB_OK;
    case CRB_OPT_BAND_PREPASS: f->band_prepass = value ? 1 : 0; return CRB_OK;
    case CRB_OPT_RASTER_SHAPE: f->raster_shape = (value >= 1 && value <= 3) ? value : 0; return CRB_OK;
    default: return fail(CRB_ERR_INVALID, "unknown option %d", option);
    }
}

int crb_sync(crb_filler *f, void *stream)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    CU(cudaSetDevice(f->device));
    { int jrc = join_pending(f, (cudaStream_t)stream); if (jrc) return jrc; }
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    return CRB_OK;
}

int crb_readback_stats(crb_filler *f, int64_t *tiles_copied, int reset, void *stream)
{
    if (check_filler(f) || !tiles_copied) return fail(CRB_ERR_INVALID, "NULL argument");
    CU(cudaSetDevice(f->device));
    { int jrc = join_pending(f, (cudaStream_t)stream); if (jrc) return jrc; }
    unsigned long long n = 0;
    if (f->tiles_copied) {
        CU(cudaMemcpyAsync(&n, f->tiles_copied, 8, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
        CU(cudaStreamSynchronize((cudaStream_t)stream));
        if (reset) CU(cudaMemsetAsync(f->tiles_copied, 0, 8, (cudaStream_t)stream));
    }
    *tiles_copied = (int64_t)((n + TH - 1) / TH);   // the device counter counts 32-pixel tile rows
    return CRB_OK;
}

int crb_readback_reset(crb_filler *f, void *stream)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    CU(cudaSetDevice(f->device));
    { int jrc = join_pending(f, (cudaStream_t)stream); if (jrc) return jrc; }
    if (f->shown_busy) CU(cudaMemsetAsync(f->shown_busy, 0, 4 * (size_t)(f->shown_tiles > 0 ? f->shown_tiles : 1), (cudaStream_t)stream));
    return CRB_OK;
}

int64_t crb_launch_count(const crb_filler *f) { return f ? f->launches : 0; }

int crb_phase_cycles(uint64_t out[16], int reset)
{
    if (!out) return fail(CRB_ERR_INVALID, "out is NULL");
    unsigned long long h[16];
    CU(cudaMemcpyFromSymbol(h, g_phase, sizeof(h)));
    for (int i = 0; i < 16; ++i) out[i] = h[i];
    if (reset) {
        memset(h, 0, sizeof(h));
        CU(cudaMemcpyToSymbol(g_phase, h, sizeof(h)));
    }
    return CRB_OK;
}

int crb_selftest_fdiv(int device, uint64_t samples, unsigned seed, uint64_t *mismatches, uint32_t first_bad[2])
{
    if (!mismatches) return fail(CRB_ERR_INVALID, "mismatches is NULL");
    CU(cudaSetDevice(device));
    unsigned long long *d_out = nullptr, h_out[3] = {0, 0, 0};
    CU(cudaMalloc(&d_out, sizeof(h_out)));
    CU(cudaMemset(d_out, 0, sizeof(h_out)));
    k_selftest_fdiv<<<148 * 8, NT>>>(samples, seed, d_out);
    cudaError_t e = cudaMemcpy(h_out, d_out, sizeof(h_out), cudaMemcpyDeviceToHost);
    cudaFree(d_out);
    if (e != cudaSuccess) return fail(CRB_ERR_CUDA, "k_selftest_fdiv failed: %s", cudaGetErrorString(e));
    *mismatches = h_out[0];
    if (first_bad) { first_bad[0] = (uint32_t)h_out[1]; first_bad[1] = (uint32_t)h_out[2]; }
    return CRB_OK;
}

int crb_profile(crb_filler *f, int enable)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    CU(cudaSetDevice(f->device));
    if (enable && !f->prof_ev) {
        f->prof_ev = new (std::nothrow) cudaEvent_t[2 * PROF_MAX];
        if (!f->prof_ev) return fail(CRB_ERR_INVALID, "out of host memory");
        for (int i = 0; i < 2 * PROF_MAX; ++i) CU(cudaEventCreate(&f->prof_ev[i]));
    }
    f->prof_on = enable != 0;
    f->prof_n = 0;
    return CRB_OK;
}

int crb_profile_read(crb_filler *f, int *launches, double *total_ms)
{
    if (check_filler(f)) return CRB_ERR_INVALID;
    CU(cudaSetDevice(f->device));
    double tot = 0.0;
    for (int i = 0; i < f->prof_n; ++i) {
        float ms = 0.f;
        CU(cudaEventSynchronize(f->prof_ev[2 * i + 1]));
        CU(cudaEventElapsedTime(&ms, f->prof_ev[2 * i], f->prof_ev[2 * i + 1]));
        tot += ms;
    }
    if (launches) *launches = f->prof_n;
    if (total_ms) *total_ms = tot;
    f->prof_n = 0;
    return CRB_OK;
}

}  // extern "C"
