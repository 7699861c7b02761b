/*
 * crender_b200.h -- C ABI of libcrender_b200.so: the B200 (sm_100a) implementation of the Version C
 * rendering hot path of oKatanaaa/Cython3DModelRenderer.
 *
 * The reference has no C ABI: its boundary is the Cython extension type `AdvancedPixelBufferFiller`
 * (crender/cy/pixel_buffer_filler/advanced_pixel_buffer_filler.pyx:20), whose `cdef` methods are not
 * callable from outside.  Each entry point below names the reference lines it stands in for ("pyx" is that
 * file).  A maintainer binds these from the .pyx (`cdef extern from "crender_b200.h"`) or, as this repo
 * does, from Python with ctypes -- both are shown in INTEGRATION.md.
 *
 * Conventions
 *   - plain C types only; every pointer is either a HOST pointer or a DEVICE pointer as documented;
 *   - every function returns CRB_OK (0) or a negative CRB_ERR_* code; crb_last_error() gives the text of the
 *     calling thread's most recent failure;
 *   - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream).  Calls are asynchronous
 *     with respect to the host unless the name says "host" or "sync";
 *   - a filler is not re-entrant (same as the reference object), different fillers are independent.
 *   - triangle arrays are [T,3,3] float32, C-contiguous: (triangle, vertex, xyz | BGR | normal xyz), exactly
 *     `model._vertices_by_triangles/_colors_by_triangles/_normals_by_triangles` (pyx:94-96).
 *   - output buffers: z [h,w] f32, colour [h,w,3] f32, normals [h,w,3] f32, row-major, y-up (pyx:65-67).
 */
#ifndef CRENDER_B200_H
#define CRENDER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define CRB_VERSION 100

#define CRB_OK 0
#define CRB_ERR_INVALID (-1)   /* bad argument (NULL, negative size, unsupported resolution) */
#define CRB_ERR_CUDA (-2)      /* a CUDA runtime call or kernel launch failed                */
#define CRB_ERR_ZERODIV (-3)   /* where the reference raises ZeroDivisionError (pyx:59,84,86) */
#define CRB_ERR_STATE (-4)     /* buffers / workspace not bound                              */
#define CRB_ERR_OVERFLOW (-5)  /* triangle-tile pair list exceeded the workspace; see crb_status */

/* crb_render* flags */
#define CRB_CLEAR_FIRST 1u     /* fresh-filler semantics (z=1e6, colour=normals=0, pyx:65-67) fused into the frame */
#define CRB_PATH_ATOMIC 2u     /* differential path: per-triangle raster with global 64-bit atomicMin + deferred
                                  shading (no binning).  Same results; kept for cross-checking the tiled path. */
#define CRB_GURO 4u            /* N1: fuse GuroIllumination (guro_illumination.py:20-27) into the shading pass   */
#define CRB_NO_SYNC 8u         /* crb_render_host only: return once the work is queued; crb_sync() before reading
                                  the host outputs or reusing the host inputs (frame pipelining over several fillers) */

#define CRB_DEFER_JOIN 32u     /* crb_render_views only: return without ordering `stream` behind the rasterizer (which runs on an
                                  internal stream), so that the NEXT batch's setup / binning kernels overlap this batch's
                                  rasterization.  The outputs may only be used on `stream` after crb_join(); every other
                                  entry point that touches the filler joins by itself. */
#define CRB_HOST_PAGEABLE 64u   /* crb_render_host only: v / c / n are ordinary (pageable) host memory, e.g. the NumPy arrays of a
                                  reference Model.  They are staged through a process-wide ring of pinned buffers by a few worker
                                  threads, chunk by chunk, each chunk's host-to-device copy in flight while the next is being
                                  staged; the arrays have been read completely when the call returns (CRB_NO_SYNC included).
                                  Without the flag the three pointers must be page-locked (they are handed to cudaMemcpyAsync). */
#define CRB_SYNC_UPLOAD 128u    /* crb_render_host + CRB_NO_SYNC: return once v / c / n have left host memory (the caller may then reuse
                                  or free them), with the frame itself still in flight.  For page-locked inputs that are not a
                                  private staging copy -- e.g. a Model's own arrays registered with crb_host_register */
#define CRB_DL_SPARSE 16u      /* crb_render_host + CRB_CLEAR_FIRST only: sparse read-back.  The caller promises that the host
                                  output arrays still hold what the previous CRB_DL_SPARSE call of this filler left in them
                                  (fresh-filler values -- z 1e6, colour 0, normals 0 -- before the first call, or after
                                  crb_readback_reset).  Only tiles that are busy now or were busy in that previous frame are
                                  then copied (at the granularity of 32-pixel tile rows), by a kernel writing into the pinned + mapped host arrays; the arrays end up
                                  bit-identical to a full download.  The arrays must come from cudaHostAlloc /
                                  cudaHostRegister (e.g. torch pin_memory). */
#define CRB_TEXTURE 1024u      /* per-pixel texturing (every render entry point; an extension, the reference textures vertices only):
                                  `c` holds texture coordinates (u, v, ignored) per corner instead of colours.  They are interpolated
                                  like colours, and the winning fragment's colour is the texel of the texture bound with
                                  crb_bind_texture at row = clip(int32((1 - v) * th), 0, th-1), col = clip(int32(u * tw), 0, tw-1)
                                  (float32, int32 as x86-64 converts: NaN and out-of-range give INT32_MIN) -- model.py:147-150's
                                  rule -- as float BGR, lit afterwards by CRB_GURO.  Without a bound texture: CRB_ERR_STATE. */
#define CRB_TEX_PERSPECTIVE 2048u  /* with CRB_TEXTURE: perspective-correct coordinates.  Per corner w = 1 / z, z the camera-space depth
                                      the projection divides by (after the view transform for crb_render_views); (u*w, v*w, w) are
                                      interpolated like colours to (U, V, W), then u = U / W, v = V / W (float32, correctly rounded; no
                                      clipping: z == 0 or corners on both sides of the camera plane give whatever IEEE gives, and the
                                      texel rule then maps NaN to row / column 0). */
#define CRB_TEX_BILINEAR 4096u     /* with CRB_TEXTURE: bilinear filtering instead of the nearest texel (DESIGN 2).  sx = u*tw - 0.5,
                                      sy = (1 - v)*th - 0.5, each clamped with fmin(fmax(s, -1), tw or th) (NaN -> -1); the four
                                      texels around (sx, sy), indices clamped to the texture, blended in float32 as
                                      (t00*gx + t01*fx)*gy + (t10*gx + t11*fx)*fy with fx = sx - floor(sx), gx = 1 - fx (same for y).
                                      At texel centres this is the nearest texel.  Either mode bit without CRB_TEXTURE: CRB_ERR_INVALID
                                      on every render entry point. */
#define CRB_TEX_TRILINEAR 8192u    /* with CRB_TEXTURE: trilinear mip filtering (DESIGN 2) of the chain bound with crb_bind_texture_mips
                                      (L levels, level 0 the texture).  Per pixel, from the record's corners and denominators:
                                      gx = ((y2-y1)/l03, (y0-y2)/l13, (y1-y0)/l23), gy = ((x1-x2)/l03, (x2-x0)/l13, (x0-x1)/l23), and for
                                      corner values a_k, a_x = (a0*gx0 + a1*gx1) + a2*gx2 (a_y alike).  Affine: ux = u_x, vx = v_x, ...;
                                      with CRB_TEX_PERSPECTIVE ux = (U_x - u*W_x) / W, vx = (V_x - v*W_x) / W (y alike).  p = ux*tw,
                                      q = vx*th, r = uy*tw, s = vy*th (level 0's size); r2 = fmax(p*p + q*q, r*r + s*s);
                                      L2 = (k - 1) + (2f - 1) with r2 = f * 2^k, f in [0.5, 1) (frexp; r2 = 0: -inf, +inf: +inf, NaN: NaN);
                                      lc = fmin(fmax(0.5*L2, 0), L-1) (NaN -> 0); l0 = floor(lc), fr = lc - l0, l1 = min(l0 + 1, L-1);
                                      colour = c0*(1 - fr) + c1*fr with c0, c1 CRB_TEX_BILINEAR's blend on levels l0, l1.  float32, one
                                      rounding per operation.  Where lc == 0 this is CRB_TEX_BILINEAR bit for bit.  Without CRB_TEXTURE,
                                      or with CRB_TEX_BILINEAR: CRB_ERR_INVALID; no chain bound: CRB_ERR_STATE. */

/* which-buffer masks for crb_download / crb_render_host */
#define CRB_BUF_Z 1u
#define CRB_BUF_COLOR 2u
#define CRB_BUF_NORMALS 4u
#define CRB_BUF_ALL 7u

typedef struct crb_filler crb_filler;

/* ---- library ------------------------------------------------------------------------------------------- */
int crb_version(void);
const char *crb_last_error(void);
int crb_device_count(int *count);

/* ---- frame memory shared between the ranks (processes) of one node -------------------------------------------------
 * No reference counterpart (the reference is one process).  SURVEY 8e / BASELINE north_star: screen-row bands over N GPUs
 * "with a final gather over NVLink".  Here the gather is the rasterizer's own stores: the destination rank allocates the
 * whole frame (crb_shared_alloc: cudaMalloc + CUDA IPC handle), sends the 64-byte handle to the other ranks through
 * whatever channel it has (torch.distributed in the Python host), they map it (crb_shared_open: peer access over
 * NVLink / NVSwitch is enabled by the mapping) and bind the rows of their band inside it as their output buffers
 * (crb_bind_buffers with pointers into the mapped frame).  After a stream synchronisation on every rank and a barrier the
 * destination rank holds the complete frame.  crb_shared_close unmaps (other ranks), crb_shared_free releases (owner). */
#define CRB_SHARED_HANDLE_BYTES 64
int crb_shared_alloc(int device, size_t bytes, void **ptr, unsigned char handle[CRB_SHARED_HANDLE_BYTES]);
int crb_shared_open(int device, const unsigned char handle[CRB_SHARED_HANDLE_BYTES], void **ptr);
int crb_shared_close(int device, void *ptr);
int crb_shared_free(int device, void *ptr);

/* Page-locks (cudaHostRegister) / releases an existing host allocation, so that crb_render_host can read it in place instead of
 * through a staging copy -- for callers that render the same host arrays again and again (a reference Model's
 * _vertices_by_triangles / _colors_by_triangles / _normals_by_triangles are ordinary NumPy memory).  crb_host_register fails
 * with CRB_ERR_CUDA for memory that cannot be registered (already registered, read-only mappings, ...): fall back to copying. */
int crb_host_register(void *ptr, size_t bytes);
int crb_host_unregister(void *ptr);

/* ---- constructor pieces: pyx:39-77 (__cinit__) and pyx:83-90 (_init_projection_matrix) ------------------- */

/* Host only.  proj = row-major 4x4 float32 identical to the reference's proj_mat:
 * f = (float)(1/tan(fov/2/180*pi)) in double on the float fov, a = (float)(h/w), q = z_far/(z_far-z_near),
 * P00 = f/a, P11 = f, P22 = q, P23 = 1, P32 = -z_near*q (all float).  CRB_ERR_ZERODIV where the reference
 * raises (w == 0, h == 0, z_far == z_near). */
int crb_projection(int h, int w, float fov, float z_near, float z_far, float proj[16]);

/* Creates a filler bound to CUDA device `device`.  No buffers are allocated yet: bind caller-owned device
 * memory with crb_bind_buffers / crb_bind_workspace, or let the library own them (crb_alloc_owned). */
int crb_create(int h, int w, float fov, float z_near, float z_far, int device, crb_filler **out);
void crb_destroy(crb_filler *f);

int crb_get_size(const crb_filler *f, int *h, int *w);        /* pyx:80-81 get_size */
int crb_get_projection(const crb_filler *f, float proj[16]);  /* the cdef attribute proj_mat */

/* Restrict the filler to rows [row0,row1) of the h x w image (screen-tile-band sharding, SURVEY 8e).  The bound
 * buffers then hold only those rows ([row1-row0, w, ...]).  Per-pixel arithmetic does not depend on the band, so the
 * concatenated bands equal the full-frame result bit for bit.  Default band is [0,h). */
int crb_set_band(crb_filler *f, int row0, int row1);

/* ---- memory ------------------------------------------------------------------------------------------------ */

/* Device pointers to caller-owned buffers (e.g. torch tensors): z [rows,w], color [rows,w,3], normals [rows,w,3]. */
int crb_bind_buffers(crb_filler *f, float *z, float *color, float *normals);

/* Scratch needed to render up to max_triangles triangles in up to max_views simultaneous views with room for
 * pair_capacity (triangle,tile) pairs (0 = default heuristic). */
size_t crb_workspace_bytes(const crb_filler *f, int64_t max_triangles, int max_views, int64_t pair_capacity);
int crb_bind_workspace(crb_filler *f, void *workspace, size_t bytes, int64_t max_triangles, int max_views,
                       int64_t pair_capacity, void *stream);

/* Library-owned alternative (cudaMalloc): output buffers + workspace.  For hosts without a device allocator. */
int crb_alloc_owned(crb_filler *f, int64_t max_triangles, int max_views, int64_t pair_capacity);
int crb_device_buffers(const crb_filler *f, float **z, float **color, float **normals);

/* z = 1e6, colour = 0, normals = 0 (pyx:65-67), asynchronous on `stream`. */
int crb_init_buffers(crb_filler *f, void *stream);

/* ---- per-pixel texturing (CRB_TEXTURE) ----------------------------------------------------------------------- */

/* bgr: DEVICE uint8 [th,tw,3] (cv2.imread's layout) -> out: DEVICE uint32 [th,tw], texel = B | G << 8 | R << 16, on the current
 * device, asynchronous on `stream`.  CRB_ERR_INVALID for NULL pointers, th or tw < 1, or th * tw >= 2^31. */
int crb_pack_texture(const uint8_t *bgr, int th, int tw, uint32_t *out, void *stream);

/* Binds packed texels (crb_pack_texture; caller-owned DEVICE memory that must outlive the renders using it, like
 * crb_bind_buffers) as the texture of CRB_TEXTURE renders.  texels = NULL unbinds.  CRB_ERR_INVALID for th or tw < 1,
 * th * tw >= 2^31, or a pointer that is not 4-byte aligned. */
int crb_bind_texture(crb_filler *f, const uint32_t *texels, int th, int tw);

/* Mip chain of a [th,tw] texture for CRB_TEX_TRILINEAR: L = 1 + floor(log2(max(th, tw))) levels, level k+1 of size
 * max(1, th_k >> 1) x max(1, tw_k >> 1), row-major and back to back from level 0 (the packed texture).  Writes L to *levels and
 * the chain's total texels to *texels (either may be NULL).  CRB_ERR_INVALID for th or tw < 1, th * tw >= 2^31, or a chain of
 * 2^31 texels or more. */
int crb_mip_layout(int th, int tw, int *levels, long long *texels);

/* bgr: DEVICE uint8 [th,tw,3] -> out: DEVICE uint32, the whole chain (crb_mip_layout's texels): level 0 as crb_pack_texture
 * packs it, then each level from the one before, per channel (t[r0][c0] + t[r0][c1] + t[r1][c0] + t[r1][c1] + 2) >> 2 in integers,
 * r0 = min(2r, th_k - 1), r1 = min(2r + 1, th_k - 1), columns alike.  Current device, asynchronous on `stream`.
 * CRB_ERR_INVALID as crb_mip_layout, or for NULL pointers. */
int crb_pack_texture_mips(const uint8_t *bgr, int th, int tw, uint32_t *out, void *stream);

/* Binds a chain (crb_pack_texture_mips; caller-owned DEVICE memory, 4-byte aligned) of a [th,tw] texture.  It serves
 * CRB_TEX_TRILINEAR, and nearest and bilinear renders from level 0, exactly as crb_bind_texture of level 0 would.  chain = NULL
 * unbinds; crb_bind_texture replaces it.  CRB_ERR_INVALID as crb_mip_layout. */
int crb_bind_texture_mips(crb_filler *f, const uint32_t *chain, int th, int tw);

/* ---- render_model: pyx:92-104 -> project (pyx:106-130) + cull/bbox/raster/z-test/writes (pyx:177-244) ------- */

/* v, c, n: DEVICE pointers, [T,3,3] f32.  Composites into the bound buffers exactly like successive
 * render_model calls on one reference filler (n_threads=1 order: min depth wins, equal depth -> higher triangle
 * index / later call wins).  Inputs are never written. */
int crb_render(crb_filler *f, const float *v, const float *c, const float *n, int64_t T, unsigned flags,
               void *stream);

/* Same, all pointers HOST memory (pinned recommended): H2D of the three arrays, render, D2H of the buffers named in
 * `download_mask` (CRB_BUF_*; NULL pointers allowed for buffers not requested), then a stream synchronize (unless
 * CRB_NO_SYNC).  This is the call that replaces the body of render_model for a host-resident caller.  In the synchronous
 * form a frame that did not fit the (triangle,tile) pair list never passes silently: a library-owned workspace
 * (crb_alloc_owned) is grown and the frame drawn again, a caller-owned one returns CRB_ERR_OVERFLOW with the buffers
 * untouched (see crb_status).  With CRB_NO_SYNC the caller checks crb_status itself. */
int crb_render_host(crb_filler *f, const float *v, const float *c, const float *n, int64_t T, unsigned flags,
                    unsigned download_mask, float *z_out, float *color_out, float *normals_out, void *stream);

/* Tuning switches (defaults: all on).  CRB_OPT_CHUNK_PIPELINE: crb_render_views runs the setup / binning kernels of launch
 * i+1 on an internal stream beside the rasterizer of launch i (two workspace sets).  CRB_OPT_TMA: tensor-map (TMA box) stores
 * for the fused clear and the shaded rows where the layout allows.  Results do not depend on any of them. */
#define CRB_OPT_CHUNK_PIPELINE 1
#define CRB_OPT_TMA 2
#define CRB_OPT_TMA_ROWS 3   /* shaded colour / normal rows of busy tiles as TMA boxes (1), staged 16-byte vector stores (0) or
                                12-byte stores straight from registers (2).  Only builds with -DCRB_LARGE_OUT_STAGE have a rasterizer
                                shape that stages rows (24 KB of shared memory per CTA); the shipped shapes store from registers
                                whatever this says -- smaller CTAs without the staging measured 12-15 % faster (DESIGN 6c) */
#define CRB_OPT_BAND_PREPASS 4   /* band-sharded fillers (crb_set_band): a streaming pre-pass lists the 256-triangle chunks that
                                    can reach the band, and the setup / binning kernels visit only those (1, default) */
#define CRB_OPT_RASTER_CTAS 5    /* > 0: fixed k_raster grid (a grid smaller than the busy tiles makes every CTA walk several tiles);
                                    0 (default): sized from the busy-tile count the previous launch reported */
#define CRB_OPT_SPLIT_HEAVY 6    /* single-view launches cut tiles with many triangles into four row bands rasterized by
                                    different CTAs (default 1) */
#define CRB_OPT_WIDE_KERNEL 7    /* triangles that span more than 12 tiles are listed by k_fill and scattered by a kernel of their own
                                    (k_fill_wide, a warp per triangle; launched only while frames contain such triangles); 0: k_fill
                                    scatters them itself (default 1) */
#define CRB_OPT_RASTER_SHAPE 8   /* CTA shape of the tile rasterizer: 0 (default) chosen per launch from the busy tiles and the triangles
                                    per busy tile the previous launch posted; 1: 128 threads, 96 triangles staged per pass, 8 CTAs per
                                    SM (tiles of many triangles, frames of a few waves); 2: 128 threads, 24 triangles per pass, 12 CTAs
                                    per SM (large batches of ordinary tiles); 3: 256 threads, 128 triangles per pass, 6 CTAs per SM
                                    (frames that do not fill the machine once).  Results do not depend on it. */
int crb_set_option(crb_filler *f, int option, int value);

/* Orders `stream` behind rasterizer work left in flight by CRB_DEFER_JOIN (no host synchronisation). */
int crb_join(crb_filler *f, void *stream);

/* Waits for everything queued on `stream` (pairs with CRB_NO_SYNC). */
int crb_sync(crb_filler *f, void *stream);

/* Batched views (config C5; the reference has no camera stage -- views are made by mutating the model on the host,
 * crender/cy/data_structures/model.py:238-256).  views: DEVICE [n_views,16] f32 = {R (9, row-major), p (3), q (3), pad}:
 *   v' = R (v - p) + q,   n' = R n     evaluated per component as ((r0*d0 + r1*d1) + r2*d2) + q, float32, no FMA.
 * Each view is rendered with fresh-filler semantics into its own slab of z_out [n_views,rows,w], color_out /
 * normals_out [n_views,rows,w,3] (DEVICE).  Any of the three output pointers may be NULL (buffer not wanted).
 * color_u8_out, if not NULL, additionally receives run.py:26's output stage on device: [n_views,rows,w,3] uint8,
 * rows flipped (image[::-1]) and truncated like .astype('uint8'). */
int crb_render_views(crb_filler *f, const float *v, const float *c, const float *n, int64_t T, const float *views /* NULL: one untransformed view */,
                     int n_views, float *z_out, float *color_out, float *normals_out, uint8_t *color_u8_out,
                     unsigned flags, const float light[3], void *stream);

/* Row exchange of the uint8 image (SURVEY 8e, config C5 "view-sharded ... with NCCL gather"; no reference counterpart --
 * run.py is one process).  While n_bands > 0, crb_render_views writes run.py:26's flipped uint8 image of its views NOT into
 * color_u8_out (pass NULL there) but row band by row band into other GPUs' memory, from inside the rasterizer: image row r
 * (after the flip) of the call's view k belongs to band d = r / rows_per_band and is stored at
 *     band_base[d] + ((k * rows_per_band + (r - d * rows_per_band)) * w + x) * 3
 * band_base[d] = a device address valid on THIS GPU (own memory, or rank d's receive buffer mapped with crb_shared_open:
 * the stores then cross NVLink / NVSwitch while the frame is rasterized) -- the collective is the kernel's own stores,
 * no staging copy and no NCCL call; a stream synchronisation on every rank plus a barrier completes the exchange.
 * n_bands = 1 with rows_per_band = rows is a gather of whole images into one rank; n_bands = N the all-to-all after which
 * rank d holds rows [d*rows_per_band, (d+1)*rows_per_band) of every rank's views.  Requirements: 1 <= n_bands <=
 * CRB_MAX_EXCHANGE, n_bands * rows_per_band == rows of the filler, every band_base 16-byte aligned.  n_bands = 0 ends it. */
#define CRB_MAX_EXCHANGE 8
int crb_set_u8_exchange(crb_filler *f, int n_bands, int rows_per_band, void *const *band_base);

/* run.py's product from host arrays in one call (SURVEY 8f N3): H2D of the three arrays, a fresh-filler frame whose only
 * output is run.py:26's `image[::-1].astype('uint8')` -- written by the rasterizer itself, lit like GuroIllumination
 * (renderer.py:48, guro_illumination.py:20-27) when flags has CRB_GURO and `light` is the normalised, negated direction --
 * and D2H of those (rows x w x 3) bytes into `image_host`.  `image_dev`: device scratch of the same size.  `status_pinned`
 * (optional): crb_status_async behind the frame.  CRB_NO_SYNC returns without waiting.  The filler's float32 buffers are
 * not touched. */
int crb_render_image_host(crb_filler *f, const float *v, const float *c, const float *n, int64_t T, unsigned flags,
                          const float light[3], uint8_t *image_dev, uint8_t *image_host, uint64_t status_pinned[4], void *stream);

/* Writes the camera-space arrays a view produces ([T,3,3] each, DEVICE) -- what the reference would be handed as
 * model._vertices_by_triangles / _normals_by_triangles for that view.  Used to feed the oracle in parity tests. */
int crb_transform_view(crb_filler *f, const float *v, const float *n, int64_t T, const float *view /* device [16] */,
                       float *v_out, float *n_out, void *stream);

/* ---- N1 / N3 post-passes on the bound buffers --------------------------------------------------------------- */

/* GuroIllumination.draw_illumination on the bound colour/normal buffers, in place (guro_illumination.py:20-27).
 * light = the already negated + normalised direction the reference keeps in self.light_direction. */
int crb_guro(crb_filler *f, const float light[3], void *stream);

/* run.py:26: image[::-1].astype('uint8') of the colour buffer -> out_u8 DEVICE [rows,w,3]. */
int crb_color_u8_flipped(crb_filler *f, uint8_t *out_u8, void *stream);

/* ---- transfers and status ------------------------------------------------------------------------------------- */
int crb_download(crb_filler *f, unsigned mask, float *z_host, float *color_host, float *normals_host, void *stream);
int crb_upload(crb_filler *f, unsigned mask, const float *z_host, const float *color_host, const float *normals_host,
               void *stream);

/* Synchronises `stream` and reports the last frame's bookkeeping: pairs_needed = (triangle,tile) pairs the frame
 * produced; if it exceeded the workspace's pair capacity the frame was NOT drawn (buffers untouched) and the return
 * value is CRB_ERR_OVERFLOW -- re-bind a workspace with pair_capacity >= pairs_needed and render again. */
int crb_status(crb_filler *f, int64_t *pairs_needed, int64_t *pair_capacity, void *stream);

/* Pair capacity of the bound workspace (0 if none); no device interaction. */
int64_t crb_pair_capacity(const crb_filler *f);

/* The same without blocking: queues the copy of the four status words of the two workspace sets (pairs of the last frame,
 * largest overflowing demand; per set) into `pinned` (page-locked host memory) behind the work already on `stream`.
 * Once the stream has passed that point the caller tests max(pinned[1], pinned[3]) > pair capacity itself (frame skipped:
 * call crb_status for the report and the reset) -- pipelined callers poll an event instead of paying a synchronous round
 * trip per frame. */
int crb_status_async(crb_filler *f, uint64_t pinned[4], void *stream);

/* Sparse read-back bookkeeping.  The read-back works on 32-pixel tile rows (896 bytes for all three buffers): a row crosses
 * PCIe when it holds something now or held something in the frame the host arrays show.  *tiles_copied = rows copied since the
 * last reset of the counter / 32, rounded up (tile equivalents of 32x32 pixels, 28 KB); crb_readback_reset declares that the
 * caller's host arrays hold fresh-filler values again. */
int crb_readback_stats(crb_filler *f, int64_t *tiles_copied, int reset, void *stream);
int crb_readback_reset(crb_filler *f, void *stream);

/* Number of kernel launches issued by this filler since creation (bench.py's gpu_launches). */
int64_t crb_launch_count(const crb_filler *f);

/* Self-test (GPU): the rasterizer replaces `x / d` for a per-triangle constant d by a correctly rounded quotient computed
 * from rcp.rn(d) and two FMA residual steps.  This checks that sequence against the division instruction on `samples`
 * pseudo-random + adversarial operand pairs; *mismatches must come back 0.  first_bad = bit patterns (a, d) of one
 * failing pair, if any. */
int crb_selftest_fdiv(int device, uint64_t samples, unsigned seed, uint64_t *mismatches, uint32_t first_bad[2]);

/* Measurement aid: while enabled, every launch of the dominant kernel (the tile rasterizer + shader, k_raster) is
 * bracketed by CUDA events on the launching stream.  crb_profile_read waits for them and returns how many launches
 * were timed since the last read and their summed device time.  Not usable inside CUDA-graph capture. */
int crb_profile(crb_filler *f, int enable);
int crb_profile_read(crb_filler *f, int *launches, double *total_ms);

/* Development aid: warp-cycles spent per phase of k_raster, accumulated on the current device since the last reset.
 * All zeros unless the library was built with -DCRB_PHASE_TIMING (the product build is not). */
int crb_phase_cycles(uint64_t out[16], int reset);

/* Development aid: with CRB_TRACE=1 in the environment crb_render_host brackets its stages (upload, render, read-back) with
 * CUDA events; this writes one line per call -- index, filler, four times in microseconds since the first call -- and
 * forgets them.  Writes an empty file otherwise. */
int crb_trace_dump(const char *path);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif

#ifdef __cplusplus
}
#endif
#endif /* CRENDER_B200_H */
