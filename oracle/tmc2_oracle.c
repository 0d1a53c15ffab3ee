/*
 * tmc2_oracle.c -- CPU oracle (plain C, one thread).  TEST INFRASTRUCTURE ONLY; see tmc2_oracle.h.
 *
 * Every function cites the reference lines (tmc2-rs, /root/reference/src/...) whose algorithm it
 * restates.  Semantics follow the reference's RELEASE build: integer arithmetic wraps (usize/u16),
 * asserts/unwraps/unimplemented!() become status codes instead of panics.
 *
 * Compile with -ffp-contract=off: the colour conversion must round every f64 operation on its own,
 * as rustc does (it never contracts mul+add into an FMA).
 */
#include "tmc2_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

typedef uint64_t usize; /* Rust usize on the reference's 64-bit targets */

/* ------------------------------------------------------------------------------------------------
 * A growing vector with Rust's Vec::push policy (amortised doubling, min cap 4) so that the CPU
 * baseline pays the same reallocation pattern as the reference's per-point pushes.
 * ---------------------------------------------------------------------------------------------- */
typedef struct vec {
  unsigned char* data;
  size_t len, cap, elem;
} vec;

static void vec_init(vec* v, size_t elem) { v->data = NULL; v->len = 0; v->cap = 0; v->elem = elem; }
static void vec_free(vec* v) { free(v->data); v->data = NULL; v->len = v->cap = 0; }
static int vec_reserve(vec* v, size_t extra) {
  size_t need = v->len + extra;
  if (need <= v->cap) return 0;
  size_t ncap = v->cap * 2;
  if (ncap < need) ncap = need;
  if (ncap < 4) ncap = 4;
  unsigned char* nd = (unsigned char*)realloc(v->data, ncap * v->elem);
  if (!nd) return -1;
  v->data = nd; v->cap = ncap;
  return 0;
}
static inline int vec_push(vec* v, const void* e) {
  if (v->len == v->cap && vec_reserve(v, 1)) return -1;
  memcpy(v->data + v->len * v->elem, e, v->elem);
  v->len++;
  return 0;
}
static int vec_extend(vec* dst, const vec* src) { /* Vec::extend(iter) */
  if (vec_reserve(dst, src->len)) return -1;
  if (src->len) memcpy(dst->data + dst->len * dst->elem, src->data, src->len * src->elem);
  dst->len += src->len;
  return 0;
}

/* PointSet3, codec.rs:20-36 */
typedef struct point_set3 {
  vec positions;           /* Vector3<u16> */
  vec colors;              /* Vector3<u8>  */
  vec colors16bit;         /* Vector3<u16> */
  vec point_patch_indexes; /* (usize, usize) */
  int with_colors;
} point_set3;

static void ps_init(point_set3* ps) {
  vec_init(&ps->positions, 6); vec_init(&ps->colors, 3); vec_init(&ps->colors16bit, 6);
  vec_init(&ps->point_patch_indexes, 16); ps->with_colors = 0;
}
static void ps_free(point_set3* ps) {
  vec_free(&ps->positions); vec_free(&ps->colors); vec_free(&ps->colors16bit); vec_free(&ps->point_patch_indexes);
}
/* codec.rs:45-53 add_point */
static inline size_t ps_add_point(point_set3* ps, const uint16_t pos[3]) {
  vec_push(&ps->positions, pos);
  if (ps->with_colors) {
    const uint8_t grey[3] = {127, 127, 127};
    const uint16_t zero[3] = {0, 0, 0};
    vec_push(&ps->colors, grey);
    vec_push(&ps->colors16bit, zero);
  }
  const usize pp[2] = {0, 0};
  vec_push(&ps->point_patch_indexes, pp);
  return ps->positions.len - 1;
}
/* codec.rs:61-70 append_point_set */
static void ps_append(point_set3* dst, const point_set3* src) {
  vec_extend(&dst->positions, &src->positions);
  vec_extend(&dst->colors, &src->colors);
  vec_extend(&dst->colors16bit, &src->colors16bit);
  vec_extend(&dst->point_patch_indexes, &src->point_patch_indexes);
}

/* ------------------------------------------------------------------------------------------------
 * Image access, decoder.rs:973-1020.  Strides are explicit (the reference assumes stride == width).
 * ---------------------------------------------------------------------------------------------- */
static inline int occ_get(const tmc2_gof* g, const tmc2_frame* f, usize u, usize v, uint8_t* out) {
  if (!(u < g->occ_width && v < g->occ_height)) return TMC2_ERR_INVALID_ARG; /* assert decoder.rs:974 */
  *out = f->occ[v * f->occ_stride + u];
  return TMC2_OK;
}
static inline uint16_t geo_get(const tmc2_frame* f, int map, usize x, usize y) { /* channel 0 */
  return f->geo[map][y * f->geo_stride + x];
}
static inline uint16_t attr_get(const tmc2_frame* f, int map, int channel, usize x, usize y) {
  if (channel == 0) return f->attr_y[map][y * f->attr_stride_y + x];          /* decoder.rs:976 */
  const uint16_t* pl = channel == 1 ? f->attr_u[map] : f->attr_v[map];
  return pl[(y / 2) * f->attr_stride_c + (x / 2)];                             /* decoder.rs:977 */
}

/* ------------------------------------------------------------------------------------------------
 * Patch helpers, decoder.rs:827-888.
 * ---------------------------------------------------------------------------------------------- */
/* decoder.rs:853-867 patch_to_canvas_helper.  usize arithmetic wraps exactly like the release build;
 * `size_scale` is 1 in REFERENCE mode (size_uv0 stays in blocks -- the reference's quirk) and
 * `resolution` in SPEC mode. */
static inline void patch_to_canvas_helper(const tmc2_patch* p, usize u, usize v, usize resolution, usize size_scale,
                                          usize* x, usize* y) {
  const usize u0 = (usize)p->u0 * resolution, v0 = (usize)p->v0 * resolution;
  const usize size_u0 = (usize)p->size_u0 * size_scale, size_v0 = (usize)p->size_v0 * size_scale;
  switch (p->patch_orientation) {
    case TMC2_ORIENT_DEFAULT: *x = u + u0; *y = v + v0; break;
    case TMC2_ORIENT_ROT90:   *x = size_v0 - 1 - v + u0; *y = u + v0; break;
    case TMC2_ORIENT_ROT180:  *x = size_u0 - 1 - u + u0; *y = size_v0 - 1 - v + v0; break;
    case TMC2_ORIENT_ROT270:  *x = v + u0; *y = size_u0 - 1 - u + v0; break;
    case TMC2_ORIENT_MIRROR:  *x = size_u0 - 1 - u + u0; *y = v + v0; break;
    case TMC2_ORIENT_MROT90:  *x = size_v0 - 1 - v + u0; *y = size_u0 - 1 - u + v0; break;
    case TMC2_ORIENT_MROT180: *x = u + u0; *y = size_v0 - 1 - v + v0; break;
    case TMC2_ORIENT_MROT270: *x = v + u0; *y = u + v0; break;
    case TMC2_ORIENT_SWAP:    *x = v + u0; *y = u + v0; break;
    default:                  *x = (usize)-1; *y = (usize)-1; break; /* FromPrimitive would not produce it */
  }
}

int orc_patch_to_canvas(const tmc2_patch* p, uint32_t occupancy_resolution, int orientation_mode, int is_block,
                        uint64_t u, uint64_t v, uint64_t canvas_stride, uint64_t canvas_height,
                        uint64_t* x, uint64_t* y) {
  /* decoder.rs:827-837 (block: resolution 1) and :840-850 (pixel: resolution = occupancy_resolution) */
  const usize res = is_block ? 1 : occupancy_resolution;
  const usize scale = (orientation_mode == TMC2_ORIENTATION_SPEC) ? res : 1;
  patch_to_canvas_helper(p, u, v, res, scale, x, y);
  if (!(*x < canvas_stride && *y < canvas_height)) return TMC2_ERR_PATCH_OUT_OF_CANVAS; /* assert :835/:848 */
  return TMC2_OK;
}

/* decoder.rs:881-888 generate_normal_coordinate */
static inline usize generate_normal_coordinate(const tmc2_patch* p, uint16_t depth) {
  const usize d = depth;
  if (p->projection_mode == 0) return d + (usize)p->d1;
  const usize m = (usize)p->d1 > d ? (usize)p->d1 : d; /* max(d1, depth) - depth */
  return m - d;
}
/* decoder.rs:871-878 generate_point (truncating `as u16` casts) */
void orc_patch_generate_point(const tmc2_patch* p, uint64_t u, uint64_t v, uint16_t depth, uint16_t out[3]) {
  out[0] = out[1] = out[2] = 0;
  out[p->normal_axis] = (uint16_t)generate_normal_coordinate(p, depth);
  out[p->tangent_axis] = (uint16_t)(u * (usize)p->lod_x + (usize)p->u1);
  out[p->bitangent_axis] = (uint16_t)(v * (usize)p->lod_y + (usize)p->v1);
}

/* ------------------------------------------------------------------------------------------------
 * Argument checks shared by the entry points: what the reference asserts or would panic on.
 * ---------------------------------------------------------------------------------------------- */
static int check_gof(const tmc2_gof* g, uint32_t frame_index) {
  if (!g || !g->frames || frame_index >= g->frame_count) return TMC2_ERR_INVALID_ARG;
  const tmc2_params* P = &g->params;
  if (P->occupancy_resolution == 0 || P->occupancy_precision == 0) return TMC2_ERR_INVALID_ARG;
  if (P->enable_size_quantization || P->multiple_streams || P->pbf_enabled || P->enhanced_occupancy_map ||
      P->point_local_reconstruction || P->single_map_pixel_interleaving || P->use_additional_points_patch)
    return TMC2_ERR_UNSUPPORTED; /* unimplemented!() codec.rs:285,303,314,399,402,454,494 */
  /* own spec: colour thresholds scale by 2^(bitdepth-8); samples are u16, so a deeper bit depth means nothing.  Checked
   * here rather than in color_smoothing so that frames without points are refused too. */
  if (P->color_smoothing && P->attribute_count && P->attribute_bitdepth > 16) return TMC2_ERR_INVALID_ARG;
  return TMC2_OK;
}

/* ------------------------------------------------------------------------------------------------
 * codec.rs:205-250 generate_block_to_patch_from_occupancy_map_video
 * ---------------------------------------------------------------------------------------------- */
int orc_generate_block_to_patch_from_occupancy_map_video(const tmc2_gof* g, uint32_t frame_index,
                                                         uint64_t* block_to_patch) {
  int st = check_gof(g, frame_index);
  if (st) return st;
  const tmc2_frame* f = &g->frames[frame_index];
  const usize res = g->params.occupancy_resolution, prec = g->params.occupancy_precision;
  const int mode = g->params.orientation_mode;
  const usize bw = g->width / res, bh = g->height / res; /* codec.rs:212-213 */
  memset(block_to_patch, 0, (size_t)(bw * bh) * sizeof(uint64_t));
  for (usize pi = 0; pi < f->patch_count; ++pi) {            /* codec.rs:217 */
    const tmc2_patch* p = &f->patches[pi];
    for (usize v0 = 0; v0 < p->size_v0; ++v0) {              /* :218 */
      for (usize u0 = 0; u0 < p->size_u0; ++u0) {            /* :219 */
        usize bx, by;
        st = orc_patch_to_canvas(p, (uint32_t)res, mode, 1, u0, v0, bw, bh, &bx, &by); /* :220-225 */
        if (st) return st;
        const usize block_index = by * bw + bx;
        usize non_zero_pixel = 0;
        for (usize v1 = 0; v1 < res; ++v1) {                 /* :227 patch.occupancy_resolution */
          const usize v = v0 * res + v1;
          for (usize u1 = 0; u1 < res; ++u1) {               /* :229 */
            const usize u = u0 * res + u1;
            usize x, y;
            st = orc_patch_to_canvas(p, (uint32_t)res, mode, 0, u, v, g->width, g->height, &x, &y); /* :231-232 */
            if (st) return st;
            uint8_t o; /* left_top_in_frame is always (0,0) (context.rs:402 never set) */
            st = occ_get(g, f, x / prec, y / prec, &o);      /* :235-239 */
            if (st) return st;
            non_zero_pixel += o;
          }
        }
        if (non_zero_pixel > 0) block_to_patch[block_index] = pi + 1; /* :242-244 */
      }
    }
  }
  return TMC2_OK;
}

/* ------------------------------------------------------------------------------------------------
 * codec.rs:517-565 generate_points.  created[1] is always Some for map_count 2.
 * ---------------------------------------------------------------------------------------------- */
static inline void generate_points(const tmc2_gof* g, const tmc2_frame* f, const tmc2_patch* p, usize u, usize v,
                                   usize x, usize y, uint16_t point0[3], uint16_t point1[3]) {
  /* :534 depth = sample / 4: libavcodec hands out 10-bit containers for nominally 8-bit depth */
  orc_patch_generate_point(p, u, v, (uint16_t)(geo_get(f, 0, x, y) / 4), point0);
  const uint16_t d1 = (uint16_t)(geo_get(f, 1, x, y) / 4);   /* :548 */
  if (g->params.absolute_d1) {                               /* :549-550 */
    orc_patch_generate_point(p, u, v, d1, point1);
  } else {
    point1[0] = point0[0]; point1[1] = point0[1]; point1[2] = point0[2];
    if (p->projection_mode == 0) point1[p->normal_axis] = (uint16_t)(point1[p->normal_axis] + d1); /* :551-554 */
    else                         point1[p->normal_axis] = (uint16_t)(point1[p->normal_axis] - d1); /* :555-558 */
  }
}

/* ------------------------------------------------------------------------------------------------
 * codec.rs:661-687 convert_yuv10_to_rgb8.  Operation order and rounding exactly as written there.
 * ---------------------------------------------------------------------------------------------- */
static inline uint8_t clamp_u8(double x) {
  if (x < 0.) return 0;
  if (x > 255.) return 255;
  return (uint8_t)x;
}
void orc_convert_yuv10_to_rgb8(const uint16_t yuv[3], uint8_t rgb[3]) {
  const double offset = 512., scale = 1023.;
  const double y = (double)yuv[0], u = (double)yuv[1], v = (double)yuv[2];
  volatile double t; /* keep every product a separately rounded double, whatever the optimiser thinks */
  t = 1.57480 * (v - offset);            const double r = y + t;
  t = 0.18733 * (u - offset);            double gg = y - t;
  t = 0.46813 * (v - offset);            gg = gg - t;
  t = 1.85563 * (u - offset);            const double b = y + t;
  rgb[0] = clamp_u8(floor(r / scale * 255.));
  rgb[1] = clamp_u8(floor(gg / scale * 255.));
  rgb[2] = clamp_u8(floor(b / scale * 255.));
}

/* ------------------------------------------------------------------------------------------------
 * codec.rs:256-514 generate_point_cloud (with color_point_cloud :569-658 called at :502-511).
 * ---------------------------------------------------------------------------------------------- */
typedef struct gpc_result {
  point_set3 reconstruct;
  vec partition;       /* usize */
  vec point_to_pixel;  /* Vector3<usize> */
  uint8_t* occupancy_map;
} gpc_result;

static int generate_point_cloud(const tmc2_gof* g, uint32_t frame_index, const uint64_t* block_to_patch,
                                gpc_result* R) {
  const tmc2_frame* f = &g->frames[frame_index];
  const tmc2_params* P = &g->params;
  const usize res = P->occupancy_resolution, prec = P->occupancy_precision;
  const usize width = g->width, height = g->height;
  const usize bw = width / res, bh = height / res;                 /* :269-270 */
  const usize map_count = (usize)P->map_count_minus1 + 1;          /* :271 */
  int st;

  ps_init(&R->reconstruct);
  if (P->attribute_count > 0) R->reconstruct.with_colors = 1;      /* :274-276 add_colors */
  vec_init(&R->partition, sizeof(usize));
  vec_init(&R->point_to_pixel, 3 * sizeof(usize));

  /* :288-300 occupancy map upscaling from the video, nearest neighbour */
  R->occupancy_map = (uint8_t*)calloc((size_t)(width * height + 1), 1);
  if (!R->occupancy_map) return TMC2_ERR_INTERNAL;
  for (usize v = 0; v < height; ++v)
    for (usize u = 0; u < width; ++u) {
      uint8_t o;
      st = occ_get(g, f, u / prec, v / prec, &o);
      if (st) return st;
      R->occupancy_map[v * width + u] = o;
    }

  /* :317-320 the geometry video must hold frames f*M .. f*M+M-1 */
  const usize video_frame_index = (usize)frame_index * map_count;
  if ((usize)g->geo_video_frames < video_frame_index + map_count) return TMC2_ERR_SHORT_VIDEO;
  /* :415-432: created_points[1] is None for a single map and gets unwrapped -> panic */
  if (map_count != 2) return TMC2_ERR_MAP_COUNT;
  if (!f->geo[0] || !f->geo[1]) return TMC2_ERR_INVALID_ARG;

  for (usize patch_index = 0; patch_index < f->patch_count; ++patch_index) {   /* :352 */
    const tmc2_patch* p = &f->patches[patch_index];
    for (usize v0 = 0; v0 < p->size_v0; ++v0) {                                /* :371 */
      for (usize u0 = 0; u0 < p->size_u0; ++u0) {                              /* :372 */
        usize bx, by;
        st = orc_patch_to_canvas(p, (uint32_t)res, P->orientation_mode, 1, u0, v0, bw, bh, &bx, &by); /* :373-378 */
        if (st) return st;
        if (block_to_patch[by * bw + bx] != patch_index + 1) continue;        /* :379 */
        for (usize v1 = 0; v1 < res; ++v1) {                                   /* :382 */
          const usize v = v0 * res + v1;
          for (usize u1 = 0; u1 < res; ++u1) {                                 /* :384 */
            const usize u = u0 * res + u1;
            usize x, y;
            st = orc_patch_to_canvas(p, (uint32_t)res, P->orientation_mode, 0, u, v, width, height, &x, &y); /* :386 */
            if (st) return st;
            if (R->occupancy_map[y * width + x] == 0) continue;               /* :393-396 */
            uint16_t created[2][3];
            generate_points(g, f, p, u, v, x, y, created[0], created[1]);     /* :405-413 */
            for (usize i = 0; i < 2; ++i) {                                    /* :421 */
              if (i != 0 && created[i][0] == created[0][0] && created[i][1] == created[0][1] &&
                  created[i][2] == created[0][2])
                continue;                                                      /* :422-428 unconditional dedup */
              if (p->axis_of_additional_plane != 0) return TMC2_ERR_UNSUPPORTED; /* :437 unimplemented!() */
              const size_t point_index = ps_add_point(&R->reconstruct, created[i]); /* :432 */
              usize* pp = (usize*)(R->reconstruct.point_patch_indexes.data + point_index * 16);
              pp[0] = 0 /* tile_index */; pp[1] = patch_index;                /* :433 */
              vec_push(&R->partition, &patch_index);                           /* :452 */
              const usize px[3] = {x, y, i};
              vec_push(&R->point_to_pixel, px);                                /* :463-472 */
            }
          }
        }
      }
    }
  }

  /* :502-511 -> color_point_cloud, codec.rs:569-658 (attribute_count is 0 or 1) */
  if (P->attribute_count > 0 && R->reconstruct.positions.len != 0) {           /* :578-580 early return */
    if (g->attr_video_frames < 2) return TMC2_ERR_SHORT_VIDEO;                 /* :589-590 unwrap */
    const usize shift = (usize)frame_index * map_count;                        /* :620-624 */
    const size_t n = R->point_to_pixel.len;
    const usize* ptp = (const usize*)R->point_to_pixel.data;
    uint16_t* c16 = (uint16_t*)R->reconstruct.colors16bit.data;
    for (size_t i = 0; i < n; ++i) {                                           /* :626 */
      const usize x = ptp[3 * i + 0], y = ptp[3 * i + 1], z = ptp[3 * i + 2];
      if (!(z < map_count)) return TMC2_ERR_UNSUPPORTED;                       /* :641-643 */
      if ((usize)g->attr_video_frames <= z + shift) return TMC2_ERR_SHORT_VIDEO; /* :637 unwrap */
      if (!f->attr_y[z] || !f->attr_u[z] || !f->attr_v[z]) return TMC2_ERR_INVALID_ARG;
      for (int c = 0; c < 3; ++c) c16[3 * i + c] = attr_get(f, (int)z, c, x, y); /* :638-640 */
    }
  }
  return TMC2_OK;
}

/* ================================================================================================
 * Post-processing: NOT in the reference (stubs at decoder.rs:291-299, codec.rs:498-500).  This is the
 * repository's own integer specification, modelled on the structure of MPEG TMC2's grid smoothing
 * (identifyBoundaryPoints / addGridCentroid / gridFiltering / smoothPointCloudGrid and the colour
 * counterparts).  Every quantity is an exact integer; the CUDA kernels must match bit for bit.
 * "parity unpinned" with respect to upstream.  DESIGN.md holds the prose version of this spec.
 * ============================================================================================== */

/* K5: boundary type of the pixel (x,y) on the full-resolution occupancy map. */
static uint8_t boundary_type_of(const uint8_t* occ, usize W, usize H, usize x, usize y) {
  if (x == 0 || y == 0 || x == W - 1 || y == H - 1) return 1;
  if (occ[y * W + x - 1] == 0 || occ[y * W + x + 1] == 0 || occ[(y - 1) * W + x] == 0 || occ[(y + 1) * W + x] == 0)
    return 1;
  for (int dy = -2; dy <= 2; ++dy)
    for (int dx = -2; dx <= 2; ++dx) {
      const int64_t xx = (int64_t)x + dx, yy = (int64_t)y + dy;
      if (xx < 0 || yy < 0 || xx >= (int64_t)W || yy >= (int64_t)H) continue;
      if (occ[(usize)yy * W + (usize)xx] == 0) return 2;
    }
  return 0;
}

/* Sparse cell table: open addressing, key = cx | cy<<10 | cz<<20 (grid width <= 1024 per axis). */
typedef struct cell {
  uint32_t key, count, pmin, pmax;
  uint64_t s[3];   /* geometry: sum x,y,z ; colour: sum Y,U,V */
  uint64_t sy2;    /* colour only: sum of Y^2 */
} cell;
typedef struct cell_table { cell* c; uint64_t mask; } cell_table;
#define CELL_EMPTY 0xFFFFFFFFu

static int table_init(cell_table* t, uint64_t n_points) {
  uint64_t cap = 16;
  while (cap < 2 * n_points + 1) cap <<= 1;
  t->c = (cell*)malloc((size_t)cap * sizeof(cell));
  if (!t->c) return -1;
  for (uint64_t i = 0; i < cap; ++i) { t->c[i].key = CELL_EMPTY; }
  t->mask = cap - 1;
  return 0;
}
static inline uint64_t hash_key(uint32_t k) { uint64_t h = (uint64_t)k * 0x9E3779B97F4A7C15ull; return h >> 20; }
static cell* table_find(const cell_table* t, uint32_t key, int insert) {
  uint64_t i = hash_key(key) & t->mask;
  for (;;) {
    cell* c = &t->c[i];
    if (c->key == key) return c;
    if (c->key == CELL_EMPTY) {
      if (!insert) return NULL;
      c->key = key; c->count = 0; c->pmin = 0xFFFFFFFFu; c->pmax = 0; c->s[0] = c->s[1] = c->s[2] = 0; c->sy2 = 0;
      return c;
    }
    i = (i + 1) & t->mask;
  }
}

typedef struct grid_geom { uint32_t g, w, disth, th; } grid_geom;
static int grid_geom_init(grid_geom* G, uint32_t grid_size, uint32_t bitdepth) {
  if (grid_size < 1 || bitdepth == 0 || bitdepth > 16) return TMC2_ERR_INVALID_ARG;
  const uint32_t max_size = 1u << bitdepth;
  G->g = grid_size;
  G->w = (max_size + grid_size - 1) / grid_size;
  if (G->w > 1024) return TMC2_ERR_UNSUPPORTED;
  G->disth = grid_size / 2 > 1 ? grid_size / 2 : 1;
  G->th = grid_size * G->w;
  return TMC2_OK;
}
static inline int in_grid(const grid_geom* G, const uint16_t p[3]) {
  return p[0] < G->th && p[1] < G->th && p[2] < G->th;
}
static inline uint32_t cell_key(uint32_t cx, uint32_t cy, uint32_t cz) { return cx | (cy << 10) | (cz << 20); }

/* The 2x2x2 neighbourhood and its trilinear weights for a point, shared by K6 and K7.
 * Returns 0 when the point is skipped by the border test. */
typedef struct nbhd { uint32_t key[8]; int valid[8]; uint64_t wgt[8]; uint64_t w3; } nbhd;
static int neighbourhood(const grid_geom* G, const uint16_t p[3], nbhd* N) {
  if (!in_grid(G, p)) return 0;
  for (int a = 0; a < 3; ++a)
    if (p[a] < G->disth || (uint32_t)p[a] + G->disth >= G->th) return 0;
  int32_t s[3]; uint64_t wa[3];
  for (int a = 0; a < 3; ++a) {
    const uint32_t c = p[a] / G->g, rem = p[a] - c * G->g;
    s[a] = (int32_t)c + (rem < G->g / 2 ? -1 : 0);
    wa[a] = 2ull * (uint64_t)((int64_t)p[a] - (int64_t)s[a] * (int64_t)G->g - (int64_t)(G->g / 2)) + 1ull;
  }
  const uint64_t g2 = 2ull * G->g;
  N->w3 = g2 * g2 * g2;
  for (int k = 0; k < 8; ++k) {
    const int dx = k & 1, dy = (k >> 1) & 1, dz = (k >> 2) & 1;
    const int32_t cx = s[0] + dx, cy = s[1] + dy, cz = s[2] + dz;
    N->valid[k] = cx >= 0 && cy >= 0 && cz >= 0 && (uint32_t)cx < G->w && (uint32_t)cy < G->w && (uint32_t)cz < G->w;
    N->key[k] = N->valid[k] ? cell_key((uint32_t)cx, (uint32_t)cy, (uint32_t)cz) : CELL_EMPTY;
    N->wgt[k] = (dx ? wa[0] : g2 - wa[0]) * (dy ? wa[1] : g2 - wa[1]) * (dz ? wa[2] : g2 - wa[2]);
  }
  return 1;
}

/* K6: grid geometry smoothing.  positions are updated in place; returns the number of moved points. */
static int geometry_smoothing(const tmc2_params* P, uint64_t n, uint16_t* pos, const uint64_t* partition,
                              const uint8_t* btype, uint64_t* moved) {
  grid_geom G;
  int st = grid_geom_init(&G, P->grid_size, P->geometry_bitdepth_3d);
  *moved = 0;
  if (st) return st;
  cell_table T;
  if (table_init(&T, n)) return TMC2_ERR_INTERNAL;
  /* pass 1: per-cell sums, counts and the min / max patch index seen */
  for (uint64_t k = 0; k < n; ++k) {
    const uint16_t* p = pos + 3 * k;
    if (!in_grid(&G, p)) continue;
    cell* c = table_find(&T, cell_key(p[0] / G.g, p[1] / G.g, p[2] / G.g), 1);
    c->count++;
    c->s[0] += p[0]; c->s[1] += p[1]; c->s[2] += p[2];
    const uint32_t pa = (uint32_t)partition[k];
    if (pa < c->pmin) c->pmin = pa;
    if (pa > c->pmax) c->pmax = pa;
  }
  /* pass 2: filter boundary points (type 1) against the trilinear blend of the 8 surrounding cell means */
  const uint64_t thr = P->threshold_smoothing;
  for (uint64_t k = 0; k < n; ++k) {
    if (btype[k] != 1) continue;
    uint16_t* p = pos + 3 * k;
    nbhd N;
    if (!neighbourhood(&G, p, &N)) continue;
    const cell* cs[8]; int other = 0;
    for (int j = 0; j < 8; ++j) {
      cs[j] = N.valid[j] ? table_find(&T, N.key[j], 0) : NULL;
      if (cs[j] && cs[j]->count > 0 && cs[j]->pmin != cs[j]->pmax) other = 1;
    }
    if (!other) continue;
    uint64_t C[3] = {0, 0, 0}, cntw = 0;
    for (int j = 0; j < 8; ++j) {
      for (int a = 0; a < 3; ++a) {
        uint64_t m = 256ull * p[a];                                             /* empty cell -> the point itself */
        if (cs[j] && cs[j]->count > 0) m = (256ull * cs[j]->s[a] + cs[j]->count / 2) / cs[j]->count; /* mean, Q8 */
        C[a] += N.wgt[j] * m;
      }
      if (cs[j]) cntw += N.wgt[j] * cs[j]->count;
    }
    const uint64_t count = cntw / N.w3;
    if (count == 0) continue;
    uint64_t c4[3]; uint64_t D2 = 0;
    for (int a = 0; a < 3; ++a) {
      c4[a] = (C[a] + N.w3 / 2) / N.w3;                                         /* blended centroid, Q8 */
      const int64_t d = (int64_t)(256ull * p[a]) - (int64_t)c4[a];
      D2 += (uint64_t)(d * d);
    }
    const uint64_t m = thr > count ? thr : count;
    const unsigned __int128 lhs = (unsigned __int128)2 * count * D2 + 65536u;   /* dist2 = count*|d|^2/65536 + 1/2 */
    const unsigned __int128 rhs = (unsigned __int128)262144u * m;               /* >= 2*max(threshold, count)      */
    if (lhs >= rhs) {
      uint16_t q[3]; int changed = 0;
      for (int a = 0; a < 3; ++a) {
        uint64_t r = (c4[a] + 128) >> 8;
        if (r > 65535) r = 65535;
        q[a] = (uint16_t)r;
        changed |= q[a] != p[a];
      }
      p[0] = q[0]; p[1] = q[1]; p[2] = q[2];
      *moved += (uint64_t)changed;
    }
  }
  free(T.c);
  return TMC2_OK;
}

/* K7: grid colour smoothing on the 16-bit YUV colours; cells are indexed by the pre-geometry-smoothing positions. */
static int color_smoothing(const tmc2_params* P, uint64_t n, const uint16_t* pos, uint16_t* c16,
                           const uint64_t* partition, const uint8_t* btype, uint64_t* recoloured) {
  grid_geom G;
  int st = grid_geom_init(&G, P->cgrid_size, P->geometry_bitdepth_3d);
  *recoloured = 0;
  if (st) return st;
  cell_table T;
  if (table_init(&T, n)) return TMC2_ERR_INTERNAL;
  const uint64_t cs_scale = P->attribute_bitdepth > 8 ? (1ull << (P->attribute_bitdepth - 8)) : 1ull;
  const uint64_t t_smooth = P->threshold_color_smoothing * cs_scale;
  const uint64_t t_diff = P->threshold_color_difference * cs_scale;
  const uint64_t t_var = P->threshold_color_variation * cs_scale;
  /* pass 1: colour statistics of the SECOND-RING points (type 2): pixels next to, but not on, a patch outline.  The
   * outline pixels themselves (type 1) carry the colour bleeding that this stage removes, so they are filtered
   * (pass 2) but do not vote.  This is what gives boundary type 2 its purpose. */
  for (uint64_t k = 0; k < n; ++k) {
    if (btype[k] != 2) continue;
    const uint16_t* p = pos + 3 * k;
    if (!in_grid(&G, p)) continue;
    cell* c = table_find(&T, cell_key(p[0] / G.g, p[1] / G.g, p[2] / G.g), 1);
    c->count++;
    const uint16_t* col = c16 + 3 * k;
    c->s[0] += col[0]; c->s[1] += col[1]; c->s[2] += col[2];
    c->sy2 += (uint64_t)col[0] * col[0];
    const uint32_t pa = (uint32_t)partition[k];
    if (pa < c->pmin) c->pmin = pa;
    if (pa > c->pmax) c->pmax = pa;
  }
  for (uint64_t k = 0; k < n; ++k) {
    if (btype[k] != 1) continue;
    const uint16_t* p = pos + 3 * k;
    uint16_t* col = c16 + 3 * k;
    nbhd N;
    if (!neighbourhood(&G, p, &N)) continue;
    const cell* cs[8]; int other = 0;
    for (int j = 0; j < 8; ++j) {
      cs[j] = N.valid[j] ? table_find(&T, N.key[j], 0) : NULL;
      if (cs[j] && cs[j]->count > 0 && cs[j]->pmin != cs[j]->pmax) other = 1;
    }
    if (!other) continue;
    uint64_t C[3] = {0, 0, 0};
    for (int j = 0; j < 8; ++j) {
      int usable = cs[j] && cs[j]->count > 0;
      uint64_t mean[3] = {0, 0, 0};
      if (usable) {
        const uint64_t cnt = cs[j]->count;
        for (int a = 0; a < 3; ++a) mean[a] = (256ull * cs[j]->s[a] + cnt / 2) / cnt;  /* Q8 */
        /* luminance variation: var(Y) = (cnt*sumY2 - sumY^2)/cnt^2 must not exceed t_var^2 */
        const unsigned __int128 num = (unsigned __int128)cnt * cs[j]->sy2 - (unsigned __int128)cs[j]->s[0] * cs[j]->s[0];
        const unsigned __int128 lim = (unsigned __int128)(t_var * cnt) * (t_var * cnt);
        if (num > lim) usable = 0;
        /* luminance difference between the cell mean and the point */
        const int64_t dy = (int64_t)mean[0] - (int64_t)(256ull * col[0]);
        if ((uint64_t)(dy < 0 ? -dy : dy) > 256ull * t_diff) usable = 0;
      }
      for (int a = 0; a < 3; ++a) C[a] += N.wgt[j] * (usable ? mean[a] : 256ull * col[a]);
    }
    uint16_t q[3]; uint64_t dist = 0;
    for (int a = 0; a < 3; ++a) {
      const uint64_t c4 = (C[a] + N.w3 / 2) / N.w3;
      uint64_t r = (c4 + 128) >> 8;
      if (r > 65535) r = 65535;
      q[a] = (uint16_t)r;
      const int64_t d = (int64_t)q[a] - (int64_t)col[a];
      dist += (uint64_t)(d < 0 ? -d : d) * (a == 0 ? 10u : 1u);
    }
    if (dist >= t_smooth && dist > 0) {
      col[0] = q[0]; col[1] = q[1]; col[2] = q[2];
      *recoloured += 1;
    }
  }
  free(T.c);
  return TMC2_OK;
}

/* ------------------------------------------------------------------------------------------------
 * The per-frame body of the driver loop, decoder.rs:188-311.
 * ---------------------------------------------------------------------------------------------- */
int orc_reconstruct_frame(const tmc2_gof* g, uint32_t frame_index, orc_frame** out) {
  if (!out) return TMC2_ERR_INVALID_ARG;
  *out = NULL;
  int st = check_gof(g, frame_index);
  if (st) return st;
  const tmc2_params* P = &g->params;
  const usize res = P->occupancy_resolution;
  const usize blocks = (g->width / res) * (g->height / res);

  orc_frame* F = (orc_frame*)calloc(1, sizeof(orc_frame));
  if (!F) return TMC2_ERR_INTERNAL;
  F->block_count = blocks;
  F->block_to_patch = (uint64_t*)calloc((size_t)(blocks ? blocks : 1), sizeof(uint64_t));

  /* decoder.rs:249-255 */
  st = orc_generate_block_to_patch_from_occupancy_map_video(g, frame_index, F->block_to_patch);
  if (st) { orc_frame_free(F); return st; }

  /* decoder.rs:258-272 */
  gpc_result R;
  memset(&R, 0, sizeof R);
  st = generate_point_cloud(g, frame_index, F->block_to_patch, &R);
  if (st) {
    ps_free(&R.reconstruct); vec_free(&R.partition); vec_free(&R.point_to_pixel); free(R.occupancy_map);
    orc_frame_free(F);
    return st;
  }

  /* decoder.rs:195-198,278: a fresh PointSet3 per frame, the tile's points appended (a full copy) */
  point_set3 reconstruct;
  ps_init(&reconstruct);
  if (P->attribute_count > 0) reconstruct.with_colors = 1;
  ps_append(&reconstruct, &R.reconstruct);
  ps_free(&R.reconstruct);

  const uint64_t n = reconstruct.positions.len;
  F->point_count = n;
  F->with_colors = (uint8_t)reconstruct.with_colors;
  F->occupancy_map = R.occupancy_map;
  F->partition = (uint64_t*)R.partition.data;          /* ownership moves */
  F->point_to_pixel = (uint64_t*)R.point_to_pixel.data;
  F->point_patch_indexes = (uint64_t*)reconstruct.point_patch_indexes.data;
  F->positions = (uint16_t*)reconstruct.positions.data;
  F->colors = (uint8_t*)reconstruct.colors.data;
  F->colors16bit = (uint16_t*)reconstruct.colors16bit.data;

  /* decoder.rs:291-299 hook points (own spec, see above) */
  if ((P->geometry_smoothing || P->color_smoothing) && n > 0) {
    F->boundary_type = (uint8_t*)malloc((size_t)n);
    for (uint64_t k = 0; k < n; ++k)
      F->boundary_type[k] = boundary_type_of(F->occupancy_map, g->width, g->height, F->point_to_pixel[3 * k],
                                             F->point_to_pixel[3 * k + 1]);
    F->positions_presmooth = (uint16_t*)malloc((size_t)n * 6);
    memcpy(F->positions_presmooth, F->positions, (size_t)n * 6);
    if (P->geometry_smoothing) {
      st = geometry_smoothing(P, n, F->positions, F->partition, F->boundary_type, &F->smoothed_positions);
      if (st) { orc_frame_free(F); return st; }
    }
    if (P->color_smoothing && reconstruct.with_colors) {
      F->colors16bit_presmooth = (uint16_t*)malloc((size_t)n * 6);
      memcpy(F->colors16bit_presmooth, F->colors16bit, (size_t)n * 6);
      /* own spec: the colour grid is built on the RECONSTRUCTED (pre-geometry-smoothing) positions, so both
       * post-processing stages depend only on the unpack output and can share one pass over the points */
      st = color_smoothing(P, n, F->positions_presmooth, F->colors16bit, F->partition, F->boundary_type, &F->smoothed_colors);
      if (st) { orc_frame_free(F); return st; }
    }
  }

  /* decoder.rs:301-305 -> codec.rs:88-94 convert_yuv16_to_rgb8 (ColorFormat is always Yuv420) */
  if (reconstruct.with_colors)
    for (uint64_t i = 0; i < n; ++i) orc_convert_yuv10_to_rgb8(F->colors16bit + 3 * i, F->colors + 3 * i);

  *out = F;
  return TMC2_OK;
}

void orc_frame_free(orc_frame* f) {
  if (!f) return;
  free(f->positions); free(f->colors); free(f->colors16bit); free(f->point_patch_indexes); free(f->partition);
  free(f->point_to_pixel); free(f->occupancy_map); free(f->block_to_patch); free(f->boundary_type);
  free(f->positions_presmooth); free(f->colors16bit_presmooth);
  free(f);
}

int64_t orc_time_frames(const tmc2_gof* g, uint32_t first, uint32_t count) {
  int64_t total = 0;
  for (uint32_t k = 0; k < count; ++k) {
    orc_frame* F = NULL;
    const int st = orc_reconstruct_frame(g, first + k, &F);
    if (st) return -(int64_t)st;
    total += (int64_t)F->point_count;
    orc_frame_free(F);
  }
  return total;
}
