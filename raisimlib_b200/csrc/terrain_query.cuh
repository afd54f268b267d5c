// Terrain sensing: batched height scans and ray tests against the Ground plane / the HeightMap(s) the narrow phase collides with
// (rsb_batch_height_scan, rsb_batch_ray_test; conventions in DESIGN.md section 2).  Included by batch.cu after step_kernel.cuh
// (TerrainDesc, f3 helpers).  These kernels read the terrain and the state; they write nothing but the caller's output rows.
//
// Surface: cell (ix, iy) holds tri 0 = (P00, P10, P11) and tri 1 = (P00, P11, P01), pair index = 2 * cell + tri (narrow_phase.cuh).
#pragma once

namespace rsb {

constexpr int TQ_TILE = 8;             // cells per side of one tile of the ray test's coarse grid
constexpr int TQ_FRAME_WORDS = 16;     // frame record of a pattern: body (int bits), position in the body (3), rotation in the body (9), pad
constexpr float TQ_TIE = 1e-6f;        // two hits closer than this along the ray are a tie: the lower pair index wins (narrow-phase rule)

// height range of every TQ_TILE x TQ_TILE-cell tile of every map (built on the host by rsb_batch_set_heightmap(s)), [map][ty][tx]
struct TqTiles {
  const float2* mm;   // (min, max) over the tile's vertices
  int nx, ny;         // tiles per map along x, y
  float hmin, hmax;   // range of the whole atlas
};

// where a frame's pose comes from: body 0 of a floating base straight from the gc rows, any other body from the getters' pose buffers
struct TqPose {
  const float* gc; int gc_stride;
  const float* R; const float* p;      // [env][nb][9], [env][nb][3] (rsb_batch_get_body_poses layout; valid after ensure_kinematics)
  int nb, floating;
};

// world pose (p, R row-major) of frame record `fr` in environment `env`
__device__ __forceinline__ void tq_frame_pose(const TqPose& ps, const float* __restrict__ fr, int env, f3& p, float R[9]) {
  const int body = __float_as_int(__ldg(fr));
  float Rb[9]; f3 pb;
  if (body == 0 && ps.floating) {
    const float* q = ps.gc + (size_t)env * ps.gc_stride;
    float w = __ldg(q + 3), x = __ldg(q + 4), y = __ldg(q + 5), z = __ldg(q + 6);
    const float inv = 1.0f / sqrtf(w * w + x * x + y * y + z * z);
    w *= inv; x *= inv; y *= inv; z *= inv;
    Rb[0] = 1.f - 2.f * (y * y + z * z); Rb[1] = 2.f * (x * y - w * z); Rb[2] = 2.f * (x * z + w * y);
    Rb[3] = 2.f * (x * y + w * z); Rb[4] = 1.f - 2.f * (x * x + z * z); Rb[5] = 2.f * (y * z - w * x);
    Rb[6] = 2.f * (x * z - w * y); Rb[7] = 2.f * (y * z + w * x); Rb[8] = 1.f - 2.f * (x * x + y * y);
    pb = mk(__ldg(q), __ldg(q + 1), __ldg(q + 2));
  } else {
    const float* r = ps.R + ((size_t)env * ps.nb + body) * 9;
    const float* o = ps.p + ((size_t)env * ps.nb + body) * 3;
#pragma unroll
    for (int k = 0; k < 9; k++) Rb[k] = __ldg(r + k);
    pb = mk(__ldg(o), __ldg(o + 1), __ldg(o + 2));
  }
  const f3 fp = mk(__ldg(fr + 1), __ldg(fr + 2), __ldg(fr + 3));
  p = pb + mulR(Rb, fp);
  float Rf[9];
#pragma unroll
  for (int k = 0; k < 9; k++) Rf[k] = __ldg(fr + 4 + k);
  matmul3(Rb, Rf, R);
}

// terrain height at (x, y); outside the map the nearest border point (HeightMap::getHeight)
__device__ __forceinline__ float tq_height(const TerrainDesc& t, int hm_offset, float x, float y) {
  if (t.type == 1) return t.ground_z;
  const float gx = fminf(fmaxf((x - t.x0) / t.dx, 0.f), t.xmax), gy = fminf(fmaxf((y - t.y0) / t.dy, 0.f), t.ymax);
  const int ix = min((int)gx, t.xs - 2), iy = min((int)gy, t.ys - 2);
  const float fx = gx - (float)ix, fy = gy - (float)iy;
  const float* H = t.h + hm_offset + iy * t.xs + ix;
  const float h00 = __ldg(H), h10 = __ldg(H + 1), h01 = __ldg(H + t.xs), h11 = __ldg(H + t.xs + 1);
  return fx >= fy ? h00 + (h10 - h00) * fx + (h11 - h10) * fy : h00 + (h11 - h01) * fx + (h01 - h00) * fy;
}

// TQ_SCAN_PPT points of one (env, frame) per thread: the pose is computed once for them and their height gathers are independent.
// Thread g of the (env, frame) group takes points g, g + G, g + 2G, ... (G = ceil(P / TQ_SCAN_PPT)), so that the writes of a warp stay
// contiguous: out[e * out_stride + f * P + k] = z of frame f - height at (p_f + Rz(yaw_f) [x_k, y_k]).
// pat = frame records [F][TQ_FRAME_WORDS] then the points [P][2].  Threads of one (env, frame) read the same pose words (L1 broadcast).
constexpr int TQ_SCAN_PPT = 4;
__global__ void __launch_bounds__(256) rsb_height_scan_kernel(TerrainDesc t, TqPose ps, const float* __restrict__ pat, int F, int P, int env_begin,
                                                              int env_count, float* __restrict__ out, int out_stride) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int G = (P + TQ_SCAN_PPT - 1) / TQ_SCAN_PPT, per_env = F * G;
  if (i >= (long long)env_count * per_env) return;
  const int le = (int)(i / per_env), r = (int)(i - (long long)le * per_env), f = r / G, g = r - f * G;
  const int env = env_begin + le;
  f3 p; float R[9];
  tq_frame_pose(ps, pat + f * TQ_FRAME_WORDS, env, p, R);
  // heading frame: rotation about z by atan2(R10, R00); cos / sin of it without the trigonometry (atan2(0, 0) = 0)
  const float nrm = sqrtf(R[0] * R[0] + R[3] * R[3]);
  const float c = nrm > 0.f ? R[0] / nrm : 1.f, s = nrm > 0.f ? R[3] / nrm : 0.f;
  const int hm_offset = t.env_map ? __ldg(t.env_map + env) * t.map_words : 0;
  const float2* pts = reinterpret_cast<const float2*>(pat + F * TQ_FRAME_WORDS);
  float* o = out + (size_t)le * out_stride + f * P;
#pragma unroll
  for (int j = 0; j < TQ_SCAN_PPT; j++) {
    const int k = g + j * G;
    if (k < P) {
      const float2 xy = __ldg(pts + k);
      o[k] = p.z - tq_height(t, hm_offset, p.x + c * xy.x - s * xy.y, p.y + s * xy.x + c * xy.y);
    }
  }
}

struct TqHit { float t; f3 n; int pair; };

// keep the smallest t; a hit within TQ_TIE of the best is a tie that the lower pair index wins
__device__ __forceinline__ void tq_offer(TqHit& b, float tt, f3 n, int pair) {
  if (tt < b.t - TQ_TIE || (tt <= b.t + TQ_TIE && pair < b.pair)) { b.t = tt; b.n = n; b.pair = pair; }
}

// [ta, tb] &= the parameters where o + t d lies in [lo, hi] along one axis
__device__ __forceinline__ void tq_clip(float o, float d, float lo, float hi, float& ta, float& tb) {
  if (d == 0.f) {
    if (!(o >= lo && o <= hi)) ta = INFINITY;
    return;
  }
  const float t1 = (lo - o) / d, t2 = (hi - o) / d;
  ta = fmaxf(ta, fminf(t1, t2)); tb = fminf(tb, fmaxf(t1, t2));
}

// Amanatides-Woo walk along one axis of a grid whose cells are `scale` map cells wide, in map-cell coordinates u(t) = go + t gd
struct TqAxis {
  int c, step, lo, hi;
  float go, gd, scale, tnext;   // tnext: parameter where the ray leaves cell c along this axis (+inf when it never does)
  __device__ __forceinline__ void init(float go_, float gd_, float ts, float scale_, int lo_, int hi_) {
    go = go_; gd = gd_; scale = scale_; lo = lo_; hi = hi_;
    c = min(max((int)floorf((go + ts * gd) / scale), lo), hi);
    step = gd > 0.f ? 1 : -1;
    next();
  }
  // recomputed from the integer cell index at every step: no drift along long rays, and a zero gd gives +inf through the same code
  __device__ __forceinline__ void next() { tnext = gd == 0.f ? INFINITY : ((float)(c + (step > 0)) * scale - go) / gd; }
};

// both triangles of cell (ix, iy); arithmetic relative to the cell corner keeps float32 precision far from the map centre
__device__ __forceinline__ void tq_cell(const TerrainDesc& t, const float* H, int ix, int iy, f3 o, f3 d, float len, TqHit& best) {
  const float* c = H + iy * t.xs + ix;
  const float h00 = __ldg(c), h10 = __ldg(c + 1), h01 = __ldg(c + t.xs), h11 = __ldg(c + t.xs + 1);
  const float ox = o.x - (t.x0 + (float)ix * t.dx), oy = o.y - (t.y0 + (float)iy * t.dy), oz = o.z - h00;
  const int cell = iy * (t.xs - 1) + ix;
  constexpr float E = 1e-5f;   // in cells: a ray through a shared edge hits both triangles (watertight), the tie rule picks one
#pragma unroll
  for (int tri = 0; tri < 2; tri++) {
    // plane of the triangle: z - h00 = ax x' + ay y' (x', y' relative to the corner); tri 0 = (P00, P10, P11), tri 1 = (P00, P11, P01)
    const float ax = (tri == 0 ? h10 - h00 : h11 - h01) * t.inv_dx, ay = (tri == 0 ? h11 - h10 : h01 - h00) * t.inv_dy;
    const float den = d.z - ax * d.x - ay * d.y;
    if (den == 0.f) continue;                                        // parallel to the plane
    const float tt = (ax * ox + ay * oy - oz) / den;
    if (!(tt >= 0.f && tt <= len)) continue;
    const float fx = (ox + tt * d.x) * t.inv_dx, fy = (oy + tt * d.y) * t.inv_dy;
    const bool in = tri == 0 ? (fx <= 1.f + E && fy >= -E && fy <= fx + E) : (fx >= -E && fy <= 1.f + E && fx <= fy + E);
    if (!in) continue;
    const float inv = 1.0f / sqrtf(ax * ax + ay * ay + 1.f);
    tq_offer(best, tt, mk(-ax * inv, -ay * inv, inv), 2 * cell + tri);
  }
}

// first crossing of o + t d (|d| = 1), t in [0, len], with the terrain; best.pair < 0: no hit
__device__ TqHit tq_ray(const TerrainDesc& t, const TqTiles& tl, int env, f3 o, f3 d, float len) {
  TqHit best; best.t = INFINITY; best.n = mk(0.f, 0.f, 0.f); best.pair = 0x7fffffff;
  if (t.type == 1) {
    const float tt = (t.ground_z - o.z) / d.z;                        // d.z = 0: +-inf or NaN, rejected below
    if (tt >= 0.f && tt <= len) { best.t = tt; best.n = mk(0.f, 0.f, 1.f); best.pair = 0; }
  } else if (t.type == 2) {
    // level 0: clip to the map rectangle (nothing outside it is hit, hm_cell_range) and to the height range of the atlas
    float ta = 0.f, tb = len;
    tq_clip(o.x, d.x, t.x0, t.x0 + t.xmax * t.dx, ta, tb);
    tq_clip(o.y, d.y, t.y0, t.y0 + t.ymax * t.dy, ta, tb);
    tq_clip(o.z, d.z, tl.hmin - 1e-4f, tl.hmax + 1e-4f, ta, tb);
    if (ta <= tb) {
      const int map = t.env_map ? __ldg(t.env_map + env) : 0;
      const float* H = t.h + (size_t)map * t.map_words;
      const float2* mm = tl.mm + (size_t)map * tl.nx * tl.ny;
      const float gox = (o.x - t.x0) * t.inv_dx, goy = (o.y - t.y0) * t.inv_dy, gdx = d.x * t.inv_dx, gdy = d.y * t.inv_dy;
      // level 1: tiles of TQ_TILE x TQ_TILE cells, skipped when the ray's z range over the tile misses the tile's [min, max]
      TqAxis TX, TY;
      TX.init(gox, gdx, ta, (float)TQ_TILE, 0, tl.nx - 1); TY.init(goy, gdy, ta, (float)TQ_TILE, 0, tl.ny - 1);
      float tin = ta;
      for (;;) {
        const float tout = fminf(fminf(TX.tnext, TY.tnext), tb);
        const float z0 = o.z + tin * d.z, z1 = o.z + tout * d.z;
        const float2 r = __ldg(mm + TY.c * tl.nx + TX.c);
        if (fmaxf(z0, z1) >= r.x - 1e-4f && fminf(z0, z1) <= r.y + 1e-4f) {
          // level 2: the cells of this tile along the ray, both triangles of each
          TqAxis CX, CY;
          CX.init(gox, gdx, tin, 1.f, TX.c * TQ_TILE, min(TX.c * TQ_TILE + TQ_TILE - 1, t.xs - 2));
          CY.init(goy, gdy, tin, 1.f, TY.c * TQ_TILE, min(TY.c * TQ_TILE + TQ_TILE - 1, t.ys - 2));
          float cin = tin;
          for (;;) {
            tq_cell(t, H, CX.c, CY.c, o, d, len, best);
            const float cout = fminf(CX.tnext, CY.tnext);
            if (cout >= tout) break;
            if (CX.tnext < CY.tnext) { CX.c += CX.step; if (CX.c < CX.lo || CX.c > CX.hi) break; cin = CX.tnext; CX.next(); }
            else { CY.c += CY.step; if (CY.c < CY.lo || CY.c > CY.hi) break; cin = CY.tnext; CY.next(); }
            if (cin > best.t + TQ_TIE) break;                          // the first cell that holds a hit ends the walk (ties: one cell more)
          }
        }
        if (tout >= tb || tout > best.t + TQ_TIE) break;
        if (TX.tnext < TY.tnext) { TX.c += TX.step; if (TX.c < TX.lo || TX.c > TX.hi) break; tin = TX.tnext; TX.next(); }
        else { TY.c += TY.step; if (TY.c < TY.lo || TY.c > TY.hi) break; tin = TY.tnext; TY.next(); }
      }
    }
  }
  if (best.pair == 0x7fffffff) best.pair = -1;
  return best;
}

// One thread per (env, frame, ray): neighbouring lanes hold neighbouring rays of one sensor and write neighbouring 32-byte records.
// F >= 1: pat = frame records [F][TQ_FRAME_WORDS], origins [R][3], unit directions [R][3], all fixed in the frame; out [env][F][R].
// F == 0: org / dir = world-frame rays [env_count][R][3] (directions normalised here; zero -> miss); out [env][R].
__global__ void __launch_bounds__(256) rsb_ray_test_kernel(TerrainDesc t, TqTiles tl, TqPose ps, const float* __restrict__ pat, int F,
                                                           const float* __restrict__ org, const float* __restrict__ dir, int R, float len,
                                                           int env_begin, int env_count, rsb_ray_hit* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int per_env = max(F, 1) * R;
  if (i >= (long long)env_count * per_env) return;
  const int le = (int)(i / per_env), r = (int)(i - (long long)le * per_env), k = r % R;
  const int env = env_begin + le;
  f3 o, d;
  if (F > 0) {
    const int f = r / R;
    f3 p; float Rw[9];
    tq_frame_pose(ps, pat + f * TQ_FRAME_WORDS, env, p, Rw);
    const float* ro = pat + F * TQ_FRAME_WORDS + 3 * k;
    const float* rd = pat + F * TQ_FRAME_WORDS + 3 * R + 3 * k;
    o = p + mulR(Rw, mk(__ldg(ro), __ldg(ro + 1), __ldg(ro + 2)));
    d = mulR(Rw, mk(__ldg(rd), __ldg(rd + 1), __ldg(rd + 2)));
  } else {
    const size_t w = ((size_t)le * R + k) * 3;
    o = mk(__ldg(org + w), __ldg(org + w + 1), __ldg(org + w + 2));
    d = mk(__ldg(dir + w), __ldg(dir + w + 1), __ldg(dir + w + 2));
  }
  const float dd = dot(d, d);
  TqHit h;
  if (dd > 0.f && dd < INFINITY) { d = (1.0f / sqrtf(dd)) * d; h = tq_ray(t, tl, env, o, d, len); }
  else { h.t = INFINITY; h.n = mk(0.f, 0.f, 0.f); h.pair = -1; }
  rsb_ray_hit rec;
  if (h.pair >= 0) {
    rec.distance = h.t;
    rec.position[0] = o.x + h.t * d.x; rec.position[1] = o.y + h.t * d.y; rec.position[2] = o.z + h.t * d.z;
    rec.normal[0] = h.n.x; rec.normal[1] = h.n.y; rec.normal[2] = h.n.z;
  } else {
    rec.distance = INFINITY;
    rec.position[0] = rec.position[1] = rec.position[2] = 0.f; rec.normal[0] = rec.normal[1] = rec.normal[2] = 0.f;
  }
  rec.pair_index = h.pair;
  out[i] = rec;
}

}  // namespace rsb
