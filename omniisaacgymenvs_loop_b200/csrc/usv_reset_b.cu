// Scene rebuild of the LIVE CaptureXY task for the envs that reset (SURVEY rows B5, B6): obstacle placement by rejection
// sampling  [ref: OIGE/tasks/USV/USV_capture_xy_static_obs.py:936-1060]  and the per-env potential field of BatchedMapGPU
// [ref: OIGE/tasks/USV/d_multi_gemini.py:66-104 occupancy + SDF, :135-192 cost-to-go wavefront, :194-271 potential field].
//
// The reference runs 225 Jacobi sweeps of an 8-neighbour min-plus relaxation as ~30 torch ops per sweep over the whole
// (B,150,150) batch in HBM.  Here ONE CTA owns one env: the 150x150 cost buffer lives in shared memory (94 KB with an +inf halo,
// two scenes per SM) and is relaxed in place until nothing changes -- the same fixed point, bit for bit, as the reference's Jacobi
// sweeps (see the comment at scene_cost_kernel).  The reference's BATCH-GLOBAL maxima (max finite cost, max repulsion: quirk 9 of
// SURVEY appendix C) and its per-scene min / max normalisation are reductions over cells whose inputs do not depend on those
// maxima except through ONE scalar factor, so the cost kernel takes all of them in its write-out pass and the field itself is a
// plain elementwise map:
//   scene_cost_kernel  : obstacles (warp 0) -> free mask -> wavefront -> raw cost into field[env]; per-scene statistics (min / max
//                        finite cost, min / max repulsion over finite-cost and over unreachable cells, flags) into the workspace,
//                        batch maxima by atomicMax
//   scene_field_kernel : field[env] = norm(G) + 0.5 norm(J) per cell, any number of CTAs per scene (no reduction left)
// A cell the wavefront never reaches has G = 1.5 x (batch max cost) and a repulsion 20 q^2 * rep with rep = clamp(G * 0.2 / 3, 0, 1) the
// same for every such cell: fl(a * rep) is monotone in a, so min / max over those cells are taken on 20 q^2 and scaled afterwards,
// bit for bit what the reference's max over the products gives.  (r01 / early r02 ran a third kernel for the batch max of J and two
// passes in the field kernel: 31 + 68 us of a 260 us control step at 16 384 envs.)
// Both kernels are persistent grids striding over the compacted list of resetting envs (or over a dense batch for the
// standalone builder entry), so their cost is ~0 when nothing resets.
#include <math_constants.h>
#include "philox.cuh"
#include "usv_step_core.cuh"

namespace usv {

constexpr int kG = USV_B_GRID;       // 150
constexpr int kGP = kG + 2;          // padded rows / columns (halo of +inf)
constexpr int kGS = kGP + 1;         // row stride of the padded buffer, 153 words: the four 8-row groups of a tile pass (8 rows apart) fall on
                                     // banks 0-7 / 8-15 / 16-23 / 24-31 (8 * 153 mod 32 == 8), one conflict-free wavefront per load
constexpr int kGPR = kGP + 2;        // rows of the padded buffer: the halo plus two spare +inf rows (a tile pass always reads 10 rows)
constexpr int kCells = kG * kG;
constexpr int kColIters = (kG + 31) / 32;  // 5
constexpr int kMaxSweeps = (int)(kG * 1.5);  // 225  (d_multi_gemini.py:160)
constexpr int kNearCap = USV_B_OBSTACLES * 18 * 18;   // cells with one obstacle within kReach on both axes: an interval of 2 x 1.701 holds <= 18 cell centres
constexpr float kObstR = 0.5f;
// wavefront tiles: 8 columns x 32 rows, one warp per tile pass; lane = (column cx = lane & 7, row group g = lane >> 3), 8 rows per lane.
// Inside a lane's column the pass is a Gauss-Seidel walk down and back up (a value crosses the lane's 8 rows in one pass), across
// columns and row groups it is Jacobi: a value crosses a tile in <= 8 passes sideways and <= 4 vertically.  (r01 / early r02: 32
// columns x 8 rows, pure Jacobi: up to 32 passes to cross sideways, ~20 passes per tile and scene in the instrumented run.)
constexpr int kTileW = 8, kBandRows = 8, kGroups = 4, kTileH = kGroups * kBandRows;
constexpr int kChunks = (kG + kTileW - 1) / kTileW, kBands = (kG + kTileH - 1) / kTileH, kTiles = kChunks * kBands;  // 19 x 5 = 95
constexpr int kActStride = 96;       // tile-active flags per sweep parity
constexpr float kReach = 1.7f + 1e-3f;  // an obstacle matters to a cell only within 0.5 (radius) + 0.5 + 0.7 (influence) of its centre

// counters (uint32[8]) in the workspace
enum { CW_COUNT = 0, CW_MAXCOST = 1, CW_MAXJ = 2, CW_INSIDE = 3, CW_HAVE = 4, CW_MAXJ_INF = 5, CW_WORDS = 8 };
// CW_MAXJ: batch max of the repulsion over finite-cost cells; CW_MAXJ_INF: batch max of 20 q^2 over unreachable cells (scaled by rep later)

// per-scene statistics (floats) written by the cost kernel, read by the field kernel
enum { SS_MIN_COST = 0, SS_MAX_COST = 1, SS_JFIN_MIN = 2, SS_JFIN_MAX = 3, SS_JINF_MIN = 4, SS_JINF_MAX = 5, SS_FLAGS = 6, SS_WORDS = 8 };
enum { SSF_HAS_INF = 1, SSF_HAS_INSIDE = 2, SSF_HAS_JFIN = 4, SSF_HAS_JINF = 8 };

struct SceneIO {
  // list mode (list != nullptr): env id = list[j]; obstacles in bconsts (AoSoA), target in consts, field[env]
  const int32_t* list;
  const uint32_t* count;  // number of list entries (device)
  float* bconsts;
  const float* consts;
  // dense mode: j-th scene of a batch of m
  const float* obstacles;  // [m,16,2]
  const float* targets;    // [m,2]
  int64_t m;
  float* field;            // [*,150,150]
  float* cost_out;         // dense mode only, or NULL
  const float* lin;        // [150] cell-centre coordinates (torch.linspace(-14.9, 14.9, 150))
  float* stats;            // [scenes][SS_WORDS] per-scene statistics (workspace)
};

__device__ __forceinline__ int64_t scene_count(const SceneIO& io) { return io.list ? (int64_t)*io.count : io.m; }

// bit j set: obstacle j is within kReach of grid row cy (|dy| <= dist), i.e. it can make a cell of that row occupied / repelled
__device__ __forceinline__ uint32_t row_obstacle_mask(float cy, const float* s_oy) {
  uint32_t m = 0;
#pragma unroll
  for (int j = 0; j < USV_B_OBSTACLES; ++j) m |= (fabsf(cy - s_oy[j]) <= kReach) ? (1u << j) : 0u;
  return m;
}
// min over the obstacles of `mask` of the centre distance, minus the radius  (d_multi_gemini.py:84-92).  torch.norm over a 2-vector
// evaluates sqrt(fma(y, y, x*x)) (ATen's sum-of-squares accumulation, CPU and CUDA): spelled out, because the occupancy is the sign
// of this and the repulsion term amplifies 1 ulp of it by ~1e3 next to an obstacle.  Restricted to `mask` the result is exact
// wherever it is below kReach - 0.5 and +inf-ish (>= that) elsewhere -- every consumer only distinguishes values below 1.2
// (occupancy: <= 0; repulsion: sdf - 0.5 < 0.7)
__device__ __forceinline__ float cell_sdf_masked(float cx, float cy, const float* s_ox, const float* s_oy, uint32_t mask) {
  float best = CUDART_INF_F;
  while (mask) {
    const int j = __ffs(mask) - 1;
    mask &= mask - 1;
    const float dx = __fsub_rn(cx, s_ox[j]), dy = __fsub_rn(cy, s_oy[j]);
    best = fminf(best, sqrtf(__fmaf_rn(dy, dy, __fmul_rn(dx, dx))));
  }
  return __fsub_rn(best, kObstR);
}

// stage the 16 obstacle centres + target of scene j in smem (s_sc[0..15]=x, [16..31]=y, [32]=tx, [33]=ty); returns env id
__device__ __forceinline__ int64_t load_scene(const SceneIO& io, int64_t j, float* s_sc) {
  const int64_t env = io.list ? (int64_t)io.list[j] : j;
  if (threadIdx.x < USV_B_OBSTACLES) {
    const int t = threadIdx.x;
    if (io.list) {
      const float* bc = io.bconsts + tile_base(env, USV_BC_COUNT);
      s_sc[t] = bc[(USV_BC_OBST + 2 * t) * kTile];
      s_sc[16 + t] = bc[(USV_BC_OBST + 2 * t + 1) * kTile];
    } else {
      s_sc[t] = io.obstacles[(j * USV_B_OBSTACLES + t) * 2];
      s_sc[16 + t] = io.obstacles[(j * USV_B_OBSTACLES + t) * 2 + 1];
    }
  } else if (threadIdx.x == 32) {
    if (io.list) {
      const float* c = io.consts + tile_base(env, USV_C_COUNT);
      s_sc[32] = c[USV_C_TX * kTile];
      s_sc[33] = c[USV_C_TY * kTile];
    } else {
      s_sc[32] = io.targets[j * 2];
      s_sc[33] = io.targets[j * 2 + 1];
    }
  }
  return env;
}

// get_spawns obstacle placement for one env by warp 0 (lanes 0..15 = obstacles)  [ref :970-1047]
__device__ __forceinline__ void place_obstacles(const UsvStepParams& p, uint64_t step, uint64_t gid, float tx, float ty, float& ox, float& oy) {
  const int j = threadIdx.x & 31;
  const Uniform4 r0 = philox_uniform4(p.seed, gid, step, RS_RESET_0);
  float sx, sy;
  spawn_xy(p, r0, tx, ty, sx, sy);  // the same draw reset_env() of the step kernel will use for the pose
  const float mnx = tx - 12.0f, mny = ty - 12.0f;
  const float spx = (tx + 12.0f) - mnx, spy = (ty + 12.0f) - mny;
  auto draw = [&](int round) {
    const Uniform4 u = philox_uniform4(p.seed, gid, step, RS_OBST + (uint32_t)round * 8u + (uint32_t)((j & 15) >> 1));
    ox = __fadd_rn(__fmul_rn((j & 1) ? u.c : u.a, spx), mnx);  // rand * (max - min) + min: two roundings, as torch
    oy = __fadd_rn(__fmul_rn((j & 1) ? u.d : u.b, spy), mny);
  };
  auto invalid = [&]() {
    const float dsx = ox - sx, dsy = oy - sy, dtx = ox - tx, dty = oy - ty;
    bool inv = (sqrtf(__fmaf_rn(dsy, dsy, __fmul_rn(dsx, dsx))) < 3.0f) || (sqrtf(__fmaf_rn(dty, dty, __fmul_rn(dtx, dtx))) < 3.0f);
    const bool vj = ox < 900.0f;
#pragma unroll
    for (int i = 0; i < USV_B_OBSTACLES; ++i) {
      const float xi = __shfl_sync(0xffffffffu, ox, i), yi = __shfl_sync(0xffffffffu, oy, i);
      const float ddx = ox - xi, ddy = oy - yi;
      // S1: only the higher index of a conflicting pair is re-drawn
      if (i < j && vj && xi < 900.0f && __fadd_rn(__fmul_rn(ddx, ddx), __fmul_rn(ddy, ddy)) < 2.5f * 2.5f) inv = true;
    }
    return inv && j < USV_B_OBSTACLES;
  };
  draw(0);
  for (int it = 0; it < 20; ++it) {
    const bool inv = invalid();
    if (!(__ballot_sync(0xffffffffu, inv) & 0xffffu)) break;
    if (inv) draw(it + 1);
  }
  if (invalid()) { ox = 999.0f; oy = 999.0f; }  // leftovers go to limbo
}

// ---- cost-to-go -------------------------------------------------------------------------------------------------------------
// The reference's 225 Jacobi sweeps converge to the greatest fixed point of  d(c) = min(d(c), min_nb fl(d(nb) + w))  with d = 0 at the
// target; fl(d + w) is monotone in d, so ANY fair asynchronous (chaotic) iteration from +inf reaches the same fixed point bit for
// bit.  That licenses an in-place relaxation: ONE 150x150 buffer per scene (94 KB instead of 185 KB: two scenes per SM, which removes
// the second wave of the typical ~150 resets per control step on 148 SMs), relaxed tile by tile (8 columns x 32 rows; inside a lane's 8
// rows a pass walks down and back up feeding each new value into the next row), a warp staying on its tile until it stops changing
// before the CTA meets at the sweep barrier; tiles whose inputs did not change are skipped, and the scene ends at the first sweep
// without a change.  The 225th Jacobi iterate IS the fixed point whenever every shortest path has <= 225 hops; a hop
// costs >= 1, so "max finite cost < 224" proves it.  Otherwise (or when the target cell is not free: its 0 is overwritten after one
// Jacobi sweep, which an asynchronous order does not reproduce) the scene is redone by literal Jacobi sweeps through a global scratch
// (the env's own field slot) -- never seen with the task's obstacle placement, covered by a dense-batch test.
constexpr int kCostThreads = 512, kCostWarps = kCostThreads / 32;
constexpr int kAsyncSweepCap = 4 * kMaxSweeps;
constexpr int kInner = 16;            // passes of a warp over its tile per outer sweep (a value crosses a tile in <= 8; 12..32 time alike)
constexpr float kJacobiSafeCost = 224.0f;

__device__ __forceinline__ float block_reduce_max_cost(float v, float* s_red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) s_red[warp] = v;
  __syncthreads();
  v = (lane < kCostWarps) ? s_red[lane] : -CUDART_INF_F;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// cost-independent part of the repulsion of one cell: dist_to_edge = sdf - obstacle_radius (d_multi_gemini.py:220) and 20 q^2 with
// q = 1/d - 1/0.7 inside the influence radius (0 outside)
struct CellGeom { float edge, raw; };
__device__ __forceinline__ CellGeom cell_geom(float sdf) {
  CellGeom g;
  g.edge = __fsub_rn(sdf, kObstR);
  g.raw = 0.0f;
  if (g.edge < 0.7f) {
    const float dcl = fmaxf(g.edge, 1e-3f);
    const float q = __fsub_rn(__fdiv_rn(1.0f, dcl), 1.42857146f);  // 1.0/d - fp32(1/0.7)
    g.raw = __fmul_rn(20.0f, __fmul_rn(q, q));
  }
  return g;
}
// rep = clamp(G * 0.2 / 3, 0, 1): the factor that ties the repulsion to the cost-to-go
__device__ __forceinline__ float cell_rep(float vis) { return fminf(fmaxf(__fdiv_rn(__fmul_rn(vis, 0.2f), 3.0f), 0.0f), 1.0f); }

__device__ __forceinline__ bool cell_free(const unsigned char* s_free, int x, int y) {
  return (s_free[((y / kTileH) * kChunks + x / kTileW) * 32 + ((y % kTileH) / kBandRows) * kTileW + x % kTileW] >> (y % kBandRows)) & 1u;
}

// literal Jacobi sweeps (d_multi_gemini.py:160-190): cur = buf (shared), nxt = tmp (global), early exit at the first unchanged sweep
__device__ void jacobi_exact(float* buf, float* __restrict__ tmp, const unsigned char* s_free, int txi, int tyi) {
  for (int q = threadIdx.x; q < kGPR * kGS; q += kCostThreads) buf[q] = CUDART_INF_F;
  __syncthreads();
  if (threadIdx.x == 0) buf[(tyi + 1) * kGS + txi + 1] = 0.0f;
  __syncthreads();
  for (int sweep = 0; sweep < kMaxSweeps; ++sweep) {
    int chg = 0;
    for (int cell = threadIdx.x; cell < kCells; cell += kCostThreads) {
      const int y = cell / kG, x = cell - y * kG;
      const float* c = buf + (y + 1) * kGS + x + 1;
      const float mc = c[0];
      float best = CUDART_INF_F;
      if (cell_free(s_free, x, y)) {
        const float a = fminf(fminf(c[-1], c[1]), fminf(c[-kGS], c[kGS])) + 1.0f;
        const float b = fminf(fminf(c[-kGS - 1], c[-kGS + 1]), fminf(c[kGS - 1], c[kGS + 1])) + 1.414f;
        best = fminf(mc, fminf(a, b));
      }
      tmp[cell] = best;
      chg |= (best != mc) ? 1 : 0;
    }
    const int any = __syncthreads_or(chg);
    for (int cell = threadIdx.x; cell < kCells; cell += kCostThreads) {
      const int y = cell / kG, x = cell - y * kG;
      buf[(y + 1) * kGS + x + 1] = tmp[cell];
    }
    __syncthreads();
    if (!any) break;
  }
}

__global__ void __launch_bounds__(kCostThreads, 2) scene_cost_kernel(SceneIO io, uint32_t* __restrict__ counters, int place,
                                                                     const __grid_constant__ UsvStepParams p,
                                                                     const uint64_t* __restrict__ step_offset) {
  const uint64_t step = p.step_counter + (step_offset ? *step_offset : 0ull);   // device-side addend: CUDA-graph replays
  extern __shared__ __align__(16) float smem[];
  float* buf = smem;                  // padded 152 x 152, +inf halo
  float* s_sc = buf + kGPR * kGS;     // 34 floats
  float* s_red = s_sc + 64;           // 32 floats
  int* s_act = reinterpret_cast<int*>(s_red + 32);        // [2][96] tile-active flags of the current / next sweep
  uint32_t* s_rowmask = reinterpret_cast<uint32_t*>(s_act + 2 * kActStride);  // [150] obstacles that can matter on a grid row
  uint32_t* s_colmask = s_rowmask + 160;                                      // [150] ... on a grid column
  unsigned char* s_free = reinterpret_cast<unsigned char*>(s_colmask + 160);  // [95][32] free bits of a lane's 8 cells of a tile
  unsigned short* s_near = reinterpret_cast<unsigned short*>(s_free + kTiles * 32);   // [kNearCap] cells within reach of an obstacle
  int* s_nnear = reinterpret_cast<int*>(s_red + 31);                          // their count (s_red holds 16 partials)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t total = scene_count(io);
  for (int64_t j = blockIdx.x; j < total; j += gridDim.x) {
    int64_t env = io.list ? (int64_t)io.list[j] : j;
    if (place) {
      // B5: re-draw the obstacles of this env (list mode only), publish them to bconsts and smem
      if (warp == 0) {
        const float* c = io.consts + tile_base(env, USV_C_COUNT);
        const float tx = c[USV_C_TX * kTile], ty = c[USV_C_TY * kTile];
        float ox = 0.0f, oy = 0.0f;
        place_obstacles(p, step, (uint64_t)(p.env_id_offset + env), tx, ty, ox, oy);
        if (lane < USV_B_OBSTACLES) {
          float* bc = io.bconsts + tile_base(env, USV_BC_COUNT);
          bc[(USV_BC_OBST + 2 * lane) * kTile] = ox;
          bc[(USV_BC_OBST + 2 * lane + 1) * kTile] = oy;
          s_sc[lane] = ox;
          s_sc[16 + lane] = oy;
        }
        if (lane == 0) { s_sc[32] = tx; s_sc[33] = ty; }
      }
    } else {
      env = load_scene(io, j, s_sc);
    }
    {                                      // +inf everywhere, halo and spare rows included (16-byte stores; kGPR * kGS = 23 562 words)
      const float4 inf4 = make_float4(CUDART_INF_F, CUDART_INF_F, CUDART_INF_F, CUDART_INF_F);
      float4* b4 = reinterpret_cast<float4*>(buf);
      for (int q = threadIdx.x; q < (kGPR * kGS) / 4; q += kCostThreads) b4[q] = inf4;
      if (threadIdx.x < (kGPR * kGS) % 4) buf[((kGPR * kGS) / 4) * 4 + threadIdx.x] = CUDART_INF_F;
    }
    if (threadIdx.x < 2 * kActStride) s_act[threadIdx.x] = 0;
    if (threadIdx.x == 0) *s_nnear = 0;
    __syncthreads();
    // an obstacle within kReach of a cell is within kReach of its row AND of its column: the AND of the two masks leaves the one
    // or two obstacles a cell can feel (none for most cells)
    if (threadIdx.x < kG) s_rowmask[threadIdx.x] = row_obstacle_mask(io.lin[threadIdx.x], s_sc + 16);
    else if (threadIdx.x >= 256 && threadIdx.x < 256 + kG) s_colmask[threadIdx.x - 256] = row_obstacle_mask(io.lin[threadIdx.x - 256], s_sc);
    // target cell: ((pos + map/2) / cell).long().clamp(0, 149)   (d_multi_gemini.py:148-155)
    const int txi = min(max((int)__fdiv_rn(s_sc[32] + 15.0f, 0.2f), 0), kG - 1);
    const int tyi = min(max((int)__fdiv_rn(s_sc[33] + 15.0f, 0.2f), 0), kG - 1);
    if (threadIdx.x == 0) {
      buf[(tyi + 1) * kGS + txi + 1] = 0.0f;
      const int tc = txi / kTileW, tb = tyi / kTileH;
      for (int db = -1; db <= 1; ++db)
        for (int dc = -1; dc <= 1; ++dc)
          if (tc + dc >= 0 && tc + dc < kChunks && tb + db >= 0 && tb + db < kBands) s_act[(tb + db) * kChunks + tc + dc] = 1;
    }
    __syncthreads();
    // free bits of the 95 tiles (dealt round-robin to the warps, so that the ring of tiles the wavefront is crossing is spread over
    // all of them): one byte per lane = its 8 rows
    for (int t = warp; t < kTiles; t += kCostWarps) {
      const int chunk = t % kChunks, band = t / kChunks;
      const int x = chunk * kTileW + (lane & 7), y0 = band * kTileH + (lane >> 3) * kBandRows;
      uint32_t fm = 0;
      if (x < kG) {
        const uint32_t cmask = s_colmask[x];
        const float cx = io.lin[x];
#pragma unroll
        for (int i = 0; i < kBandRows; ++i) {
          const int y = y0 + i;
          if (y >= kG) break;
          const bool border = (y == 0) || (y == kG - 1) || (x == 0) || (x == kG - 1);
          const uint32_t mask = s_rowmask[y] & cmask;
          if (mask) {                                  // the statistics pass walks these densely
            const int k = atomicAdd(s_nnear, 1);
            if (k < kNearCap) s_near[k] = (unsigned short)(y * kG + x);
          }
          const float sdf = cell_sdf_masked(cx, io.lin[y], s_sc, s_sc + 16, mask);
          if (!border && !(sdf <= 0.0f)) fm |= 1u << i;
        }
      }
      s_free[t * 32 + lane] = (unsigned char)fm;
    }
    __syncthreads();
    bool exact = cell_free(s_free, txi, tyi);      // CTA-uniform
    if (exact) {
      int sweep = 0;
      for (; sweep < kAsyncSweepCap; ++sweep) {
        int* act_cur = s_act + (sweep & 1) * kActStride;
        int* act_nxt = s_act + ((sweep + 1) & 1) * kActStride;
        int any_change = 0;
        for (int t = warp; t < kTiles; t += kCostWarps) {
          if (!act_cur[t]) continue;                 // warp-uniform
          __syncwarp();
          if (lane == 0) act_cur[t] = 0;             // consumed; writers of this sweep only touch act_nxt
          const int chunk = t % kChunks, band = t / kChunks;
          const int cxl = lane & 7, grp = lane >> 3;
          const int x = chunk * kTileW + cxl;
          const int y0 = min(band * kTileH + grp * kBandRows, kG - 6);   // a group wholly below the grid (no free bit) reads in bounds
          const int xc = min(x, kG - 1);
          const uint32_t freemask = s_free[t * 32 + lane];
          const int bot = min(band * kTileH + kTileH, kG) - 1 - y0;      // bit of the tile's bottom row in this lane's byte, if 0..7
          // Temporal blocking: the warp relaxes ITS tile up to kInner times (until it stops changing) before the CTA-wide barrier, so a
          // value crosses a whole tile per outer sweep instead of one cell (legal: any fair asynchronous order reaches the same fixed
          // point).
          bool e_left = false, e_right = false, e_up = false, e_dn = false, changed = false, more = true;
          for (int inner = 0; inner < kInner && more; ++inner) {
            // one pass over the tile: all 10 x 3 window values are loaded first -- unconditionally, the buffer carries two spare +inf
            // rows below the halo so that the last rows read in bounds -- then the 8 cells of the lane's column are relaxed from
            // registers, walking down and back up with each new value fed into the next row (the left / right columns stay as loaded).
            // No branch: a lane outside the grid or a row below it has no free bit, so the mask alone gates the store.  (With guarded
            // loads and a per-row `if (free)` the compiler sank every row's loads behind a divergent branch of the row before: ~1100
            // cycles per pass in the r02 instrumented run against ~200 instructions.)
            const float* rp = buf + y0 * kGS + xc + 1;    // padded row y0 == grid row y0 - 1
            float wl[kBandRows + 2], wc[kBandRows + 2], wr[kBandRows + 2], was[kBandRows];
#pragma unroll
            for (int r = 0; r < kBandRows + 2; ++r) {
              wl[r] = rp[r * kGS - 1];
              wc[r] = rp[r * kGS];
              wr[r] = rp[r * kGS + 1];
            }
#pragma unroll
            for (int i = 0; i < kBandRows; ++i) {         // down
              was[i] = wc[i + 1];
              const float a = fminf(fminf(wl[i + 1], wr[i + 1]), fminf(wc[i], wc[i + 2])) + 1.0f;
              const float b = fminf(fminf(wl[i], wr[i]), fminf(wl[i + 2], wr[i + 2])) + 1.414f;
              const float best = fminf(wc[i + 1], fminf(a, b));
              wc[i + 1] = ((freemask >> i) & 1u) ? best : wc[i + 1];
            }
            uint32_t chg = 0;
#pragma unroll
            for (int i = kBandRows - 1; i >= 0; --i) {    // and back up: only the row below can have moved since the walk down
              const float best = fminf(wc[i + 1], wc[i + 2] + 1.0f);
              if (i < kBandRows - 1) wc[i + 1] = ((freemask >> i) & 1u) ? best : wc[i + 1];
              const bool upd = wc[i + 1] != was[i];
              if (upd) buf[(y0 + i + 1) * kGS + xc + 1] = wc[i + 1];
              chg |= upd ? (1u << i) : 0u;
            }
            const uint32_t any_b = __ballot_sync(0xffffffffu, chg != 0u);
            more = any_b != 0u;
            if (more) {
              changed = true;
              e_left |= (any_b & 0x01010101u) != 0u;      // column 0 of any row group
              e_right |= (any_b & 0x80808080u) != 0u;     // column 7
              e_up |= __any_sync(0xffffffffu, grp == 0 && (chg & 1u)) != 0;
              e_dn |= __any_sync(0xffffffffu, bot >= 0 && bot < kBandRows && ((chg >> bot) & 1u)) != 0;
            }
            __syncwarp();
          }
          // activate for the next outer sweep exactly the tiles whose inputs changed: a neighbour when a cell on the shared edge
          // changed, this tile only if it ran out of passes while still changing
          if (changed) {
            any_change = 1;
            if (lane < 9) {
              const int dc = lane % 3 - 1, db = lane / 3 - 1;
              const bool self = dc == 0 && db == 0;
              const bool need = self ? more : ((dc == 0 || (dc < 0 ? e_left : e_right)) && (db == 0 || (db < 0 ? e_up : e_dn)));
              const int c2 = chunk + dc, b2 = band + db;
              if (need && c2 >= 0 && c2 < kChunks && b2 >= 0 && b2 < kBands) act_nxt[b2 * kChunks + c2] = 1;
            }
          }
        }
        if (!__syncthreads_or(any_change)) break;
      }
      exact = sweep < kAsyncSweepCap;
    }
    float* out = io.field + env * (int64_t)kCells;
    float mx = -1.0f, mn = CUDART_INF_F;
    int far_fin = 0, far_inf = 0;
    for (int pass = 0; pass < 2; ++pass) {
      if (pass == 1 || !exact) jacobi_exact(buf, out, s_free, txi, tyi);
      // raw cost -> field[env] (and the optional dense cost output); max finite cost
      mx = -1.0f;
      mn = CUDART_INF_F;
      far_fin = 0;
      far_inf = 0;
#pragma unroll 1
      for (int y = warp; y < kG; y += kCostWarps) {
        const uint32_t rmask = s_rowmask[y];
#pragma unroll
        for (int ci = 0; ci < kColIters; ++ci) {
          const int x = lane + 32 * ci;
          if (x < kG) {
            const float c = buf[(y + 1) * kGS + x + 1];
            out[y * kG + x] = c;
            if (io.cost_out) io.cost_out[j * (int64_t)kCells + y * kG + x] = c;
            const bool fin = c < CUDART_INF_F, far = (rmask & s_colmask[x]) == 0u;
            if (fin) { mx = fmaxf(mx, c); mn = fminf(mn, c); }
            far_fin |= (far && fin) ? 1 : 0;      // cells no obstacle reaches: repulsion 0, not inside
            far_inf |= (far && !fin) ? 1 : 0;
          }
        }
      }
      mx = block_reduce_max_cost(mx, s_red);
      if (pass == 1 || !exact || mx < kJacobiSafeCost) break;   // the fixed point is the 225th Jacobi iterate
    }
    // per-scene statistics for the field kernel + the batch maxima of the repulsion, from the converged costs still in shared memory.
    // Min / max cost and "is there a cell no obstacle reaches" came out of the write-out loop above; the distance / repulsion terms are
    // evaluated only for the queued cells that an obstacle does reach (~20 % of the grid), every lane busy.
    float jfmn = CUDART_INF_F, jfmx = -1.0f, jimn = CUDART_INF_F, jimx = -1.0f, jall_fin = 0.0f, jall_inf = 0.0f;
    int has_inf = far_inf, has_inside = 0;
    const int nnear = min(*s_nnear, kNearCap);
    for (int k = threadIdx.x; k < nnear; k += kCostThreads) {
      const int q = s_near[k];
      const int y = q / kG, x = q - y * kG;
      const float c = buf[(y + 1) * kGS + x + 1];
      const CellGeom g = cell_geom(cell_sdf_masked(io.lin[x], io.lin[y], s_sc, s_sc + 16, s_rowmask[y] & s_colmask[x]));
      const bool inside = g.edge <= 0.0f;
      has_inside |= inside ? 1 : 0;
      if (c < CUDART_INF_F) {
        const float J = (g.raw > 0.0f) ? __fmul_rn(g.raw, cell_rep(c)) : 0.0f;   // 0 * rep == 0: the division is skipped
        jall_fin = fmaxf(jall_fin, J);
        if (!inside) { jfmn = fminf(jfmn, J); jfmx = fmaxf(jfmx, J); }
      } else {
        has_inf = 1;
        jall_inf = fmaxf(jall_inf, g.raw);
        if (!inside) { jimn = fminf(jimn, g.raw); jimx = fmaxf(jimx, g.raw); }
      }
    }
    far_fin = __syncthreads_or(far_fin);
    far_inf = __syncthreads_or(far_inf);
    if (far_fin) { jfmn = fminf(jfmn, 0.0f); jfmx = fmaxf(jfmx, 0.0f); }   // the unreached-by-any-obstacle cells: J = 0 (20 q^2 = 0)
    if (far_inf) { jimn = fminf(jimn, 0.0f); jimx = fmaxf(jimx, 0.0f); }
    mn = -block_reduce_max_cost(-mn, s_red);
    jfmn = -block_reduce_max_cost(-jfmn, s_red);
    jfmx = block_reduce_max_cost(jfmx, s_red);
    jimn = -block_reduce_max_cost(-jimn, s_red);
    jimx = block_reduce_max_cost(jimx, s_red);
    jall_fin = block_reduce_max_cost(jall_fin, s_red);
    jall_inf = block_reduce_max_cost(jall_inf, s_red);
    has_inf = __syncthreads_or(has_inf);
    has_inside = __syncthreads_or(has_inside);
    if (threadIdx.x == 0) {
      float* st = io.stats + j * SS_WORDS;
      st[SS_MIN_COST] = mn;
      st[SS_MAX_COST] = mx;       // -1 when no cell is reachable
      st[SS_JFIN_MIN] = jfmn;
      st[SS_JFIN_MAX] = jfmx;
      st[SS_JINF_MIN] = jimn;
      st[SS_JINF_MAX] = jimx;
      st[SS_FLAGS] = __uint_as_float((has_inf ? SSF_HAS_INF : 0u) | (has_inside ? SSF_HAS_INSIDE : 0u) | (jfmx >= 0.0f ? SSF_HAS_JFIN : 0u) |
                                     (jimx >= 0.0f ? SSF_HAS_JINF : 0u));
      // non-negative floats order like their bit patterns
      if (mx >= 0.0f) {
        atomicMax(counters + CW_MAXCOST, __float_as_uint(mx));
        atomicOr(counters + CW_HAVE, 1u);
      }
      atomicMax(counters + CW_MAXJ, __float_as_uint(jall_fin));
      atomicMax(counters + CW_MAXJ_INF, __float_as_uint(jall_inf));
      if (has_inside) atomicOr(counters + CW_INSIDE, 1u);
    }
    __syncthreads();
  }
}

__device__ __forceinline__ float global_vis_inf(const uint32_t* counters, int have) {
  // max_val = cost[finite].max() over the BATCH (fallback 100), times 1.5
  const float max_val = have ? __uint_as_float(counters[CW_MAXCOST]) : 100.0f;
  return __fmul_rn(max_val, 1.5f);
}

// field[env] = (G - min G) / (max G - min G + 1e-6) + 0.5 (J - min J) / (max J - min J + 1e-6)  (d_multi_gemini.py:205-271), one cell per
// thread-iteration; a scene is cut into kFieldChunks row blocks so that ~150 scenes spread over every SM instead of one CTA each
constexpr int kFieldThreads = 256, kFieldChunks = 10, kFieldRows = kG / kFieldChunks;   // 15 rows = 2250 cells per item
static_assert(kFieldRows * kFieldChunks == kG, "row blocks must tile the grid");

__global__ void __launch_bounds__(kFieldThreads) scene_field_kernel(SceneIO io, const uint32_t* __restrict__ counters) {
  __shared__ float s_sc[64];
  __shared__ uint32_t s_rowmask[kFieldRows];
  __shared__ uint32_t s_colmask[kG];
  const int64_t total = scene_count(io);
  const float vis_inf = global_vis_inf(counters, counters[CW_HAVE] != 0u);
  const float rep_inf = cell_rep(vis_inf);
  // batch max of J before the inside override (:236): finite-cost cells as they are, unreachable ones scaled by their common rep
  const float cur_max = fmaxf(__uint_as_float(counters[CW_MAXJ]), __fmul_rn(__uint_as_float(counters[CW_MAXJ_INF]), rep_inf));
  const bool any_inside = counters[CW_INSIDE] != 0u;
  const float high = (cur_max > 1e-6f) ? __fmul_rn(cur_max, 10.0f) : 100.0f;
  for (int64_t item = blockIdx.x; item < total * kFieldChunks; item += gridDim.x) {
    const int64_t j = item / kFieldChunks;
    const int y0 = (int)(item - j * kFieldChunks) * kFieldRows;
    __syncthreads();                     // the previous item's readers of s_sc / s_rowmask are done
    const int64_t env = load_scene(io, j, s_sc);
    __syncthreads();
    if (threadIdx.x < kFieldRows) s_rowmask[threadIdx.x] = row_obstacle_mask(io.lin[y0 + threadIdx.x], s_sc + 16);
    else if (threadIdx.x >= 64 && threadIdx.x < 64 + kG) s_colmask[threadIdx.x - 64] = row_obstacle_mask(io.lin[threadIdx.x - 64], s_sc);
    // per-scene extrema from the cost kernel's statistics
    const float* st = io.stats + j * SS_WORDS;
    const uint32_t fl = __float_as_uint(st[SS_FLAGS]);
    float gmn = st[SS_MIN_COST], gmx = (st[SS_MAX_COST] >= 0.0f) ? st[SS_MAX_COST] : -CUDART_INF_F;
    if (fl & SSF_HAS_INF) { gmn = fminf(gmn, vis_inf); gmx = fmaxf(gmx, vis_inf); }
    float jmn = CUDART_INF_F, jmx = -CUDART_INF_F;
    if (fl & SSF_HAS_JFIN) { jmn = st[SS_JFIN_MIN]; jmx = st[SS_JFIN_MAX]; }
    if (fl & SSF_HAS_JINF) { jmn = fminf(jmn, __fmul_rn(st[SS_JINF_MIN], rep_inf)); jmx = fmaxf(jmx, __fmul_rn(st[SS_JINF_MAX], rep_inf)); }
    if (fl & SSF_HAS_INSIDE) { jmn = fminf(jmn, high); jmx = fmaxf(jmx, high); }   // a scene with an inside cell makes any_inside true
    const float gden = __fadd_rn(__fsub_rn(gmx, gmn), 1e-6f), jden = __fadd_rn(__fsub_rn(jmx, jmn), 1e-6f);
    __syncthreads();
    float* f = io.field + env * (int64_t)kCells + y0 * kG;
    // all of the thread's costs are requested before the first one is used: one L2 round trip per item instead of three
    constexpr int kPer = (kFieldRows * kG + kFieldThreads - 1) / kFieldThreads;   // 9
    float cst[kPer];
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const int q = threadIdx.x + k * kFieldThreads;
      cst[k] = (q < kFieldRows * kG) ? f[q] : 0.0f;
    }
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const int q = threadIdx.x + k * kFieldThreads;
      if (q < kFieldRows * kG) {
        const int r = q / kG, x = q - r * kG;
        const float cost = cst[k];
        const float vis = (cost == CUDART_INF_F) ? vis_inf : cost;  // torch.where(isinf(cost), max_val*1.5, cost)
        const uint32_t mask = s_rowmask[r] & s_colmask[x];
        float J = 0.0f;
        if (mask) {            // most cells feel no obstacle: no distance, no repulsion
          const CellGeom g = cell_geom(cell_sdf_masked(io.lin[x], io.lin[y0 + r], s_sc, s_sc + 16, mask));
          if (g.raw > 0.0f) J = __fmul_rn(g.raw, (cost == CUDART_INF_F) ? rep_inf : cell_rep(cost));
          if (any_inside && g.edge <= 0.0f) J = high;
        }
        const float gn = __fdiv_rn(__fsub_rn(vis, gmn), gden);
        const float jd = __fsub_rn(J, jmn);
        const float jn = (jd == 0.0f) ? 0.0f : __fdiv_rn(jd, jden);   // +0 / jden == +0 (jden >= 1e-6): the division is skipped
        f[q] = __fadd_rn(gn, __fmul_rn(0.5f, jn));
      }
    }
  }
}

// reset_buf -> compact list of env ids (order irrelevant: scenes are independent, the batch maxima commutative)
__global__ void compact_resets_kernel(const int64_t* __restrict__ reset_buf, int64_t n, int32_t* __restrict__ list,
                                      uint32_t* __restrict__ counters) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (reset_buf[i] != 0) list[atomicAdd(counters + CW_COUNT, 1u)] = (int32_t)i;
  }
}

static size_t cost_smem_bytes() { return (size_t)(kGPR * kGS + 64 + 32 + 2 * kActStride + 160 + 160) * sizeof(float) + (size_t)kTiles * 32 + (size_t)kNearCap * 2; }

static int launch_scene(const SceneIO& io, uint32_t* counters, int place, const UsvStepParams* p, const uint64_t* step_offset,
                        cudaStream_t s) {
  ensure_dynamic_smem(scene_cost_kernel, cost_smem_bytes());
  const int grid = num_sms();
  scene_cost_kernel<<<2 * grid, kCostThreads, cost_smem_bytes(), s>>>(io, counters, place, *p, step_offset);   // two scenes per SM
  scene_field_kernel<<<8 * grid, kFieldThreads, 0, s>>>(io, counters);
  return finish_launch(2);
}

}  // namespace usv

using namespace usv;

extern "C" {

// workspace: [CW_WORDS counters][n int32 reset list, padded to 16 B][n x SS_WORDS per-scene statistics]
static int64_t stats_offset_bytes(int64_t n) { return (int64_t)CW_WORDS * 4 + (((n < 0 ? 0 : n) * 4 + 15) & ~(int64_t)15); }
int64_t usv_live_scene_workspace_bytes(int64_t n) { return stats_offset_bytes(n) + (n < 0 ? 0 : n) * (int64_t)(SS_WORDS * 4); }

int usv_live_reset_scene_f32(const UsvEnvBuffers* b, const UsvLiveBuffers* lb, const float* cell_centres, void* workspace,
                             int64_t n, const UsvStepParams* p, void* stream) {
  if (!b || !lb || !p || !cell_centres || !workspace) return USV_E_NULL;
  if (n < 0 || n > 0x7fffffffLL) return USV_E_SIZE;
  if (!b->consts || !b->reset_buf || !lb->bconsts || !lb->field) return USV_E_NULL;
  if (b->consts_stride < n || lb->bconsts_stride < n || (b->consts_stride & 31) || (lb->bconsts_stride & 31)) return USV_E_SIZE;
  if ((uintptr_t)workspace & 15) return USV_E_ALIGN;
  if (n == 0) return USV_OK;
  cudaStream_t s = (cudaStream_t)stream;
  uint32_t* counters = (uint32_t*)workspace;
  int32_t* list = (int32_t*)(counters + CW_WORDS);
  cudaMemsetAsync(counters, 0, CW_WORDS * sizeof(uint32_t), s);
  const int cgrid = (int)((n + 255) / 256 < 1184 ? (n + 255) / 256 : 1184);
  compact_resets_kernel<<<cgrid, 256, 0, s>>>(b->reset_buf, n, list, counters);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  SceneIO io{};
  io.list = list;
  io.count = counters + CW_COUNT;
  io.bconsts = lb->bconsts;
  io.consts = b->consts;
  io.field = lb->field;
  io.lin = cell_centres;
  io.stats = (float*)((char*)workspace + stats_offset_bytes(n));
  return launch_scene(io, counters, 1, p, b->step_offset, s);
}

int usv_live_build_fields_f32(const float* obstacles, const float* targets, const float* cell_centres, float* field,
                              float* cost_out, void* workspace, int64_t m, void* stream) {
  if (!obstacles || !targets || !cell_centres || !field || !workspace) return USV_E_NULL;
  if (m < 0) return USV_E_SIZE;
  if ((uintptr_t)workspace & 15) return USV_E_ALIGN;
  if (m == 0) return USV_OK;
  cudaStream_t s = (cudaStream_t)stream;
  uint32_t* counters = (uint32_t*)workspace;
  cudaMemsetAsync(counters, 0, CW_WORDS * sizeof(uint32_t), s);
  SceneIO io{};
  io.obstacles = obstacles;
  io.targets = targets;
  io.m = m;
  io.field = field;
  io.cost_out = cost_out;
  io.lin = cell_centres;
  io.stats = (float*)((char*)workspace + stats_offset_bytes(m));
  UsvStepParams p{};
  return launch_scene(io, counters, 0, &p, nullptr, s);
}

}  // extern "C"
