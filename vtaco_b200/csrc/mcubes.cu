// GPU marching cubes over the decoded logit grid (sm_100a).
//
// Replaces the skimage.measure.marching_cubes call + vertex rescale of
// Generator3D.generate_obj_mesh_wnf (reference src/conv_onet/generation.py:268-272).
// Contract and conventions: oracle/marching_cubes.py / oracle/mc_tables.py (the
// triangulation table is generated from the rule stated there; skimage's Lewiner tables
// are not available offline — parity with skimage is UNPINNED, parity with the oracle is
// bit-exact on case indices / faces and to rounding on vertices).
//
// HBM-bound stream compaction in TWO kernels; only the first streams the grid:
//   mc_fused_kernel : 1 thread / 4 runs of 8 consecutive z points — four rows of 9 samples as float4
//              loads -> "above" bit rows -> per point 3-bit own-edge mask + triangle count; the four
//              runs are classified back to back (all loads in flight) and scanned together (two
//              block barriers); the block's exclusive prefix comes from a DECOUPLED LOOK-BACK over
//              the blocks before it (single pass, blocks take their index from a ticket so that
//              every predecessor has started); the kernel stores codes + vertex base of the active
//              runs and appends them, with their triangle base, to a work list.  No emission here:
//              a warp is one z-row of the lattice, and rows that the surface crosses in one or two
//              places ran the 8 x 3 double-precision emission loop for one or two lanes.
//   mc_emit_kernel : grid-stride over the work list only (~6 % of the runs, every lane busy): the
//              vertices of the run's own cut edges (inverse-distance weighting in double, like
//              Lewiner's code) and the faces of its cut cells; vertex ids are looked up from the
//              owners' codes / bases; output order = lattice order, then table order (the order
//              of the WORK is arbitrary, every item carries its output positions).
// Slab mode (x_emit < nx; multi-GPU extraction, SURVEY 8e "gather of mesh pieces"): the volume
// holds the rank's x-rows plus two halo rows; vertex ids are numbered over the whole volume (so a
// halo-row vertex gets the id it has as the NEXT rank's first vertices), but only vertices owned
// by rows < x_emit and faces of cells in rows < x_emit are emitted and counted.  The pieces of
// consecutive slabs then concatenate to exactly the single-volume mesh (ids + the vertex base of
// the slab).
// Batched mode (n_volumes > 1 or scene_counts): B contiguous volumes are one stacked volume of B*nx
// rows.  A run takes the level of its scene (row / nx); the last row of a scene owns no cells and no
// x-edge (the rule slab mode applies to halo rows), so no vertex or face joins two scenes.  The
// look-back prefix at a scene's first run is its vertex / face base: the emit pass subtracts the
// vertex base from face ids (ids local to the scene's vertex block) and writes the per-scene counts.
// The single-volume kernels are the BATCH = false instantiations, untouched by this mode.
// Algorithmic bytes: 4*n (grid) + 12*V + 12*F; scratch traffic adds the active blocks' codes
// and base ids.
#include "common.cuh"
#include "mc_tables.h"
#include <float.h>

namespace vtaco {

constexpr int kMcThreads = 256;   // threads per block
constexpr int kMcRun = 8;         // consecutive z points per thread

struct McParams {
  const float* grid;
  const float* halo;              // rows >= x_local are read from here (row r -> halo + (r - x_local) * ny * nz), or NULL
  int x_local;                    // rows of the sub-volume that live in `grid` (== nx without a separate halo)
  int nx, ny, nz, nzc;            // nzc = ceil(nz / kMcRun) runs per (x,y) row
  int nzc_shift, ny_shift;        // log2 when the extent is a power of two (run -> coordinates by shifts), else -1
  int vec_rows;                   // rows are read as float4: nz % 8 == 0 and grid / halo 16-byte aligned
  int x_emit;                     // rows [0, x_emit) emit vertices / faces (== nx: whole volume)
  int x_origin;                   // lattice row of the sub-volume's row 0 (vertex coordinates are global)
  long long npts, nruns;
  float level;
  const int32_t* level_keys;
  int n_level_keys;
  const float* level_ptr;
  uint8_t* code;                  // [nruns][8]: bits 0-2 own-edge mask (x,y,z), bits 3-5 triangle count (active runs only)
  uint32_t* vbase;                // [nruns]: id of the first vertex owned by the run (active runs only)
  unsigned long long* state;      // [nblocks] look-back words: flag << 62 | triangles << 31 | vertices (zeroed per call)
  uint2* work;                    // [nruns] (run, triangle base) of the runs that own triangles
  unsigned* ctrl;                 // [0] block ticket, [1] work-list length (zeroed per call)
  int nblocks, emit;
  long long* counts;
  float* verts;
  long long vcap;
  int32_t* faces;
  long long fcap;
  float voffset, vscale;
  // batched mode only
  int nxs;                        // rows per volume: row i belongs to scene i / nxs
  unsigned scene_runs;            // runs per volume (nxs * ny * nzc)
  int n_vol;
  unsigned long long* sbase;      // [n_vol][2] scratch: vertex / triangle base of each scene (prefix at its first run)
  long long* scene_counts;        // [n_vol][2]: (V, F) of each scene
};

// iso-level of scene s in batched mode: its own (min,max) key pair, else the one given level
__device__ __forceinline__ float scene_level(const McParams& P, int s) {
  if (P.level_keys) return 0.5f * (key_to_float(P.level_keys[2 * s]) + key_to_float(P.level_keys[2 * s + 1]));
  return P.level;
}

__device__ __forceinline__ float mc_level(const McParams& P) {
  if (P.level_ptr) return *P.level_ptr;
  if (P.level_keys) {
    int32_t lo = P.level_keys[0], hi = P.level_keys[1];
    for (int r = 1; r < P.n_level_keys; ++r) {
      lo = min(lo, P.level_keys[2 * r]);
      hi = max(hi, P.level_keys[2 * r + 1]);
    }
    return 0.5f * (key_to_float(lo) + key_to_float(hi));
  }
  return P.level;
}

// run -> lattice coordinates of its first point
__device__ __forceinline__ void run_coords(const McParams& P, long long run, int& i, int& j, int& k0) {
  const unsigned ru = (unsigned)run;           // nruns < 2^31 (checked by the host wrapper)
  const unsigned r = P.nzc_shift >= 0 ? ru >> P.nzc_shift : ru / (unsigned)P.nzc;
  const int kc = (int)(ru - r * (unsigned)P.nzc);
  i = (int)(P.ny_shift >= 0 ? r >> P.ny_shift : r / (unsigned)P.ny);
  j = (int)(r - (unsigned)i * (unsigned)P.ny);
  k0 = kc * kMcRun;
}

// z-row (i,j) of the sub-volume: the slab's own rows, or the halo rows kept elsewhere (the next rank's grid)
__device__ __forceinline__ const float* mc_row(const McParams& P, int i, int j) {
  return i < P.x_local ? P.grid + ((long long)i * P.ny + j) * P.nz
                       : P.halo + ((long long)(i - P.x_local) * P.ny + j) * P.nz;
}

// The one test of a corner against the level, in both kernels, so that a cell is emitted with the case it was counted
// with: IEEE sample > level.  The compare is ordered: a NaN on either side is not above, and +0 is not above -0 (a
// level of -0 selects what +0 does).
__device__ __forceinline__ bool above(float sample, float level) { return sample > level; }

// "above" bits of kMcRun+1 consecutive z samples of row (i,j), bit t <-> k0+t; rows or samples
// outside the lattice replicate the last valid sample (their cells/edges are masked out later).
__device__ __forceinline__ unsigned row_bits(const McParams& P, int i, int j, int k0, float level) {
  i = min(i, P.nx - 1);
  j = min(j, P.ny - 1);
  const float* row = mc_row(P, i, j);
  unsigned bits = 0;
  if (P.vec_rows) {        // uniform over the grid: the last run of a row takes this path too (a per-lane
                           // test sent one lane of EVERY warp through the scalar path below: 750 instructions per thread)
    const float4 a = __ldg(reinterpret_cast<const float4*>(row + k0));
    const float4 b = __ldg(reinterpret_cast<const float4*>(row + k0 + 4));
    const float c = __ldg(row + min(k0 + 8, P.nz - 1));
    // the bits by Horner's rule in float, highest sample first (exact below 2^24): a compare that yields 1.0f or 0
    // and an FMA per sample, where an integer shift-in takes a compare, a select and a shift
    float f = above(c, level);
    f = fmaf(f, 2.f, above(b.w, level));
    f = fmaf(f, 2.f, above(b.z, level));
    f = fmaf(f, 2.f, above(b.y, level));
    f = fmaf(f, 2.f, above(b.x, level));
    f = fmaf(f, 2.f, above(a.w, level));
    f = fmaf(f, 2.f, above(a.z, level));
    f = fmaf(f, 2.f, above(a.y, level));
    f = fmaf(f, 2.f, above(a.x, level));
    bits = (unsigned)f;
  } else {
#pragma unroll
    for (int t = 0; t <= kMcRun; ++t) bits |= (unsigned)above(__ldg(row + min(k0 + t, P.nz - 1)), level) << t;
  }
  return bits;
}

// codes of the 8 points of a run (see McParams::code); returns packed (ntris << 16 | nverts).
// Bit-parallel over the run: own-edge masks are XORs of the "above" rows and a cell is cut iff
// its 8 corner bits are neither all 0 nor all 1, so the ~95 % of runs that the surface does not
// touch cost a handful of logic ops; only the set bits take the per-point path.
// row_end: first row past the volume of row i (P.nx; batched mode: the end of the scene's rows).
__device__ __forceinline__ unsigned run_codes(const McParams& P, int i, int j, int k0, int row_end, unsigned r00,
                                               unsigned r10, unsigned r01, unsigned r11, unsigned long long& codes,
                                               const uint8_t* __restrict__ tri_count) {
  const bool hx = i + 1 < row_end, hy = j + 1 < P.ny;
  const int left = P.nz - k0;                                     // points of this run inside the lattice
  const unsigned m8 = left >= kMcRun ? 0xffu : ((1u << left) - 1u);
  const unsigned mz = left - 1 >= kMcRun ? 0xffu : ((1u << max(left - 1, 0)) - 1u);   // points with k+1 < nz
  const unsigned fx = hx ? ((r00 ^ r10) & m8) : 0u;
  const unsigned fy = hy ? ((r00 ^ r01) & m8) : 0u;
  const unsigned fz = (r00 ^ (r00 >> 1)) & mz;
  const unsigned any = r00 | r10 | r01 | r11, all = r00 & r10 & r01 & r11;
  // halo rows (i >= x_emit) keep their vertex flags (the numbering runs through them) but own no cells
  const unsigned cut = (hx && hy && i < P.x_emit) ? (((any | (any >> 1)) & ~(all & (all >> 1))) & mz) : 0u;
  codes = 0;
  unsigned todo = fx | fy | fz | cut;
  unsigned packed = __popc(fx) + __popc(fy) + __popc(fz);
  while (todo) {
    const int t = __ffs(todo) - 1;
    todo &= todo - 1;
    const unsigned flags = ((fx >> t) & 1u) | (((fy >> t) & 1u) << 1) | (((fz >> t) & 1u) << 2);
    unsigned nt = 0;
    if ((cut >> t) & 1u) {
      // corner c = x | y<<1 | z<<2
      const unsigned cs = ((r00 >> t) & 1u) | (((r10 >> t) & 1u) << 1) | (((r01 >> t) & 1u) << 2) |
                          (((r11 >> t) & 1u) << 3) | (((r00 >> (t + 1)) & 1u) << 4) | (((r10 >> (t + 1)) & 1u) << 5) |
                          (((r01 >> (t + 1)) & 1u) << 6) | (((r11 >> (t + 1)) & 1u) << 7);
      nt = (unsigned)tri_count[cs];     // shared-memory copy: a divergent __constant__ index is serialised per lane
    }
    codes |= (unsigned long long)(flags | (nt << 3)) << (8 * t);
    packed += nt << 16;
  }
  return packed;
}

constexpr unsigned long long kMcFlagAgg = 1ull << 62, kMcFlagPrefix = 2ull << 62, kMcValMask = (1ull << 62) - 1;

__device__ __forceinline__ unsigned long long ld_state(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_state(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// point (i,j,k) -> run index / slot within the run
__device__ __forceinline__ long long run_of(const McParams& P, int i, int j, int k) {
  return ((long long)i * P.ny + j) * P.nzc + (k >> 3);
}

constexpr int kMcSub = 4;                          // consecutive 256-run sub-blocks per CTA: 4x fewer look-back words
constexpr int kMcBlockRuns = kMcThreads * kMcSub;

// resident CTAs per SM the fused kernel is compiled for (40 registers; batched: 48) and launched with
constexpr int mc_fused_ctas_per_sm(bool batch) { return batch ? 5 : 6; }

template <bool BATCH>
__global__ void __launch_bounds__(kMcThreads, mc_fused_ctas_per_sm(BATCH)) mc_fused_kernel(const __grid_constant__ McParams P) {
  constexpr int kWarps = kMcThreads / 32;
  __shared__ int s_bid;
  __shared__ unsigned long long s_prefix;
  __shared__ uint8_t s_tricount[256];
  __shared__ unsigned s_wexcl[kMcSub * kWarps];
  __shared__ unsigned s_rows[kMcBlockRuns];
  s_tricount[threadIdx.x] = (uint8_t)__ldg(kMcTriCount + threadIdx.x);
  const float level = mc_level(P);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  // Resident CTAs draw 1 024-run blocks from a ticket counter until none is left (the grid is one wave: 2 048 blocks
  // on 6 x 148 slots were 2.3 waves, the last one a third full).  A block's index is its ticket, so every block before
  // it has been drawn by a CTA that is running: the look-back below cannot wait on work that has not started.
  for (;;) {
  __syncthreads();                                               // shared state of the previous block is no longer read
  if (threadIdx.x == 0) s_bid = (int)atomicAdd(P.ctrl, 1u);
  __syncthreads();
  const int b = s_bid;
  if (b >= P.nblocks) break;
  // ---- classify kMcSub runs per thread (run = block base + s * 256 + thread: coalesced, lattice order = (s, thread));
  //      no barrier between them, so the loads of all four runs are in flight together ----
  //      A run needs the "above" bits of rows (i,j), (i+1,j), (i,j+1), (i+1,j+1); the last two are the first two of
  //      run + nzc, which is a run of this block for all but its last nzc runs: every thread classifies its own two
  //      rows and takes the other two from shared memory (half the loads and compares).
  unsigned packed[kMcSub], inc[kMcSub];
  unsigned long long codes[kMcSub];
  unsigned own[kMcSub];                                          // r00 | r10 << 16
#pragma unroll
  for (int s = 0; s < kMcSub; ++s) {
    const long long run = (long long)b * kMcBlockRuns + s * kMcThreads + threadIdx.x;
    own[s] = 0;
    if (run < P.nruns) {
      int i, j, k0;
      run_coords(P, run, i, j, k0);
      const float lv = BATCH ? scene_level(P, i / P.nxs) : level;
      own[s] = row_bits(P, i, j, k0, lv) | (row_bits(P, i + 1, j, k0, lv) << 16);
    }
    s_rows[s * kMcThreads + threadIdx.x] = own[s];
  }
  __syncthreads();
#pragma unroll
  for (int s = 0; s < kMcSub; ++s) {
    const int local = s * kMcThreads + threadIdx.x;
    const long long run = (long long)b * kMcBlockRuns + local;
    packed[s] = 0;
    codes[s] = 0;
    if (run < P.nruns) {
      int i, j, k0;
      run_coords(P, run, i, j, k0);
      const int sc = BATCH ? i / P.nxs : 0;
      const float lv = BATCH ? scene_level(P, sc) : level;
      unsigned nxt;
      if (j + 1 >= P.ny) nxt = own[s];                           // replicated row: its cells / edges are masked out
      else if (local + P.nzc < kMcBlockRuns) nxt = s_rows[local + P.nzc];   // row (i, j+1): the same scene
      else nxt = row_bits(P, i, j + 1, k0, lv) | (row_bits(P, i + 1, j + 1, k0, lv) << 16);
      packed[s] = run_codes(P, i, j, k0, BATCH ? (sc + 1) * P.nxs : P.nx, own[s] & 0xffffu, own[s] >> 16,
                            nxt & 0xffffu, nxt >> 16, codes[s], s_tricount);
    }
  }
  // ---- one scan over the (s, thread) order: four independent warp scans, then the 32 warp totals in warp 0.
  //      fields: vertices < 2^16 (4 x 6144), triangles < 2^16 (4 x 10240) ----
#pragma unroll
  for (int s = 0; s < kMcSub; ++s) inc[s] = packed[s];
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
#pragma unroll
    for (int s = 0; s < kMcSub; ++s) {
      const unsigned t = __shfl_up_sync(0xffffffffu, inc[s], d);
      if (lane >= d) inc[s] += t;
    }
  }
  if (lane == 31) {
#pragma unroll
    for (int s = 0; s < kMcSub; ++s) s_wexcl[s * kWarps + w] = inc[s];
  }
  __syncthreads();
  unsigned total = 0;
  if (w == 0) {
    static_assert(kMcSub * kWarps == 32, "one lane per (sub-block, warp) total");
    const unsigned v = s_wexcl[lane];
    unsigned si = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned t = __shfl_up_sync(0xffffffffu, si, d);
      if (lane >= d) si += t;
    }
    s_wexcl[lane] = si - v;
    total = __shfl_sync(0xffffffffu, si, 31);
  }
  // ---- decoupled look-back (warp 0): exclusive prefix of this block over all blocks before it ----
  if (threadIdx.x < 32) {
    const unsigned long long agg = (unsigned long long)(total & 0xffffu) | ((unsigned long long)(total >> 16) << 31);
    unsigned long long prefix = 0;
    if (b > 0) {
      if (threadIdx.x == 0) st_state(P.state + b, kMcFlagAgg | agg);
      int base = b - 1;
      for (;;) {
        constexpr int kLb = 2;                                   // words per lane: 64 predecessors per round
        unsigned long long wd[kLb];
#pragma unroll
        for (int h = 0; h < kLb; ++h) {                          // lane l reads predecessors base - 32 h - l
          const int idx = base - 32 * h - (int)threadIdx.x;
          wd[h] = kMcFlagPrefix;                                 // before block 0: an empty prefix
          if (idx >= 0) wd[h] = ld_state(P.state + idx);
        }
        // a word that is not published yet ends the usable range of this round: everything nearer than the
        // nearest prefix word must be an aggregate, otherwise look again
        int first = kLb * 32, hole = kLb * 32;
#pragma unroll
        for (int h = kLb - 1; h >= 0; --h) {
          const unsigned pp = __ballot_sync(0xffffffffu, (wd[h] >> 62) == 2), zz = __ballot_sync(0xffffffffu, (wd[h] >> 62) == 0);
          if (pp) first = 32 * h + (__ffs(pp) - 1);
          if (zz) hole = 32 * h + (__ffs(zz) - 1);
        }
        if (hole < first) continue;                              // an unpublished predecessor nearer than the prefix: poll again
        unsigned long long v = 0;
#pragma unroll
        for (int h = 0; h < kLb; ++h)
          if (32 * h + (int)threadIdx.x <= first) v += wd[h] & kMcValMask;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
        prefix += v;
        if (first < kLb * 32) break;
        base -= kLb * 32;
      }
    }
    if (threadIdx.x == 0) {
      st_state(P.state + b, kMcFlagPrefix | (prefix + agg));
      s_prefix = prefix;
      if (b == P.nblocks - 1) {                                  // totals (slab mode: halo cells were classified empty)
        const unsigned long long tot = prefix + agg;
        P.counts[1] = (long long)(tot >> 31);
        P.counts[2] = (long long)(tot & 0x7fffffffull);
        if (P.x_emit >= P.nx) P.counts[0] = (long long)(tot & 0x7fffffffull);
      }
    }
  }
  __syncthreads();
  const unsigned long long pre = s_prefix;
  // ---- codes + vertex base of the active runs; every active run becomes one work item of the emit pass ----
#pragma unroll
  for (int s = 0; s < kMcSub; ++s) {
    const long long run = (long long)b * kMcBlockRuns + s * kMcThreads + threadIdx.x;
    if (run >= P.nruns) continue;
    const unsigned excl = s_wexcl[s * kWarps + w] + inc[s] - packed[s];
    const unsigned long long vb = (pre & 0x7fffffffull) + (excl & 0xffffu);
    const unsigned long long tb = (pre >> 31) + (excl >> 16);
    if (P.x_emit < P.nx && run == (long long)P.x_emit * P.ny * P.nzc) P.counts[0] = (long long)vb;   // first halo run
    if (BATCH && (unsigned)run % P.scene_runs == 0) {                // first run of a scene: its bases
      const unsigned sc = (unsigned)run / P.scene_runs;
      P.sbase[2 * sc] = vb;
      P.sbase[2 * sc + 1] = tb;
    }
    if (!packed[s]) continue;
    reinterpret_cast<unsigned long long*>(P.code)[run] = codes[s];
    P.vbase[run] = (uint32_t)vb;
    if (!P.emit) continue;
    const unsigned slot = atomicAdd(P.ctrl + 1, 1u);
    P.work[slot] = make_uint2((unsigned)run, (unsigned)tb);
  }
  }   // next ticket
}

// id of the vertex on axis `a` owned by point (i,j,k): the run's base + the vertices of the points before it
// in the run + the lower axes of the point itself
__device__ __forceinline__ int32_t vertex_id(const McParams& P, int i, int j, int k, int a) {
  const long long r = run_of(P, i, j, k);
  const unsigned long long codes = reinterpret_cast<const unsigned long long*>(P.code)[r];
  const int t = k & 7;
  const unsigned long long before = codes & ((1ull << (8 * t)) - 1ull) & 0x0707070707070707ull;
  const unsigned own = (unsigned)(codes >> (8 * t)) & 7u;
  return (int32_t)(P.vbase[r] + __popcll(before) + __popc(own & ((1u << a) - 1u)));
}

// Emit pass: EIGHT lanes per work item, lane t owns point t of the run — its (up to 3) vertices and the
// (up to 5) triangles of its cell.  One thread per run walked the 8 points serially through ~25 dependent
// global loads (59 us for the 6 % active runs of a 256^3 grid); here a lane's chain is work item -> codes ->
// grid samples -> neighbour codes / bases, and the samples of the run double as the vertex weights.
template <bool BATCH>
__global__ void __launch_bounds__(kMcThreads) mc_emit_kernel(const __grid_constant__ McParams P) {
  // case tables in shared memory: every lane indexes them with its own case (a divergent __constant__ index costs
  // one replay per distinct address); a case row is one 16-byte load
  __shared__ uint4 s_tri[256];
  __shared__ int8_t s_edge[12][4];
  {
    static_assert(kMcThreads == 256 && kMcMaxTris * 3 == 15, "one 16-byte case row per thread");
    s_tri[threadIdx.x] = __ldg(reinterpret_cast<const uint4*>(kMcTriTable) + threadIdx.x);
    if (threadIdx.x < 12) *reinterpret_cast<int*>(s_edge[threadIdx.x]) = __ldg(reinterpret_cast<const int*>(kMcEdge) + threadIdx.x);
  }
  __syncthreads();
  if (BATCH && blockIdx.x == 0) {   // per-scene counts: differences of consecutive scene bases (the last against the totals)
    for (int s = threadIdx.x; s < P.n_vol; s += kMcThreads) {
      const long long v1 = s + 1 < P.n_vol ? (long long)P.sbase[2 * s + 2] : P.counts[0];
      const long long f1 = s + 1 < P.n_vol ? (long long)P.sbase[2 * s + 3] : P.counts[1];
      P.scene_counts[2 * s] = v1 - (long long)P.sbase[2 * s];
      P.scene_counts[2 * s + 1] = f1 - (long long)P.sbase[2 * s + 1];
    }
  }
  const unsigned n_work = P.ctrl[1];
  const float level0 = mc_level(P);
  const int lane = threadIdx.x & 31, t = lane & 7;
  const unsigned warps_total = gridDim.x * (kMcThreads / 32);
  const unsigned warp_global = blockIdx.x * (kMcThreads / 32) + (threadIdx.x >> 5);
  for (unsigned base = warp_global * 4; base < n_work; base += warps_total * 4) {   // warp-uniform trip count
    const unsigned wi = base + (lane >> 3);
    const bool live = wi < n_work;
    const uint2 item = live ? P.work[wi] : make_uint2(0u, 0u);
    const long long run = item.x;
    const unsigned long long codes = live ? reinterpret_cast<const unsigned long long*>(P.code)[run] : 0ull;
    int i, j, k0;
    run_coords(P, run, i, j, k0);
    const int k = k0 + t;
    const int sc = BATCH ? i / P.nxs : 0;
    const float level = BATCH ? scene_level(P, sc) : level0;
    const double dlevel = (double)level;
    // samples of the four z-rows at this point (rows / samples outside the lattice replicate the last valid one,
    // as in row_bits: their cells / edges carry no flags)
    const int i1 = min(i + 1, P.nx - 1), j1 = min(j + 1, P.ny - 1), kc = min(k, P.nz - 1);
    const float* r00 = mc_row(P, i, j);
    const float* r10 = mc_row(P, i1, j);
    const float* r01 = mc_row(P, i, j1);
    const float* r11 = mc_row(P, i1, j1);
    const float g00 = __ldg(r00 + kc), g10 = __ldg(r10 + kc), g01 = __ldg(r01 + kc), g11 = __ldg(r11 + kc);
    // the samples one step up in z: the next lane's, except for the run's last point
    float n00 = __shfl_down_sync(0xffffffffu, g00, 1, 8), n10 = __shfl_down_sync(0xffffffffu, g10, 1, 8);
    float n01 = __shfl_down_sync(0xffffffffu, g01, 1, 8), n11 = __shfl_down_sync(0xffffffffu, g11, 1, 8);
    if (t == 7) {
      const int kn = min(k + 1, P.nz - 1);
      n00 = __ldg(r00 + kn); n10 = __ldg(r10 + kn); n01 = __ldg(r01 + kn); n11 = __ldg(r11 + kn);
    }
    const unsigned code = (unsigned)(codes >> (8 * t)) & 0xffu;
    const unsigned flags = code & 7u, nt = code >> 3;
    const unsigned long long below = codes & ((1ull << (8 * t)) - 1ull);
    // ---- vertices on the point's own cut edges (halo rows are numbered, not emitted) ----
    if (flags && i < P.x_emit) {
      unsigned long long vb = (unsigned long long)P.vbase[run] + (unsigned)__popcll(below & 0x0707070707070707ull);
      const double d0 = fabs((double)g00 - dlevel);
      const float pbase[3] = {(float)(BATCH ? i - sc * P.nxs : i + P.x_origin), (float)j, (float)k};
      const float nb[3] = {g10, g01, n00};                       // the neighbour along x, y, z
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        if (flags & (1u << a)) {
          if ((long long)vb < P.vcap) {    // capacity overflow: counted, not written (the caller re-runs with larger buffers)
            const double d1 = fabs((double)nb[a] - dlevel);
            // Lewiner's weights w = 1 / (eps + d): t = w1 / (w0 + w1) = (eps + d0) / ((eps + d0) + (eps + d1)), one
            // division instead of three (equal to the last bit or two of the double, far below the float32 result)
            // An infinite sample has weight 0, so the vertex sits at the other end, where e0 / (e0 + e1) is inf / inf
            const double e0 = (double)FLT_EPSILON + d0, e1 = (double)FLT_EPSILON + d1;
            const double tt = e0 == INFINITY && e1 < INFINITY ? 1.0 : e0 / (e0 + e1);
            float pos[3] = {pbase[0], pbase[1], pbase[2]};
            pos[a] = (float)((double)pbase[a] + tt);
            float* o = P.verts + vb * 3;
            o[0] = (pos[0] - P.voffset) * P.vscale;
            o[1] = (pos[1] - P.voffset) * P.vscale;
            o[2] = (pos[2] - P.voffset) * P.vscale;
          }
          ++vb;
        }
      }
    }
    // ---- triangles of the point's cell ----
    if (nt) {
      // corner c = x | y<<1 | z<<2
      const unsigned cs = (unsigned)above(g00, level) | ((unsigned)above(g10, level) << 1) |
                          ((unsigned)above(g01, level) << 2) | ((unsigned)above(g11, level) << 3) |
                          ((unsigned)above(n00, level) << 4) | ((unsigned)above(n10, level) << 5) |
                          ((unsigned)above(n01, level) << 6) | ((unsigned)above(n11, level) << 7);
      // triangle base of the cell: the run's + the triangle counts of the points before it (byte sum by multiplication)
      const unsigned long long tb = (unsigned long long)item.y +
          ((((below >> 3) & 0x1f1f1f1f1f1f1f1full) * 0x0101010101010101ull) >> 56);
      const uint4 row = s_tri[cs];
      for (unsigned tr = 0; tr < nt; ++tr) {
        if ((long long)(tb + tr) >= P.fcap) break;
        int32_t* o = P.faces + (tb + tr) * 3;
#pragma unroll
        for (int corner = 0; corner < 3; ++corner) {
          const int e = (int)((reinterpret_cast<const unsigned*>(&row)[(3 * tr + corner) >> 2] >> (8 * ((3 * tr + corner) & 3))) & 0xffu);
          const char4 ed = *reinterpret_cast<const char4*>(s_edge[e]);
          o[corner] = vertex_id(P, i + ed.y, j + ed.z, k + ed.w, ed.x) - (BATCH ? (int32_t)P.sbase[2 * sc] : 0);
        }
      }
    }
  }
}

// per-volume min / max of B volumes as ordered-int keys, merged into keys[2 b], keys[2 b + 1] (volume b =
// blockIdx.y): the reduction the decoder kernels perform on the logits they store, so the keys are the ones a
// single-scene decode of each volume produces.  A NaN orders beyond +-inf by its sign bit, so a volume that holds
// one has a NaN level.  vtaco_grid_minmax is the case B = 1.
__global__ void __launch_bounds__(256) volume_keys_kernel(const float* __restrict__ g, long long n,
                                                          int32_t* __restrict__ keys) {
  const float* v = g + (size_t)blockIdx.y * n;
  int32_t lo = INT32_MAX, hi = INT32_MIN;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int32_t k = float_to_key(v[i]);
    lo = min(lo, k);
    hi = max(hi, k);
  }
  lo = __reduce_min_sync(0xffffffffu, lo);
  hi = __reduce_max_sync(0xffffffffu, hi);
  if ((threadIdx.x & 31) == 0 && lo <= hi) {
    atomicMin(keys + 2 * blockIdx.y, lo);
    atomicMax(keys + 2 * blockIdx.y + 1, hi);
  }
}

__global__ void init_keys_kernel(int32_t* keys) {
  keys[0] = 0x7fffffff;
  keys[1] = (int32_t)0x80000000;
}

struct PeerTables { int32_t* t[8]; };
__global__ void publish_keys_kernel(int32_t* keys, PeerTables tabs, int n_peers, int rank) {
  const int32_t lo = keys[0], hi = keys[1];
  for (int r = 0; r < n_peers; ++r) {
    tabs.t[r][2 * rank] = lo;
    tabs.t[r][2 * rank + 1] = hi;
  }
  __threadfence_system();
  keys[0] = 0x7fffffff;
  keys[1] = (int32_t)0x80000000;
}

static long long mc_align(long long v) { return (v + 255) / 256 * 256; }

}  // namespace vtaco

using namespace vtaco;

extern "C" int64_t vtaco_mc_scratch_bytes(int32_t nx, int32_t ny, int32_t nz) {
  if (nx < 1 || ny < 1 || nz < 1) return VTACO_ERR_INVALID_ARG;
  const long long nruns = (long long)nx * ny * ((nz + kMcRun - 1) / kMcRun);
  const long long nb = (nruns + kMcThreads - 1) / kMcThreads;
  // codes (8 B / run), vertex base (4 B / run), work list (8 B / run), look-back state (8 B / block) + control words
  return mc_align(nruns * 8) + mc_align(4 * nruns) + mc_align(8 * nruns) + mc_align(8 * nb + 256);
}

extern "C" int64_t vtaco_mc_batch_scratch_bytes(int32_t n_volumes, int32_t nx, int32_t ny, int32_t nz) {
  if (n_volumes < 1 || nx < 1 || (long long)n_volumes * nx >= (1ll << 31)) return VTACO_ERR_INVALID_ARG;
  const int64_t b = vtaco_mc_scratch_bytes(n_volumes * nx, ny, nz);
  return b < 0 ? b : b + mc_align(16ll * n_volumes);
}

extern "C" int vtaco_volume_keys(const float* grid, int32_t n_volumes, int64_t n, int32_t* keys, void* stream) {
  if (!grid || !keys || n <= 0 || n_volumes < 1 || n_volumes > 65535) return VTACO_ERR_INVALID_ARG;
  long long blocks = (n + 255) / 256;
  long long cap = (long long)num_sms() * 8 / n_volumes;
  if (cap < 1) cap = 1;
  if (blocks > cap) blocks = cap;
  volume_keys_kernel<<<dim3((unsigned)blocks, (unsigned)n_volumes), 256, 0, (cudaStream_t)stream>>>(grid, n, keys);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

extern "C" int vtaco_grid_minmax(const float* grid, int64_t n, int32_t* keys, void* stream) {
  if (!grid || !keys || n <= 0) return VTACO_ERR_INVALID_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  init_keys_kernel<<<1, 1, 0, st>>>(keys);
  long long blocks = (n + 255) / 256;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  volume_keys_kernel<<<(unsigned)blocks, 256, 0, st>>>(grid, n, keys);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

extern "C" int vtaco_marching_cubes(const vtaco_mc_args* a, void* stream) {
  if (!a || !a->grid || !a->scratch || !a->counts) return VTACO_ERR_INVALID_ARG;
  if (a->nx < 1 || a->ny < 1 || a->nz < 1) return VTACO_ERR_INVALID_ARG;
  if (a->phase < 1 || a->phase > 3) return VTACO_ERR_INVALID_ARG;
  if (a->x_emit < 0 || a->x_emit > a->nx) return VTACO_ERR_INVALID_ARG;
  if (a->n_volumes < 0) return VTACO_ERR_INVALID_ARG;
  const bool batch = a->n_volumes > 1 || a->scene_counts;
  const int n_vol = a->n_volumes > 1 ? a->n_volumes : 1;
  if (batch && (!a->scene_counts || a->x_emit != 0 || a->x_origin != 0 || a->halo_rows != 0 || a->level_ptr ||
                a->n_level_keys > 1))
    return VTACO_ERR_INVALID_ARG;   // batched mode: whole volumes, one (min,max) pair or the level per volume
  const long long n = (long long)n_vol * a->nx * a->ny * a->nz;
  if (n >= (1ll << 31)) return VTACO_ERR_UNSUPPORTED;
  if ((batch ? vtaco_mc_batch_scratch_bytes(n_vol, a->nx, a->ny, a->nz) : vtaco_mc_scratch_bytes(a->nx, a->ny, a->nz)) >
      a->scratch_bytes)
    return VTACO_ERR_CAPACITY;
  if ((a->phase & 2) && ((a->vertex_capacity > 0 && !a->vertices) || (a->face_capacity > 0 && !a->faces)))
    return VTACO_ERR_INVALID_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  McParams P = {};
  if (a->halo_rows < 0 || a->halo_rows >= a->nx || (a->halo_rows > 0 && !a->halo_grid)) return VTACO_ERR_INVALID_ARG;
  P.grid = a->grid; P.nx = n_vol * a->nx; P.ny = a->ny; P.nz = a->nz; P.npts = n;
  P.halo = a->halo_rows > 0 ? a->halo_grid : nullptr;
  P.x_local = P.nx - a->halo_rows;
  P.x_emit = a->x_emit > 0 ? a->x_emit : P.nx;
  P.x_origin = a->x_origin;
  P.level = a->level; P.level_keys = a->level_keys; P.level_ptr = a->level_ptr;
  P.n_level_keys = a->n_level_keys > 1 ? a->n_level_keys : 1;
  P.nzc = (a->nz + kMcRun - 1) / kMcRun;
  // float4 row loads need 16-byte alignment; rows and runs start at multiples of 8 floats when nz % 8 == 0, so the
  // base pointers decide (any contiguous view is accepted, e.g. one starting one float into a buffer)
  P.vec_rows = (a->nz % kMcRun) == 0 && (reinterpret_cast<uintptr_t>(P.grid) & 15) == 0 &&
               (reinterpret_cast<uintptr_t>(P.halo) & 15) == 0;
  P.nzc_shift = P.ny_shift = -1;
  for (int sh = 0; sh < 31; ++sh) {
    if (P.nzc == (1 << sh)) P.nzc_shift = sh;
    if (P.ny == (1 << sh)) P.ny_shift = sh;
  }
  P.nruns = (long long)P.nx * a->ny * P.nzc;
  P.nblocks = (int)((P.nruns + kMcBlockRuns - 1) / kMcBlockRuns);
  char* s = reinterpret_cast<char*>(a->scratch);
  P.code = reinterpret_cast<uint8_t*>(s); s += mc_align(P.nruns * 8);
  P.vbase = reinterpret_cast<uint32_t*>(s); s += mc_align(4 * P.nruns);
  P.work = reinterpret_cast<uint2*>(s); s += mc_align(8 * P.nruns);
  P.state = reinterpret_cast<unsigned long long*>(s);
  P.ctrl = reinterpret_cast<unsigned*>(s + 8ll * P.nblocks);
  P.counts = reinterpret_cast<long long*>(a->counts);
  P.verts = a->vertices; P.vcap = a->vertex_capacity;
  P.faces = a->faces; P.fcap = a->face_capacity;
  P.voffset = a->voffset; P.vscale = a->vscale;
  if (batch) {
    P.nxs = a->nx;
    P.scene_runs = (unsigned)((long long)a->nx * a->ny * P.nzc);
    P.n_vol = n_vol;
    P.sbase = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(a->scratch) +
                                                    vtaco_mc_scratch_bytes(P.nx, P.ny, P.nz));
    P.scene_counts = reinterpret_cast<long long*>(a->scene_counts);
  }
  // phase 1 = count only (nothing is written to the outputs); 2 and 3 = the whole extraction (classification is
  // part of the same pass, so "emit after a count" simply runs it again with the larger buffers)
  P.emit = (a->phase & 2) ? 1 : 0;
  if (!P.emit) P.vcap = 0;
  VTACO_CUDA_CHECK(cudaMemsetAsync(P.state, 0, 8ll * P.nblocks + 16, st));
  {
    // 4.5 KB of shared memory: registers bound the CTAs per SM
    const int resident = num_sms() * mc_fused_ctas_per_sm(batch);
    const unsigned grid = P.nblocks < resident ? P.nblocks : resident;
    if (batch) mc_fused_kernel<true><<<grid, kMcThreads, 0, st>>>(P);
    else mc_fused_kernel<false><<<grid, kMcThreads, 0, st>>>(P);
  }
  if (P.emit || batch) {   // batched mode: the emit kernel also writes the per-scene counts (phase 1: one block, no work)
    long long blocks = (long long)num_sms() * 8;   // 8 lanes per work item; the kernel strides over the list
    if (blocks > (P.nruns * 8 + kMcThreads - 1) / kMcThreads) blocks = (P.nruns * 8 + kMcThreads - 1) / kMcThreads;
    if (!P.emit) blocks = 1;
    if (batch) mc_emit_kernel<true><<<(unsigned)blocks, kMcThreads, 0, st>>>(P);
    else mc_emit_kernel<false><<<(unsigned)blocks, kMcThreads, 0, st>>>(P);
  }
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

extern "C" int vtaco_publish_keys(int32_t* keys, int32_t* const* tables, int32_t n_peers, int32_t rank, void* stream) {
  if (!keys || !tables || n_peers < 1 || n_peers > 8 || rank < 0 || rank >= 8) return VTACO_ERR_INVALID_ARG;
  PeerTables t;
  for (int r = 0; r < 8; ++r) t.t[r] = r < n_peers ? tables[r] : nullptr;
  publish_keys_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(keys, t, n_peers, rank);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}
