// icp_tile.cuh -- EXPERIMENTAL (compiled with -DMVR_TS_TILE only): the two kernels of the fused ICP iteration on top of the
// block-cooperative tile search of tile_search.cuh.  Results are bit-identical to the per-thread kernels of icp.cu (all
// GPU parity tests pass with it), but on the bench workload (24 x 200k points) it is SLOWER: 1.27 ms per iteration against
// 0.72 ms (B200, round 2, profiles/r02_tile_search_experiment.txt).  Why, from ncu: a 1-D window through a staged ribbon
// still holds ~42 candidates per query (the ribbon's whole cross-section: three z slabs of cells), the same as the ~39 of
// the per-thread row walk, every candidate costs more than in registers, and the staging phases (ten block barriers, two
// block scans, eight-lane row loops) add ~39 warp-instructions per query.  Included from icp.cu inside namespace mvr.
#pragma once
#if defined(MVR_PG_XRATIO) && MVR_PG_XRATIO != 1
#error "the tile-search experiment assumes isotropic grid cells: build with -DMVR_PG_XRATIO=1"
#endif

template <bool RECIP, int EST>
__global__ void __launch_bounds__(FUSED_THREADS, (RECIP ? MVR_FWD_MINBLOCKS : MVR_FWD1_MINBLOCKS) * (256 / FUSED_THREADS)) k_icp_forward(const __grid_constant__ FwdBatch batch, int first) {
  // this pair's arguments: parameter space -> shared memory (a dynamically indexed parameter would be copied to
  // local memory and pin registers)
  __shared__ FwdArgs s_args;
  __shared__ TileSmem S;
  __shared__ int s_wcnt[FUSED_WARPS];
  __shared__ uint16_t s_open[FUSED_THREADS];
  static_assert(sizeof(FwdArgs) % 4 == 0 && sizeof(FwdArgs) / 4 <= FUSED_THREADS, "argument block");
  if (threadIdx.x < sizeof(FwdArgs) / 4) ((uint32_t*)&s_args)[threadIdx.x] = ((const uint32_t*)&batch.a[blockIdx.y])[threadIdx.x];
  __syncthreads();
  const FwdArgs& a = s_args;
  if ((int)blockIdx.x >= a.grid) return;
  IcpState* __restrict__ st = a.st;
  if (st->done) return;
  const int stride = a.grid * FUSED_THREADS;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint2* seg = reinterpret_cast<uint2*>(S.pts) + tid;   // the fallback's segment list lives in the tile's staging area
  Mat4f M;
  if (!first) {
#pragma unroll
    for (int k = 0; k < 16; ++k) M.m[k] = st->delta[k];
  }
  const float rscale = a.gt.inv_cell * 1.000001f;
  unsigned int ngate = 0;
  for (int base = blockIdx.x * FUSED_THREADS; base < a.n_valid; base += stride) {
    const int i = base + tid;
    const bool valid = i < a.n_valid;
    TileQuery me;
    me.near = false;
    me.qx = me.qy = me.qz = me.tx = me.ty = me.tz = me.rc = me.rho = 0.f;
    me.b = NnBest{MVR_INF, 0x7fffffff, -1};
    if (valid) {
      float4 p = a.cur[i];
      if (!first) {
        const float w = p.w;
        p = xform_pinned(M, p);
        p.w = w;
        a.cur[i] = p;
        if constexpr (EST == EST_SYM) a.nsrc[i] = rotate_pinned(M, a.nsrc[i]);
      }
      me.qx = p.x; me.qy = p.y; me.qz = p.z;
      fwd_seed(a, i, p, me.b);
      const float lim = fminf(me.b.d2, a.max_d2f);
      if (lim < MVR_INF) {
        me.tx = grid_t(p.x, a.gt.ox, a.gt.inv_cell); me.ty = grid_t(p.y, a.gt.oy, a.gt.inv_cell); me.tz = grid_t(p.z, a.gt.oz, a.gt.inv_cell);
        const float sq = sqrtf(lim);
        me.rc = sq * rscale + (MVR_CELL_MARGIN + 1.0e-6f * fmaxf(fabsf(me.tx), fmaxf(fabsf(me.ty), fabsf(me.tz))));
        me.rho = sq * 1.000001f;
        me.near = me.rc <= TS_RC_NEAR && a.m_valid > 0;
      }
    }
    bool open = valid;
    // no partner inside the gate so far: one bit says whether the target has anything within the gate of p's cell
    if (open && a.gmask && !(me.b.d2 <= a.max_d2f)) {
      const int cx = pg_cell(grid_t(me.qx, a.gt.ox, a.gt.inv_cell), a.gt.nx), cy = pg_cell(grid_t(me.qy, a.gt.oy, a.gt.inv_cell), a.gt.ny),
                cz = pg_cell(grid_t(me.qz, a.gt.oz, a.gt.inv_cell), a.gt.nz);
      const uint32_t wd = __ldg(a.gmask + ((size_t)cz * a.gt.ny + cy) * a.gm_stride + (cx >> 5));
      if (!((wd >> (cx & 31)) & 1u)) {
        open = false; me.near = false; a.corr_p[i] = -1;
#ifdef MVR_TS_STATS
        atomicAdd((unsigned long long*)&st->dbg[7], 1ull);
#endif
      }
    }
#if defined(MVR_TS_FIRST)
    const bool try_tile = true;
#else
    const bool try_tile = !first;   // the first iteration has no seeds: every ball is as wide as the gate
#endif
    const bool tiled = try_tile && tile_search(S, a.gt, a.tstart, a.tgt, min(a.n_valid - base, (int)FUSED_THREADS),
                                               [&](int, TileQuery& q, int) { q = me; },
                                               [&](int, const TileQuery& q) { if (q.skipped) me.near = false; else me.b = q.b; });
    if (open && me.near && tiled) { open = false; fwd_commit<RECIP>(a, i, me.b, ngate); }
    // ---- the rest: compacted, whole warps run the per-thread search
    const unsigned int bal = __ballot_sync(0xffffffffu, open);
    if (lane == 0) s_wcnt[warp] = __popc(bal);
    __syncthreads();   // also: every thread is done with the staged tile
    int ofs = 0, nopen = 0;
#pragma unroll
    for (int w = 0; w < FUSED_WARPS; ++w) { const int n = s_wcnt[w]; if (w < warp) ofs += n; nopen += n; }
#ifdef MVR_TS_STATS
    if (tid == 0) {
      if (nopen) atomicAdd((unsigned long long*)&st->dbg[3], (unsigned long long)nopen);
      if (try_tile && !tiled) atomicAdd((unsigned long long*)&st->dbg[4], 1ull);
    }
#endif
    if (nopen) {
      if (open) s_open[ofs + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)tid;
      __syncthreads();
      if (tid < nopen) {
        const int i2 = base + (int)s_open[tid];
        const float4 p2 = a.cur[i2];   // written by a thread of this block before the barrier
        NnBest b2;
        fwd_seed(a, i2, p2, b2);
        pg_search<MVR_PG_UNROLL>(a.gt, a.tstart, a.tgt, a.m_valid, p2.x, p2.y, p2.z, p2.x, p2.y, p2.z, 0.0f, 1.0f, a.max_d2f, b2, seg);
        fwd_commit<RECIP>(a, i2, b2, ngate);
      }
    }
    __syncthreads();   // the staging area and the counters are reused by the next round
  }
  if (RECIP) {
    const unsigned int wg = __reduce_add_sync(0xffffffffu, ngate);
    if (lane == 0 && wg) atomicAdd(&st->n_gate, wg);
  } else {
    // phase B: every thread sums over the points of its own index (their matches may have been written by another thread
    // of the block: the barrier at the end of the last round orders that)
    const double ox = st->ox, oy = st->oy, oz = st->oz;
    constexpr int NV = EstVals<EST>::value;
    double v[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) v[k] = 0.0;
    for (int i = blockIdx.x * FUSED_THREADS + threadIdx.x; i < a.n_valid; i += stride) {
      const int j = a.corr_p[i];
      if (j < 0) continue;
      const float4 p = a.cur[i];
      const float4 t = __ldg(a.tgt + j);
      acc_pair<EST>(v, p, t, a.nrm, a.nsrc + i, d2_pinned(p.x, p.y, p.z, t.x, t.y, t.z), ox, oy, oz);
    }
    reduce_and_finish<NV, EST == EST_SYM>(v, a.partials, st, a.log, a.grid);
  }
}

// Reciprocal half.  Only the target points some source point chose are searched: a block compacts the chosen ones
// of its `per` chunks of 256 target points (in order, deterministic) into a list in shared memory, answers the whole
// list from ONE tile (a thread owns queries k, k + 256, ...; per-thread search for what the tile cannot take), and every
// thread sums over its own mutual pairs afterwards.
#ifndef MVR_REV_MAX_CHUNKS
#define MVR_REV_MAX_CHUNKS 2
#endif
constexpr int REV_MAX_CHUNKS = MVR_REV_MAX_CHUNKS;
#ifndef MVR_TS_MIN_QUERIES
#define MVR_TS_MIN_QUERIES 32   // a list with fewer queries is not worth staging a tile for
#endif
template <int EST>
__global__ void __launch_bounds__(FUSED_THREADS, MVR_REV_MINBLOCKS * (256 / FUSED_THREADS)) k_icp_reverse(const __grid_constant__ RevBatch batch) {
  __shared__ RevArgs s_args;
  __shared__ TileSmem S;
  static_assert(sizeof(RevArgs) % 4 == 0 && sizeof(RevArgs) / 4 <= FUSED_THREADS, "argument block");
  if (threadIdx.x < sizeof(RevArgs) / 4) ((uint32_t*)&s_args)[threadIdx.x] = ((const uint32_t*)&batch.a[blockIdx.y])[threadIdx.x];
  __syncthreads();
  const RevArgs& a = s_args;
  if ((int)blockIdx.x >= a.grid) return;
  IcpState* __restrict__ st = a.st;
  if (st->done) return;
  __shared__ int s_q[REV_MAX_CHUNKS * FUSED_THREADS];   // the block's chosen target points (sorted positions), in order
  __shared__ int s_p[REV_MAX_CHUNKS * FUSED_THREADS];   // in: bits of the nearest chooser's d2; out: the mutual partner (sorted source position), -1 none
  __shared__ int s_wcnt[FUSED_WARPS];
  uint2* seg = reinterpret_cast<uint2*>(S.pts) + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  // ---- the block's list
  const int chunks = (a.m_valid + FUSED_THREADS - 1) / FUSED_THREADS;
  int qn = 0;   // the same in every thread
  for (int cc = 0; cc < a.per; ++cc) {
    const int c = blockIdx.x * a.per + cc;
    if (c >= chunks) break;
    const int j = c * FUSED_THREADS + threadIdx.x;
    uint32_t r = 0x7f800000u;
    if (j < a.m_valid) {
      r = a.rmin[j];
      if (r != 0x7f800000u) a.rmin[j] = 0x7f800000u;   // re-armed for the next iteration
    }
    const bool chosen = r != 0x7f800000u;
    const unsigned int bal = __ballot_sync(0xffffffffu, chosen);
    if (lane == 0) s_wcnt[warp] = __popc(bal);
    __syncthreads();
    int ofs = qn, tot = 0;
#pragma unroll
    for (int w = 0; w < FUSED_WARPS; ++w) { const int n = s_wcnt[w]; if (w < warp) ofs += n; tot += n; }
    if (chosen) { const int k = ofs + __popc(bal & ((1u << lane) - 1u)); s_q[k] = j; s_p[k] = (int)r; }
    qn += tot;
    __syncthreads();
  }

  // ---- phase A: the searches
  const float stretch = st->stretch;
  const float dev0 = st->dev;
  const float rscale = stretch * a.gs.inv_cell * 1.000001f;
  // query k as a tile query.  A chooser sits at exactly distance r: with the bound one ulp above it the chooser (and any
  // source point that ties with it) enters by the strict comparison; the lexicographic minimum over all source points is found.
  auto load = [&](int k, TileQuery& q, int stage) {
    const int j = s_q[k];
    const float4 t = __ldg(a.tgt + j);
    q.qx = t.x; q.qy = t.y; q.qz = t.z;
    q.b = NnBest{__uint_as_float((uint32_t)s_p[k] + 1u), 0x7fffffff, -1};
    const float sq = sqrtf(q.b.d2);
    q.rho = sq * 1.000001f;
    // the query in the frame the source was binned in
    const float ux = (float)(st->cinv[0] * t.x + st->cinv[1] * t.y + st->cinv[2] * t.z + st->cinv[3]);
    const float uy = (float)(st->cinv[4] * t.x + st->cinv[5] * t.y + st->cinv[6] * t.z + st->cinv[7]);
    const float uz = (float)(st->cinv[8] * t.x + st->cinv[9] * t.y + st->cinv[10] * t.z + st->cinv[11]);
    const float dev = dev0 + 1.0e-6f * fmaxf(fabsf(ux), fmaxf(fabsf(uy), fabsf(uz)));
    q.tx = grid_t(ux, a.gs.ox, a.gs.inv_cell); q.ty = grid_t(uy, a.gs.oy, a.gs.inv_cell); q.tz = grid_t(uz, a.gs.oz, a.gs.inv_cell);
    q.rc = sq * rscale + (MVR_CELL_MARGIN + 1.0e-6f * fmaxf(fabsf(q.tx), fmaxf(fabsf(q.ty), fabsf(q.tz))) + dev * stretch * a.gs.inv_cell * 1.000001f);
    q.near = q.rc <= TS_RC_NEAR;
    (void)stage;
  };
  unsigned int missed = 0;
  auto finish = [&](int k, const NnBest& b) {
    if (b.pos < 0) ++missed;
    const int j = s_q[k];
    const int mutual = (b.pos >= 0 && __ldg(a.corr_p + b.pos) == j) ? b.pos : -1;   // or the nearest source point chose another target
    s_p[k] = mutual;
    if (a.rnn) a.rnn[j] = mutual;
  };
  // which of this thread's queries the tile cannot take (bit h = query threadIdx.x + 256 h), decided before s_p is overwritten
  unsigned int far_bits = 0;
  for (int k = threadIdx.x, h = 0; k < qn; k += FUSED_THREADS, ++h) {
    TileQuery q;
    load(k, q, 0);
    if (!q.near) far_bits |= 1u << h;
  }
  const bool tiled = qn >= MVR_TS_MIN_QUERIES && tile_search(S, a.gs, a.sstart, a.cur, qn, load, [&](int k, const TileQuery& q) { if (q.skipped) far_bits |= 1u << (k / FUSED_THREADS); else finish(k, q.b); });
  if (!tiled) far_bits = 0xffffffffu;
#ifdef MVR_TS_STATS
  {
    int no = 0;
    for (int k = threadIdx.x, h = 0; k < qn; k += FUSED_THREADS, ++h) no += (far_bits >> h) & 1u;
    __shared__ int s_no;
    if (threadIdx.x == 0) s_no = 0;
    __syncthreads();
    if (no) atomicAdd(&s_no, no);
    __syncthreads();
    if (threadIdx.x == 0) { if (s_no) atomicAdd((unsigned long long*)&st->dbg[5], (unsigned long long)s_no); if (qn >= MVR_TS_MIN_QUERIES && !tiled) atomicAdd((unsigned long long*)&st->dbg[6], 1ull); }
  }
#endif
  // the queries the tile did not take walk the rows themselves (s_p still holds their chooser distance)
  bool any_open = false;
  for (int k = threadIdx.x, h = 0; k < qn; k += FUSED_THREADS, ++h) any_open |= ((far_bits >> h) & 1u) != 0;
  if (__syncthreads_or(any_open)) {   // every thread is done with the staged tile
    for (int k = threadIdx.x, h = 0; k < qn; k += FUSED_THREADS, ++h) {
      if (!((far_bits >> h) & 1u)) continue;
      const int j = s_q[k];
      const float4 t = __ldg(a.tgt + j);
      const float ux = (float)(st->cinv[0] * t.x + st->cinv[1] * t.y + st->cinv[2] * t.z + st->cinv[3]);
      const float uy = (float)(st->cinv[4] * t.x + st->cinv[5] * t.y + st->cinv[6] * t.z + st->cinv[7]);
      const float uz = (float)(st->cinv[8] * t.x + st->cinv[9] * t.y + st->cinv[10] * t.z + st->cinv[11]);
      const float dev = dev0 + 1.0e-6f * fmaxf(fabsf(ux), fmaxf(fabsf(uy), fabsf(uz)));
      NnBest b{__uint_as_float((uint32_t)s_p[k] + 1u), 0x7fffffff, -1};
      pg_search<MVR_PG_UNROLL>(a.gs, a.sstart, a.cur, a.n_valid, t.x, t.y, t.z, ux, uy, uz, dev, stretch, MVR_INF, b, seg);
      finish(k, b);
    }
  }
  if (missed) atomicAdd((unsigned long long*)&st->dbg[2], (unsigned long long)missed);   // must stay 0: a chooser was not found again
  __syncthreads();   // s_p is complete

  // ---- phase B: the sums over this thread's own mutual pairs
  const double ox = st->ox, oy = st->oy, oz = st->oz;
  constexpr int NV = EstVals<EST>::value;
  double v[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) v[k] = 0.0;
  for (int k = threadIdx.x; k < qn; k += FUSED_THREADS) {
    const int r = s_p[k];
    if (r < 0) continue;
    const float4 t = __ldg(a.tgt + s_q[k]);
    const float4 s = a.cur[r];
    acc_pair<EST>(v, s, t, a.nrm, a.nsrc + r, d2_pinned(t.x, t.y, t.z, s.x, s.y, s.z), ox, oy, oz);
  }
  reduce_and_finish<NV, EST == EST_SYM>(v, a.partials, st, a.log, a.grid);
}

