// K6, staged variant: global similarity of all templates at the coarsest pyramid level with the linear memories staged
// through shared memory by TMA bulk copies (cp.async.bulk + mbarrier), accumulators in registers.
//
// Why: one template reads 62 byte streams of ~1,200 B from 62 of the 1,024 linear-memory rows (2 modalities x 8 labels x
// T*T rows); over 8,000 templates that is ~0.6 GB of byte traffic per frame against a 1.2 MB working set, so the bound is
// on-chip bandwidth (shared memory, 128 B/clk/SM), not HBM.  The working set does not fit one SM's shared memory, so the
// kernel walks it in PHASES (one phase = a block of the T*T rows of one (modality, label)) through a ring of buffers:
//
//   * a persistent CTA owns a batch of templates (one warp per template slot, TPW slots per warp) and keeps their
//     packed-u8 similarity accumulators in registers for the whole kernel;
//   * one elected thread per CTA streams phase q + n_buf into the buffer that was just released.  Completion is counted in
//     bytes on an mbarrier (expect_tx); a buffer is released when every consumer warp has arrived on "empty".  (A variant
//     that fetched 1/CL of a phase per CTA of a CL-CTA cluster and multicast it was measured SLOWER - 30 vs 25 us loop: the
//     L2 -> SM stream is not the limiter, the cluster-wide buffer release is - and was removed.)
//   * features were sorted by phase once per frame geometry (k_pack_staged).  A CTA copies its templates' feature words
//     and per-phase prefix counts into shared memory, so the inner loop is: one broadcast LDS for the next feature word,
//     NW + 1 LDS of linear-memory words, NW funnel shifts, NW adds;
//   * the kernel reads the 4-BIT copy of the linear memories (two cells per byte, written by the spread job beside the byte
//     version: a response is 0, 1, 2 or 4): half the shared-memory bytes per feature.  Lane g owns the NW consecutive 32-bit words
//     [g NW, (g+1) NW) of a template's similarity map, 8 cells per word (NW odd, so the 32 lanes of one LDS fall into 32 different
//     banks at any feature offset); a window that does not start on a word boundary costs NW + 1 loads, not 2 NW: the high word of
//     one funnel shift is the low word of the next;
//   * a phase's features are taken THREE at a time: their shifted words are added as packed nibbles with one three-input add (3 x 4
//     cannot carry) and the sum is split into byte accumulators (even cells / odd cells) on the spot - no nibble state is carried, no
//     counter, no data-dependent spill branch.  When whole labels fit a buffer, 2 (or 4) consecutive labels of a modality form one
//     phase: half the per-phase bookkeeping and longer runs, i.e. more triples and fewer remainders.  Measured at C2 (in-kernel
//     timeline): loop 26.0 us with one feature at a time and nibble sums spilled every third, 22.9 us with triples, 18.5 us with
//     triples and label pairs (8 phases instead of 16).
//
// Semantics are those of similarity() / addSimilarities / the scan in matchClass (reference linemod/linemod.cpp:1130-1214,
// 1322-1338, 1487-1506) including flat addressing past a row end (DESIGN.md).  Eligibility (checked on the host): every
// template has <= 63 coarsest-level features over all modalities (so one u8 lane holds the total, 63*4 = 252) and the same
// width/height for all modalities at that level (what cropTemplates :52-96 produces); otherwise the baseline kernel runs.
#include "fl_internal.cuh"
#include <stdlib.h>
#include <mutex>

#define SS_MAXF 64                      // feature words per template (<= 63 used)
#define SS_MAX_PHASES 254

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 1-D TMA: bulk copy global -> shared, completion counted in bytes on the mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
               "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ unsigned long long globaltimer() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }

// ------------------------------------------------------------------------------------------------
// per-geometry packing for the staged kernel, one thread per template:
//   gfeat[t][0..63]  coarsest-level features of all modalities sorted by phase; word = (byte offset of the 32-bit word
//                    holding the feature's first response inside the 4-bit phase buffer) << 5 | (4 x misalignment in cells)
//   gpre[t][0..P]    prefix counts: the features of phase p are gfeat[t][gpre[t][p] .. gpre[t][p+1])
//   gmeta[t]         {template_positions (linemod.cpp:1155), number of features, class index, 0}
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_pack_staged(fl_tdb db, fl_level_geom g, fl_staged_plan plan) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= db.n_templates) return;
  const int level = db.L - 1;
  const fl_template_hdr_t* hdr = db.hdr + ((size_t)t * db.L + level) * db.M;
  uint32_t* out = plan.gfeat + (size_t)t * SS_MAXF;
  uint8_t* pre = plan.gpre + (size_t)t * plan.pre_stride;
  // counting sort by phase (n <= 63): pass 1 counts, pass 2 places
  uint8_t cur[SS_MAX_PHASES + 2];
  for (int p = 0; p <= plan.n_phases; ++p) cur[p] = 0;
  int nf = 0;
  for (int m = 0; m < db.M; ++m) {
    nf += hdr[m].feature_count;
    for (int k = 0; k < hdr[m].feature_count; ++k) {
      const fl_feature_t f = db.feat[hdr[m].feature_begin + k];
      if (f.x < 0 || f.y < 0 || f.x >= g.W || f.y >= g.H) continue;                     // linemod.cpp:1179
      const int row = (f.y % g.T) * g.T + (f.x % g.T);
      const int ph = ((m * 8 + f.label) / plan.labels_per_phase) * plan.n_rowblocks + row / plan.phase_rows;
      ++cur[ph + 1];
    }
  }
  for (int p = 0; p < plan.n_phases; ++p) cur[p + 1] = (uint8_t)(cur[p + 1] + cur[p]);   // cur[p] = first slot of phase p
  for (int p = 0; p <= plan.n_phases; ++p) pre[p] = cur[p];
  const int total = cur[plan.n_phases];
  for (int m = 0; m < db.M; ++m)
    for (int k = 0; k < hdr[m].feature_count; ++k) {
      const fl_feature_t f = db.feat[hdr[m].feature_begin + k];
      if (f.x < 0 || f.y < 0 || f.x >= g.W || f.y >= g.H) continue;
      const int row = (f.y % g.T) * g.T + (f.x % g.T);
      const int rb = row / plan.phase_rows;
      const int ph = ((m * 8 + f.label) / plan.labels_per_phase) * plan.n_rowblocks + rb;
      // cell (= nibble) index inside the phase buffer; a later label of a label group starts label_stride cells further on
      const uint32_t a = (uint32_t)((f.label % plan.labels_per_phase) * g.label_stride + (row - rb * plan.phase_rows) * g.cells + (f.y / g.T) * g.Wd + f.x / g.T);
      out[cur[ph]++] = (((a >> 3) * 4u) << 5) | ((a & 7u) << 2);                        // a = cell (= nibble) index inside the phase buffer
    }
  for (int k = total; k < SS_MAXF; ++k) out[k] = 0;
  const int wf = (hdr[0].width - 1) / g.T + 1, hf = (hdr[0].height - 1) / g.T + 1;
  const int tp = min((g.Hd - hf) * g.Wd + (g.Wd - wf) + 1, g.cells);                    // template_positions :1155
  plan.gmeta[t] = make_int4(tp, nf, db.class_of[t], 0);
}

void fl_launch_pack_staged(fl_tdb db, fl_level_geom g, fl_staged_plan plan, cudaStream_t s) {
  if (db.n_templates > 0) k_pack_staged<<<(db.n_templates + 127) / 128, 128, 0, s>>>(db, g, plan);
}

// ------------------------------------------------------------------------------------------------
#define SS_NBUF_MAX 4

// One feature of one template: lane g owns the NW consecutive 32-bit words [g*NW, (g+1)*NW) of the similarity map (8 cells per
// word), so its window is the NW + 1 consecutive words starting at its base + the feature's word offset: NW + 1 loads (instead
// of two per word), one funnel shift and one add per word.  NW is odd, so the 32 lanes of one load hit 32 different banks.
// (Moving every other add to the FMA pipe as an IMAD was measured slower: IADD3 folds two adds into one issue slot.)
// NF (1..3) features of one template at once.  Per feature the lane's window is NW + 1 consecutive words (one funnel shift per
// owned word; the high word of one shift is the low word of the next).  The NF shifted words are added as packed nibbles (a response is
// <= 4, so three of them cannot carry) and the sum goes straight into the byte accumulators: lo takes the even cells of each word, hi
// the odd ones (byte totals <= 63 x 4 = 252).  Three features per spill is what keeps the kernel off the ALU pipe: per owned word
// 3 shifts + 1 three-input add + 5 spill instructions instead of 3 x (shift + add) + 5.  Words are processed in chunks of CH so that
// the loads of all NF features of a chunk are in flight together within the register budget.
template <int NW, int NF>
__device__ __forceinline__ void accumulate_features(const uint8_t* __restrict__ lane_base, const uint32_t (&fw)[3], uint32_t (&lo)[NW], uint32_t (&hi)[NW]) {
  constexpr int CH = NW <= 7 ? NW : 6;
  const uint32_t* w0 = reinterpret_cast<const uint32_t*>(lane_base + (fw[0] >> 5));
  const uint32_t* w1 = reinterpret_cast<const uint32_t*>(lane_base + (fw[NF > 1 ? 1 : 0] >> 5));
  const uint32_t* w2 = reinterpret_cast<const uint32_t*>(lane_base + (fw[NF > 2 ? 2 : 0] >> 5));
#pragma unroll
  for (int c = 0; c < NW; c += CH) {
    uint32_t v0[CH + 1], v1[CH + 1], v2[CH + 1];
#pragma unroll
    for (int i = 0; i <= CH; ++i)
      if (c + i <= NW) {
        v0[i] = w0[c + i];
        if (NF > 1) v1[i] = w1[c + i];
        if (NF > 2) v2[i] = w2[c + i];
      }
#pragma unroll
    for (int i = 0; i < CH; ++i)
      if (c + i < NW) {
        uint32_t n = __funnelshift_r(v0[i], v0[i + 1], fw[0]);            // shift = low 5 bits of the feature word
        if (NF > 1) n += __funnelshift_r(v1[i], v1[i + 1], fw[1]);
        if (NF > 2) n += __funnelshift_r(v2[i], v2[i + 1], fw[2]);
        // odd cells (hi) and the whole word (lo).  The ALU pipe (funnel shifts, IADD3, LOP3) is the busiest unit of this kernel, the
        // FMA pipe nearly idle: the shift by 4 is a multiply-high and the two accumulations are IMADs, which leaves ONE LOP3 per
        // word on the ALU pipe instead of two LOP3 and a shift.  lo collects n itself: the even cells are lo - 16 hi, exact in
        // 32-bit wrap-around arithmetic because the true packed value fits the word
        uint32_t t;
        asm("mul.hi.u32 %0, %1, 0x10000000;" : "=r"(t) : "r"(n));
        const uint32_t h = t & 0x0F0F0F0Fu;
        lo[c + i] += n;                                                    // = even cells + 16 x odd cells (mod 2^32); the caller takes 16 x hi off at the end
        hi[c + i] += h;
      }
  }
}

// per-byte maxima of packed u8 values, two 16-bit lanes at a time: the high byte of each lane of max.u16x2 is the larger of the two
// high bytes (the high byte decides a 16-bit comparison); the low bytes are garbage and ignored
__device__ __forceinline__ uint32_t vmax_u16x2(uint32_t a, uint32_t b) { uint32_t d; asm("max.u16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b)); return d; }

// Early exit (DESIGN.md 4.1): after a phase, a slot whose every position p < template_positions has partial(p) + 4 x (features
// left) <= raw_thr can produce no candidate (a response is at most 4) and is dropped.  "Any byte >= t" over the lane's accumulator
// words: the even cells are lo - 16 hi (see accumulate_features), the odd ones hi; words wholly at or past template_positions
// (nvw = the lane's words that hold a valid cell) are left out.  Per word: 1 IMAD, 2 shifts, 4 max.u16x2.
template <int NW>
__device__ __forceinline__ bool any_byte_at_least(const uint32_t (&lo)[NW], const uint32_t (&hi)[NW], int nvw, int t) {
  uint32_t mh = 0, ml = 0;                                   // maxima of bytes 1, 3 / of bytes 0, 2 (shifted up by 8), in the high bytes
#pragma unroll
  for (int i = 0; i < NW; ++i)
    if (i < nvw) {
      const uint32_t e = lo[i] - (hi[i] << 4);
      mh = vmax_u16x2(vmax_u16x2(mh, e), hi[i]);
      ml = vmax_u16x2(vmax_u16x2(ml, e << 8), hi[i] << 8);
    }
  const uint32_t m = vmax_u16x2(mh, ml);
  return (int)max((m >> 8) & 0xFFu, m >> 24) >= t;
}

// Phase order of one CTA, computed by the producer warp after griddepcontrol.wait (the response sums are written by the front end):
// s_phase[q] = the phase visited at step q.  With the early exit, a phase whose responses are low adds little to the partial sums
// and much headroom against the bound (4 per feature it retires), so the lightest phases go first: a group of labels (one phase per
// row block) weighs the sum of its labels' responses over the frame, groups are sorted by weight, ties by index so that every CTA
// agrees, and the row blocks of a group keep their order.  Without the exit (NW = 15, FL_OPT_SIM_NO_PRUNE) or with
// FL_OPT_SIM_ROTATE, CTA b starts at phase 7 b mod n_phases, so that different SMs pull different rows out of L2.  Only the load
// of the sums stands between griddepcontrol.wait and the first phase copy; the ticket that clears them is taken after the last
// copy has been issued (release_mass).
__device__ __forceinline__ void phase_order(const fl_staged_plan& plan, bool by_mass, int lane, uint8_t* s_phase) {
  const int n_phases = plan.n_phases, nrb = plan.n_rowblocks, lpp = plan.labels_per_phase;
  const int n_groups = n_phases / nrb;                        // (modality, label) groups: M x 8 / lpp <= 32
  const uint32_t mv = __ldcg(plan.mass + lane);               // the sums of all FL_MAX_MODALITIES x 8 labels, one per lane
  uint32_t w = 0;
  for (int l = 0; l < lpp; ++l) w += __shfl_sync(0xffffffffu, mv, (lane * lpp + l) & 31);
  int rank = 0;
  for (int j = 0; j < n_groups; ++j) {
    const uint32_t wj = __shfl_sync(0xffffffffu, w, j);
    rank += wj < w || (wj == w && j < lane);
  }
  if (by_mass) {
    if (lane < n_groups)
      for (int rb = 0; rb < nrb; ++rb) s_phase[rank * nrb + rb] = (uint8_t)(lane * nrb + rb);
  } else {
    const int rot = (int)((blockIdx.x * 7u) % (unsigned)n_phases);
    for (int q = lane; q < n_phases; q += 32) s_phase[q] = (uint8_t)(q + rot < n_phases ? q + rot : q + rot - n_phases);
  }
  __syncwarp();
  if (blockIdx.x == 0) {                                      // for fl_debug_get(FL_DBG_STAGED_ORDER) (stores: nothing waits for them)
    plan.mass[FL_MASS_USED + lane] = mv;
    for (int q = lane; q < n_phases; q += 32) reinterpret_cast<uint8_t*>(plan.mass + FL_MASS_ORDER)[q] = s_phase[q];
  }
}

// One thread per CTA, once the CTA's sums have been read (phase_order) and its phases issued: the last CTA to get here clears the
// sums (ticket), so that the next frame's spread jobs start from zero without a memset.  The next front end runs after this kernel.
__device__ __forceinline__ void release_mass(const fl_staged_plan& plan) {
  __threadfence();                                            // (the reads of the sums are complete: their values were used)
  if (atomicAdd(plan.mass + FL_MASS_TICKET, 1u) == gridDim.x - 1) {
    for (int i = 0; i < FL_MASS_TICKET; ++i) plan.mass[i] = 0;
    plan.mass[FL_MASS_TICKET] = 0;
  }
}

// (Refining the candidates in this kernel's own tail was measured much slower than the separate launch - stage 143 us vs 43 + 11 us:
// candidates cluster in the few CTAs that own a matching template while the other 140 CTAs idle - and was removed.)
template <int NW, int TPW>
__global__ void __launch_bounds__(1024, 1) k_similarity_staged(const __grid_constant__ fl_tdb db, fl_level_geom g, const uint8_t* __restrict__ lm4_level, float threshold,
                                                               fl_match_t* __restrict__ cand, int cap, int* __restrict__ d_count, fl_staged_plan plan) {
  extern __shared__ __align__(128) uint8_t s_dyn[];          // [n_buf x buf_bytes][tpc x int4 meta][tpc x 64 feature words + 4][tpc x pre_stride][emission staging]
  __shared__ __align__(8) uint64_t s_full[SS_NBUF_MAX], s_empty[SS_NBUF_MAX];
  __shared__ int s_emit_lock;                                 // the CTA's emission staging area is taken by one warp at a time
  __shared__ int s_live;                                      // template slots of this CTA that may still produce a candidate (early exit)
  __shared__ int s_stop;                                      // set by the producer when it issues no more phases (see the producer)
  __shared__ __align__(8) uint64_t s_aux;                     // completion of the bulk copy of this CTA's feature lists
  __shared__ uint8_t s_phase[SS_MAX_PHASES];                  // the phase visited at each step (phase_order), written before phase 0 is issued
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n_cwarps = (blockDim.x >> 5) - 1;                 // consumer warps; the last warp is the TMA producer
  // early exit (see any_byte_at_least); NW = 15 has no registers left for its test (ptxas spills), so it accumulates every template
  const bool prune = NW < 15 && plan.prune;
  const int t_begin = blockIdx.x * plan.tpc;
  const int t_end = min(t_begin + plan.tpc, db.n_templates);
  const int n_phases = plan.n_phases, n_buf = plan.n_buf;
  uint8_t* s_buf = s_dyn;
  int4* s_meta = reinterpret_cast<int4*>(s_dyn + (size_t)n_buf * plan.buf_bytes);
  uint32_t* s_feat = reinterpret_cast<uint32_t*>(s_meta + plan.tpc);
  uint8_t* s_pre = reinterpret_cast<uint8_t*>(s_feat + plan.tpc * SS_MAXF + 4);
  unsigned long long* trace = plan.trace ? plan.trace + (size_t)blockIdx.x * 8 : nullptr;
  if (trace && tid == 0) { trace[0] = globaltimer(); unsigned smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid)); trace[5] = smid; }

  if (tid == 0) {
    s_emit_lock = 0;
    s_live = max(t_end - t_begin, 0);                         // slots without positions are taken off by the consumers' prologue
    s_stop = 0;
    for (int b = 0; b < n_buf; ++b) { mbar_init(&s_full[b], 1); mbar_init(&s_empty[b], n_cwarps); }
    mbar_init(&s_aux, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (warp != n_cwarps) {
    // consumers: this CTA's per-template records, feature words and prefix counts -> shared memory while the producer
    // already streams the first phases; slots past the end / of disabled classes get no features and no positions
    for (int i = tid; i < plan.tpc; i += n_cwarps * 32) {
      const int t = t_begin + i;
      int4 m = make_int4(0, 0, 0, 0);
      if (t < t_end) {
        m = plan.gmeta[t];
        m.w = db.L == 1 ? db.tid_of[t] : t;                   // the id candidates carry (see k_similarity_global)
        const bool on = db.class_enabled[m.z];
        if (!on) m.x = 0;                                     // no positions -> no candidates
        // raw threshold int(2 nf + (threshold / 100) 2 nf + 0.5f) in fp32 (:1487); stored biased by 1, clamped to [-1, 255];
        // a disabled class gets 255, which no u8 total exceeds
        const int nf = m.y;
        const int rt = (int)__fadd_rn(__fadd_rn((float)(2 * nf), __fmul_rn(__fdiv_rn(threshold, 100.f), (float)(2 * nf))), 0.5f);
        m.y = nf | ((on ? min(max(rt, -1), 255) + 1 : 256) << 8);
      }
      s_meta[i] = m;
    }
    // (the feature words of this CTA's templates are one contiguous block of plan.gfeat: the producer thread fetches it with a
    // single bulk copy, see below; slots past the end are never read because their prefix counts are zero)
    if (tid < 4) s_feat[plan.tpc * SS_MAXF + tid] = 0u;
    {   // prefix counts, copied as 32-bit words (pre_stride is a multiple of 4): one warp per template row
      const int wpr = plan.pre_stride >> 2;
      uint32_t* s_pre32 = reinterpret_cast<uint32_t*>(s_pre);
      const uint32_t* gpre32 = reinterpret_cast<const uint32_t*>(plan.gpre);
      // (no class lookup here: a disabled class shows up as zero positions in s_meta, which the consumers test after the
      // barrier - the template -> class -> enabled chain would otherwise sit in front of these loads)
      for (int row = warp; row < plan.tpc; row += n_cwarps) {
        const int t = t_begin + row;
        for (int c = lane; c < wpr; c += 32) s_pre32[row * wpr + c] = t < t_end ? gpre32[(size_t)t * wpr + c] : 0u;
      }
    }
    asm volatile("bar.sync 1, %0;" ::"r"(n_cwarps * 32) : "memory");   // consumers only
    if (t_end > t_begin) mbar_wait(&s_aux, 0);                // feature words have landed
    fl_grid_dep_wait();                                       // before the first write to the candidate list / counter
    fl_grid_dep_launch();
  }
  if (trace && tid == 0) trace[1] = globaltimer();

  if (warp == n_cwarps) {
    // ===== producer: one elected lane streams phase q into buffer q % n_buf as soon as every consumer warp of the cluster released it =====
    if (lane == 0 && t_end > t_begin) {                       // static data: may be fetched before the previous kernel has finished
      const uint32_t fbytes = (uint32_t)(t_end - t_begin) * SS_MAXF * 4u;
      mbar_expect_tx(&s_aux, fbytes);
      bulk_g2s(s_feat, plan.gfeat + (size_t)t_begin * SS_MAXF, fbytes, &s_aux);
    }
    fl_grid_dep_wait();                                       // the linear memories and response sums are written by the previous kernel of the stream
    phase_order(plan, prune && !plan.rotate, lane, s_phase);   // (the consumers read s_phase after their wait on s_full[0])
    if (lane == 0) {
      for (int q = 0; q < n_phases; ++q) {
        const int b = q % n_buf;
        if (q >= n_buf) mbar_wait(&s_empty[b], ((q / n_buf) - 1) & 1);
        // Early exit: no live slot left -> no more phases.  The consumers wait on s_full[b] for phase q whatever happens, so the stop
        // is announced through that barrier: s_stop is written first and a plain arrive (count 1, no bytes) completes phase q of
        // s_full[b]; the arrive releases and the consumers' wait acquires, so every consumer that sees phase q complete reads
        // s_stop = 1 and leaves the loop without arriving on s_empty (a warp still behind, at an earlier phase, may see it sooner and
        // skip that phase's work: it has no live slot either).  Nothing waits on s_empty after that.  Copies still in
        // flight are those of phases q - n_buf + 1 .. q - 1 (phase q - n_buf completed before s_empty[b] could); their buffers are
        // this CTA's shared memory, so they are waited for here before the thread exits (each of those s_full barriers completes
        // once more at most: the next use of its buffer would be a phase >= q, never issued).  s_live is read without ordering:
        // a decrement seen one phase late only costs one more phase.
        if (prune && *(volatile int*)&s_live == 0) {
          *(volatile int*)&s_stop = 1;
          mbar_arrive(&s_full[b]);
          for (int r = max(q - n_buf + 1, 0); r < q; ++r) mbar_wait(&s_full[r % n_buf], (r / n_buf) & 1);
          break;
        }
        const int p = s_phase[q];
        const int grp = p / plan.n_rowblocks, rb = p - grp * plan.n_rowblocks;
        const int ml = grp * plan.labels_per_phase;             // first (modality, label) of the group; a group never straddles modalities
        const int m = ml >> 3, lab = ml & 7;
        const uint8_t* src = lm4_level + (((size_t)m * g.mod_stride + (size_t)lab * g.label_stride + (size_t)rb * plan.phase_rows * g.cells) >> 1);   // two cells per byte
        const int rows = min(plan.phase_rows, g.T * g.T - rb * plan.phase_rows);
        // (the labels of a group are contiguous in memory, pads included: one copy)
        const uint32_t bytes = (uint32_t)(((((size_t)(plan.labels_per_phase - 1) * g.label_stride + (size_t)rows * g.cells) >> 1) + plan.halo_bytes + 15) & ~(size_t)15);
        mbar_expect_tx(&s_full[b], bytes);                    // the whole phase lands here, whoever fetches it
        bulk_g2s(s_buf + (size_t)b * plan.buf_bytes, src, bytes, &s_full[b]);
      }
      release_mass(plan);
      if (trace) trace[7] = globaltimer();
    }
  } else {
    // ===== consumers =====
    bool live[TPW];                                           // false: no positions, or dropped by the early exit (pre[s] is then NULL too)
    int left[TPW];                                            // features of the slot in the phases not visited yet (early exit)
    const uint8_t* pre[TPW];
    const uint32_t* fl[TPW];
    uint32_t lo[TPW][NW], hi[TPW][NW];
#pragma unroll
    for (int s = 0; s < TPW; ++s) {
      const int slot = warp + s * n_cwarps;
      const int t = t_begin + slot;
      const bool in = slot < plan.tpc && t < t_end && s_meta[slot < plan.tpc ? slot : 0].x > 0;   // no positions (or disabled class): no work at all
      if (slot < plan.tpc && t < t_end && !in && lane == 0) atomicSub(&s_live, 1);
      live[s] = in;
      pre[s] = s_pre + (in ? slot : 0) * plan.pre_stride;
      fl[s] = s_feat + (in ? slot : 0) * SS_MAXF;
      if (!in) pre[s] = nullptr;
      left[s] = in ? pre[s][n_phases] : 0;
#pragma unroll
      for (int i = 0; i < NW; ++i) { lo[s][i] = 0; hi[s][i] = 0; }
    }
    uint32_t par = 0;
    // loop-carried shared-memory addresses, kept opaque so that the compiler carries them in registers instead of re-deriving them
    // from the kernel parameters every phase (measured: ~90 -> ~55 instructions of per-phase overhead per warp)
    uint32_t full_a = smem_u32(&s_full[0]), empty_a = smem_u32(&s_empty[0]);
    const uint32_t ring_end = full_a + 8u * (uint32_t)n_buf;
    const uint8_t* lane_base = s_buf + lane * (NW * 4);
    const uint8_t* const lane_end = lane_base + (size_t)n_buf * plan.buf_bytes;
    const int buf_bytes = plan.buf_bytes;
    asm volatile("" : "+r"(full_a), "+r"(empty_a));
    for (int q = 0; q < n_phases; ++q) {
      asm volatile(
          "{\n"
          ".reg .pred p;\n"
          "CWAIT_LOOP:\n"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
          "@p bra CWAIT_DONE;\n"
          "bra CWAIT_LOOP;\n"
          "CWAIT_DONE:\n"
          "}\n" ::"r"(full_a), "r"(par) : "memory");
      if (*(volatile int*)&s_stop) break;                     // the producer issued no phase q (early exit, see the producer)
      const int p = s_phase[q];
      if (trace && tid == 0 && q == 0) trace[2] = globaltimer();
#pragma unroll
      for (int s = 0; s < TPW; ++s) {
        if (!pre[s]) continue;
        int k = pre[s][p];
        const int k1 = pre[s][p + 1];
        if (k < k1) {                                         // warp-uniform
          const uint32_t* fp = fl[s] + k;
          int n = k1 - k;
          while (n >= 3) {                                    // the phase's features three at a time
            const uint32_t fw[3] = {fp[0], fp[1], fp[2]};
            accumulate_features<NW, 3>(lane_base, fw, lo[s], hi[s]);
            fp += 3; n -= 3;
          }
          if (n == 2) {
            const uint32_t fw[3] = {fp[0], fp[1], 0u};
            accumulate_features<NW, 2>(lane_base, fw, lo[s], hi[s]);
          } else if (n == 1) {
            const uint32_t fw[3] = {fp[0], 0u, 0u};
            accumulate_features<NW, 1>(lane_base, fw, lo[s], hi[s]);
          }
        }
      }
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(empty_a) : "memory");   // this warp is done with the buffer
      // early exit, after the release so that the producer never waits for it.  The bound only bites once raw_thr + 1 > 4 x
      // (features left); a slot without new features keeps its verdict.  A dropped slot does no more feature work and emits nothing;
      // its warp stays in step with the ring (wait on s_full, arrive on s_empty), which costs a wait and an arrive per phase.
      if (prune) {
#pragma unroll
        for (int s = 0; s < TPW; ++s) {
          if (!pre[s]) continue;
          const int k1 = pre[s][p + 1];
          if (pre[s][p] == k1) continue;                      // warp-uniform
          left[s] -= k1 - pre[s][p];
          const int rem = left[s];
          const int4 meta = s_meta[warp + s * n_cwarps];
          const int t = (meta.y >> 8) - 4 * rem;              // (meta.y >> 8) = raw_thr + 1
          if (t <= 0) continue;
          const int nvw = min(max((meta.x - lane * (NW * 8) + 7) >> 3, 0), NW);
          if (__any_sync(0xffffffffu, any_byte_at_least<NW>(lo[s], hi[s], nvw, t))) continue;
          pre[s] = nullptr; live[s] = false;
          if (lane == 0) atomicSub(&s_live, 1);
        }
      }
      full_a += 8; empty_a += 8; lane_base += buf_bytes;
      if (full_a == ring_end) { full_a -= 8u * (uint32_t)n_buf; empty_a -= 8u * (uint32_t)n_buf; lane_base -= (size_t)n_buf * buf_bytes; par ^= 1; }
    }
    (void)lane_end;
#pragma unroll
    for (int s = 0; s < TPW; ++s)
#pragma unroll
      for (int i = 0; i < NW; ++i) lo[s][i] -= hi[s][i] << 4;          // (see accumulate_features)
    if (trace && tid == 0) trace[3] = globaltimer();
    if (trace && lane == 0) plan.trace[(size_t)plan.n_cta * 8 + 8 + ((size_t)blockIdx.x * 32 + warp) * 4] = globaltimer();       // per-warp loop end

    // threshold + candidate emission (matchClass :1487-1506).  The raw threshold was computed in the prologue.
    // Every warp first asks "any byte above the threshold?" with a few SWAR operations per accumulator word.  The rare warp that
    // has candidates copies its accumulators to a staging area in shared memory (one per CTA, taken with a lock), where the byte
    // index IS the cell index, and walks it with a COMPACT loop: the first version unrolled the per-candidate code over
    // NW x 4 x TPW register positions, ~100 KB of cold instructions whose instruction-cache misses cost a candidate-bearing
    // warp 5-10 us (measured) - and the whole kernel waits for its slowest warp.  Slots are reserved with ONE returning atomic
    // per template; the records are written ballot-compacted by all lanes in parallel.
    const int off = g.T / 2 + (g.T % 2 - 1);
    uint32_t* s_stage = reinterpret_cast<uint32_t*>(s_dyn + plan.stage_off);
#pragma unroll
    for (int s = 0; s < TPW; ++s) {
      if (!live[s]) continue;                                 // warp-uniform
      const int4 meta = s_meta[warp + s * n_cwarps];
      const int tp = meta.x, nf = meta.y & 0xFF, raw_thr = (meta.y >> 8) - 1;
      if (tp <= 0 || raw_thr >= 255) continue;                // disabled class / a u8 total cannot exceed the threshold
      // bytes >= raw_thr + 1, two 16-bit lanes at a time: e + (256 - t) carries into bit 8 exactly when e >= t
      uint32_t anyw = raw_thr < 0 ? 1u : 0u;
      if (raw_thr >= 0) {
        const uint32_t k = (uint32_t)(255 - raw_thr) * 0x00010001u;
#pragma unroll
        for (int i = 0; i < NW; ++i) {
          const uint32_t v = lo[s][i], u = hi[s][i];
          anyw |= (((v & 0x00FF00FFu) + k) | (((v >> 8) & 0x00FF00FFu) + k) | ((u & 0x00FF00FFu) + k) | (((u >> 8) & 0x00FF00FFu) + k)) & 0x01000100u;
        }
      }
      if (!__any_sync(0xffffffffu, anyw != 0)) continue;      // (cells past template_positions are filtered below)
      if (lane == 0) { while (atomicCAS(&s_emit_lock, 0, 1) != 0) __nanosleep(100); }
      __syncwarp();
#pragma unroll
      for (int i = 0; i < NW; ++i) {                          // back to one byte per cell in cell order: even cells come from lo, odd ones from hi
        s_stage[(lane * NW + i) * 2] = __byte_perm(lo[s][i], hi[s][i], 0x5140);
        s_stage[(lane * NW + i) * 2 + 1] = __byte_perm(lo[s][i], hi[s][i], 0x7362);
      }
      __syncwarp();
      // pass 1 (cheap, ~20 instructions per 128 cells): compact the (cell, raw) pairs above the threshold into a list.  A lone
      // warp runs dependent code at ~5 cycles per instruction, so the expensive per-candidate work (division, IEEE divide,
      // record stores) is done ONCE for up to 32 candidates in pass 2 instead of once per group of 32 cells.
      uint32_t* s_hits = s_stage + 2 * NW * 32;
      const int n_words_tp = (tp + 3) >> 2;
      int total = 0;
      for (int w0 = 0; w0 < n_words_tp; w0 += 32) {
        const int w = w0 + lane;
        const uint32_t v = w < n_words_tp ? s_stage[w] : 0u;
        {   // most groups of 128 cells hold no candidate: one SWAR test + one ballot rejects them
          const uint32_t k = (uint32_t)(255 - max(raw_thr, 0)) * 0x00010001u;
          const uint32_t any = raw_thr < 0 ? 1u : ((((v & 0x00FF00FFu) + k) | (((v >> 8) & 0x00FF00FFu) + k)) & 0x01000100u);
          if (!__any_sync(0xffffffffu, w < n_words_tp && any != 0)) continue;
        }
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const int raw = (int)((v >> (8 * b)) & 0xFFu), j = 4 * w + b;
          const bool hit = w < n_words_tp && j < tp && raw > raw_thr;
          const uint32_t bal = __ballot_sync(0xffffffffu, hit);
          if (hit) s_hits[total + __popc(bal & ((1u << lane) - 1))] = (uint32_t)j | ((uint32_t)raw << 16);
          total += __popc(bal);
        }
      }
      __syncwarp();
      if (total > 0) {
        // this template has candidates: pull its refinement records (and its id) towards L2 now, so that the refinement
        // kernel finds them there instead of paying two DRAM round trips per candidate
        if (db.rrec && db.L > 1) {
          const uint8_t* rec = db.rrec + (size_t)meta.w * (db.L - 1) * db.rrec_bytes;
          for (int o = lane * 128; o < (db.L - 1) * db.rrec_bytes; o += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(rec + o));
          if (lane == 31) asm volatile("prefetch.global.L2 [%0];" ::"l"(db.tid_of + meta.w));
        }
        if (trace && lane == 0) plan.trace[(size_t)plan.n_cta * 8 + 8 + ((size_t)blockIdx.x * 32 + warp) * 4 + 2] = globaltimer();   // before the atomic
        int base = 0;
        if (lane == 0) base = atomicAdd(d_count, total);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (trace && lane == 0) plan.trace[(size_t)plan.n_cta * 8 + 8 + ((size_t)blockIdx.x * 32 + warp) * 4 + 3] = globaltimer();   // after the atomic
        const int lim = cap;
        // pass 2: one lane per candidate
        for (int k = lane; k < total; k += 32) {
          const int slot = base + k;
          if (slot >= lim) break;
          const uint32_t hv = s_hits[k];
          const int j = (int)(hv & 0xFFFFu), raw = (int)(hv >> 16);
          const int r = j / g.Wd, c = j - r * g.Wd;
          const int mx = c * g.T + off, my = r * g.T + off;
          const float msim = __fadd_rn(__fdiv_rn(__fmul_rn((float)raw, 100.f), (float)(4 * nf)), 0.5f);
          fl_match_t mt;
          mt.x = mx; mt.y = my; mt.similarity = msim; mt.class_idx = meta.z; mt.template_id = meta.w;
          cand[slot] = mt;
        }
      }
      __syncwarp();
      if (lane == 0) { __threadfence_block(); atomicExch(&s_emit_lock, 0); }
    }
    // Below a zero raw threshold (only a threshold under -100 gives one) every cell of the map is a candidate (:1497-1504), also
    // the cells at and past template_positions - where the reference's map holds 0 - and every cell of a template without
    // positions.  The accumulators cover template_positions only, so these candidates are written here with a raw score of 0.
#pragma unroll
    for (int s = 0; s < TPW; ++s) {
      const int slot = warp + s * n_cwarps;
      if (slot >= plan.tpc || t_begin + slot >= t_end) continue;      // warp-uniform
      const int4 meta = s_meta[slot];
      const int nf = meta.y & 0xFF, raw_thr = (meta.y >> 8) - 1;
      const int j0 = max(meta.x, 0), n = g.cells - j0;
      if (raw_thr >= 0 || n <= 0) continue;
      int base = 0;
      if (lane == 0) base = atomicAdd(d_count, n);
      base = __shfl_sync(0xffffffffu, base, 0);
      const float msim = __fadd_rn(__fdiv_rn(__fmul_rn(0.f, 100.f), (float)(4 * nf)), 0.5f);
      for (int k = lane; k < n && base + k < cap; k += 32) {
        const int j = j0 + k, r = j / g.Wd, c = j - r * g.Wd;
        fl_match_t mt;
        mt.x = c * g.T + off; mt.y = r * g.T + off; mt.similarity = msim; mt.class_idx = meta.z; mt.template_id = meta.w;
        cand[base + k] = mt;
      }
    }
    if (trace && lane == 0) { atomicMax(&trace[6], globaltimer()); plan.trace[(size_t)plan.n_cta * 8 + 8 + ((size_t)blockIdx.x * 32 + warp) * 4 + 1] = globaltimer(); }
  }
  if (trace && tid == 0) trace[4] = globaltimer();
}

__global__ void k_stamp(unsigned long long* p) { *p = globaltimer(); }

template <int NW, int TPW>
static int launch_staged(fl_tdb db, fl_level_geom g, const uint8_t* lm4_level, float threshold, fl_match_t* cand, int cap, int* d_count,
                         fl_staged_plan plan, cudaStream_t s) {
  auto kern = k_similarity_staged<NW, TPW>;
  {   // the opt-in belongs to the (device, function) pair; per-device table, locked (handles on several devices / host threads)
    static std::mutex mu;
    static size_t configured[FL_MAX_DEVICES];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= FL_MAX_DEVICES) return -1;
    std::lock_guard<std::mutex> lk(mu);
    if ((size_t)plan.smem_bytes > configured[dev]) {
      if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, plan.smem_bytes) != cudaSuccess) return -1;
      configured[dev] = plan.smem_bytes;
    }
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.gridDim = dim3(plan.n_cta); cfg.blockDim = dim3(plan.block_threads); cfg.dynamicSmemBytes = plan.smem_bytes; cfg.stream = s;
  // Programmatic dependent launch: the CTAs become resident and run their prologue (barrier init, bulk copy of the feature lists,
  // per-template thresholds) while the front-end launch drains; they touch the linear memories and the candidate list only after
  // griddepcontrol.wait.  Measured: 79.9 -> 77.3 us per frame.  Off while the developer timeline is recorded.
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = plan.trace ? 0 : 1;
  if (plan.trace) k_stamp<<<1, 1, 0, s>>>(plan.trace + (size_t)plan.n_cta * 8);
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, db, g, lm4_level, threshold, cand, cap, d_count, plan);
  if (plan.trace) k_stamp<<<1, 1, 0, s>>>(plan.trace + (size_t)plan.n_cta * 8 + 1);
  return e == cudaSuccess ? 0 : -1;
}

// host planning: returns false if the geometry is not supported by the staged kernel.  max_positions = the largest
// template_positions (linemod.cpp:1155) over the uploaded templates: only that many cells of a similarity map are ever
// looked at, so the per-lane accumulator count NW is sized for it rather than for the whole grid.
bool fl_plan_staged(const fl_level_geom& g, int M, int n_templates, int max_positions, int n_sm, fl_staged_plan* plan) {
  // NW <= 15 covers 32 x 15 x 8 = 3,840 positions.  A larger NW would need a halo of 32 NW 4 + 16 bytes past the last row,
  // more than the FL_LM_PAD / 2 bytes of zero pad behind a label's 4-bit linear memory: larger grids use the baseline kernel.
  static const int kNW[] = {3, 5, 7, 9, 11, 13, 15};
  fl_staged_plan p;
  memset(&p, 0, sizeof p);
  const int T2 = g.T * g.T;
  if (max_positions < 1 || n_templates < 1) return false;
  if (g.Wd & 1) return false;                                  // the 4-bit linear memories exist for grids of even width only (two cells per byte)
  if (max_positions > g.cells) max_positions = g.cells;
  p.n_words = (max_positions + 7) / 8;                         // 8 cells per 32-bit word
  const int nw_min = (p.n_words + 31) / 32;
  p.nw_template = 0;
  for (int nw : kNW) if (nw >= nw_min) { p.nw_template = nw; break; }
  if (!p.nw_template) return false;                            // more than 3,840 positions (see kNW)
  p.tpw = p.nw_template > 5 ? 1 : 2;                           // register budget: 64 per thread at 1,024 threads, 3 NW accumulator words per slot
  // bytes staged past the last row of a phase: a window starts at most at the last cell of the last row and the loads run
  // unconditionally over 32 * NW + 1 words
  p.halo_bytes = 32 * p.nw_template * 4 + 16;
  if (p.halo_bytes + 16 > FL_LM_PAD / 2) return false;
  // CTAs: whole waves of the SM count, up to 31 consumer warps x TPW templates each (+ 1 producer warp)
  const int per_cta_max = 31 * p.tpw;
  int n_cta = (n_templates + per_cta_max - 1) / per_cta_max;
  n_cta = ((n_cta + n_sm - 1) / n_sm) * n_sm;
  p.tpc = (n_templates + n_cta - 1) / n_cta;
  p.n_cta = (n_templates + p.tpc - 1) / p.tpc;
  const int warps = (p.tpc + p.tpw - 1) / p.tpw;
  p.block_threads = 32 * ((warps < 1 ? 1 : warps) + 1);
  // rows per phase: the ring's buffers share the CTA's shared memory with the feature lists; a phase is the largest block of rows
  // of one (modality, label) that fits a buffer of a 2-buffer ring (fewer, larger phases beat more, smaller ones: every phase
  // boundary is a CTA-wide hand-over); a row block must start 16-byte aligned in global memory, i.e. at a multiple of 32 cells.
  // If whole labels fit with room to spare the ring gets up to 4 buffers (deeper prefetch).
  const size_t stage_bytes = (size_t)p.nw_template * (256 + 1024);   // emission staging: the map as bytes (2 NW x 32 words) + one list word per cell
  const size_t lists = (size_t)p.tpc * 16 + ((size_t)p.tpc * SS_MAXF + 4) * 4 + (size_t)p.tpc * (SS_MAX_PHASES + 2) + 32 + stage_bytes;   // upper bound (n_phases <= SS_MAX_PHASES)
  const size_t avail = 227 * 1024 - 1024;
  if (lists + 4096 > avail) return false;
  const size_t budget = ((avail - lists) / 2) & ~(size_t)127;
  int pr = 0;
  for (int cand_pr = T2; cand_pr >= 1; --cand_pr) {
    if (((size_t)cand_pr * g.cells >> 1) + p.halo_bytes + 128 > budget) continue;
    if (cand_pr != T2 && ((size_t)cand_pr * g.cells) % 32 != 0) continue;
    pr = cand_pr;
    break;
  }
  if (!pr) return false;
  p.phase_rows = pr;
  p.n_rowblocks = (T2 + pr - 1) / pr;
  // whole labels fit a buffer: put 2 or 4 consecutive labels of a modality into one phase if a 2-buffer ring still fits - every
  // phase costs each warp ~45 instructions of bookkeeping whatever it holds, and longer runs of features split into more triples
  p.labels_per_phase = 1;
  if (p.n_rowblocks == 1)
    for (int G = 4; G >= 2; G >>= 1)
      if ((((size_t)(G - 1) * g.label_stride + (size_t)T2 * g.cells) >> 1) + p.halo_bytes + 128 <= budget) { p.labels_per_phase = G; break; }
  p.n_phases = M * (8 / p.labels_per_phase) * p.n_rowblocks;
  if (p.n_phases > SS_MAX_PHASES) return false;
  const size_t phase_bytes = (((size_t)(p.labels_per_phase - 1) * g.label_stride + (size_t)pr * g.cells) >> 1) + p.halo_bytes;
  if (phase_bytes >= (1u << 24)) return false;
  p.buf_bytes = (int)((((phase_bytes + 15) & ~(size_t)15) + 127) & ~(size_t)127);
  p.pre_stride = (p.n_phases + 1 + 3) & ~3;
  const int fixed = p.tpc * 16 + (p.tpc * SS_MAXF + 4) * 4 + p.tpc * p.pre_stride + 16 + (int)stage_bytes;
  int nbuf = 2;
  while (nbuf < SS_NBUF_MAX && (size_t)(nbuf + 1) * p.buf_bytes + fixed <= 227 * 1024 - 512) ++nbuf;
  p.n_buf = p.n_phases < nbuf ? p.n_phases : nbuf;
  p.smem_bytes = p.n_buf * p.buf_bytes + p.tpc * 16 + (p.tpc * SS_MAXF + 4) * 4 + p.tpc * p.pre_stride;
  p.stage_off = (p.smem_bytes + 15) & ~15;
  p.smem_bytes = p.stage_off + (int)stage_bytes;
  if (p.smem_bytes > 227 * 1024 - 512) return false;
  p.prune = 1;
  *plan = p;
  return true;
}

int fl_launch_similarity_staged(fl_tdb db, fl_level_geom g, const uint8_t* lm4_level, float threshold, fl_match_t* cand, int cap,
                                int* d_count, fl_staged_plan plan, cudaStream_t s) {
  switch (plan.nw_template) {
    case 3: return launch_staged<3, 2>(db, g, lm4_level, threshold, cand, cap, d_count, plan, s);
    case 5: return launch_staged<5, 2>(db, g, lm4_level, threshold, cand, cap, d_count, plan, s);
    case 7: return launch_staged<7, 1>(db, g, lm4_level, threshold, cand, cap, d_count, plan, s);
    case 9: return launch_staged<9, 1>(db, g, lm4_level, threshold, cand, cap, d_count, plan, s);
    case 11: return launch_staged<11, 1>(db, g, lm4_level, threshold, cand, cap, d_count, plan, s);
    case 13: return launch_staged<13, 1>(db, g, lm4_level, threshold, cand, cap, d_count, plan, s);
    case 15: return launch_staged<15, 1>(db, g, lm4_level, threshold, cand, cap, d_count, plan, s);
  }
  return -1;
}
