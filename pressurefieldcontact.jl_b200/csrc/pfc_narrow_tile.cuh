// pfc_narrow_tile.cuh -- the small path's narrow tile kernel (pfc_small.cu includes it twice, inside its anonymous namespace).
// PFC_TILE_KERNEL names the kernel; PFC_TILE_PARAMS (true / false) says whether each problem's contact parameters come from the
// per-environment table io.params (pfc_set_contact_params) or from the scene's InsDev.  Two kernels from one source, so that the
// evaluation without a table keeps exactly its code: a run-time select at the context phase reshuffled the register allocation of the
// whole kernel (0.9 % slower on the 4096-environment batch), and so did a shared __forceinline__ body.
template <int P, int MINB>
__global__ void __launch_bounds__(32 * P, MINB) PFC_TILE_KERNEL(SceneDev sc, EvalIO io, int cap, const unsigned* __restrict__ pairs_in, unsigned* __restrict__ ticket) {
    constexpr int kTileThreads = 32 * P;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    TileSmem<P>& sm = *reinterpret_cast<TileSmem<P>*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, wib = tid >> 5;
    const long long n_prob = io.n_env * sc.n_small;
    const long long n_tile = (n_prob + P - 1) / P;
    const int sum_q = wib;   // phase 4: warp q sums problem q
    // Tiles cost between half and twice the average (67 to 153 candidates per boxes.jl environment): after its first tile a CTA draws the
    // next one from a ticket counter instead of striding (which CTA works on a tile does not change any result).
    for (long long tile = blockIdx.x; tile < n_tile;) {
        // ---- 1. problem contexts: warp q fills problem q, one element per lane
        {
            // (lane and warp numbers made opaque per tile: this phase's index and address arithmetic is redone for each tile instead
            // of being hoisted out of the tile loop, where its results would be held -- spilled -- across the clip and the quadrature)
            int lane = tid & 31, wib = tid >> 5;
            asm volatile("" : "+r"(lane), "+r"(wib));
            const long long prob = tile * P + wib;
            const long long env = prob < n_prob ? prob / sc.n_small : 0;
            const int k = prob < n_prob ? sc.small_ins[prob - env * sc.n_small] : 0;
            if (prob < n_prob && sc.ins[k].model == PFC_MODEL_REGULARIZED) {   // (bristle instructions: pfc_exact.cu)
                const InsDev& ins = sc.ins[k];
                const long long ei = env * sc.n_ins + k;
                const InsParam* cp = PFC_TILE_PARAMS ? io.params + ei : nullptr;   // this environment's contact parameters
                const double* X = io.X + 16 * ei;
                const double* twist = io.twist + 6 * ei;
                PatchCtx<double>& cx = sm.cx[wib];
                if (lane < 8) sm.fpv[wib][lane] = cp ? cp->p[lane] : ins.p[lane];   // friction parameters: read per quadrature point, so keep them on chip
                if (lane < 9) { const int i = lane / 3, j = lane % 3; cx.x21.r[lane] = X[4 * j + i]; }
                else if (lane < 12) cx.x21.t[lane - 9] = X[12 + lane - 9];
                else if (lane < 21) { const int e = lane - 12, i = e / 3, j = e % 3; cx.x12.r[e] = X[4 * i + j]; }
                else if (lane < 24) { const int i = lane - 21; cx.x12.t[i] = -(X[4 * i] * X[12] + X[4 * i + 1] * X[13] + X[4 * i + 2] * X[14]); }
                else if (lane < 27) (&cx.w_ang.x)[lane - 24] = twist[lane - 24];
                else if (lane < 30) (&cx.w_lin.x)[lane - 27] = twist[lane - 24];
                else if (lane == 30) {
                    if (cp) { cx.chi = cp->chi; cx.Ebar1 = cp->Ebar1; cx.Ebar2 = cp->Ebar2; }
                    else { cx.chi = ins.chi; cx.Ebar1 = ins.Ebar1; cx.Ebar2 = ins.Ebar2; }
                    cx.n_quad = ins.n_quad;
                } else { sm.ei[wib] = ei; sm.fp[wib] = sm.fpv[wib]; sm.ins[wib] = k; sm.n_cand[wib] = (int)io.n_pairs[ei]; sm.pflags[wib] = 0; }
            } else if (lane == 31) { sm.ei[wib] = -1; sm.n_cand[wib] = 0; sm.ins[wib] = 0; sm.fp[wib] = nullptr; sm.pflags[wib] = 0; }
        }
        __syncthreads();
        if (tid == 0) sm.next_tile = (long long)gridDim.x + atomicAdd(ticket, 1u);   // read after the tile's last barrier
        int n_cand = 0;
#pragma unroll
        for (int q = 0; q < P; ++q) n_cand += sm.n_cand[q];
        for (int j = lane; j < P * 8; j += 32) sm.wtot[wib][j >> 3][j & 7] = 0.0;   // this warp's running sums (warp-private)
        int filled = 0;          // occupied polygon slots (block-uniform)
        int c0 = 0;              // first candidate of the next round (block-uniform)
        while (true) {
            // ---- 2a. one candidate pair per thread up to its start polygon, staged in doubles [16, 32) of slot tid: until the clip
            // an occupied slot holds its start polygon in doubles [0, 16) only, and the compaction below writes nothing else
            if (c0 < n_cand) {
                const int c = c0 + tid;
                double* zr = sm.poly + tid * kPolyStride + 16;
                int n0 = 0, q = 0;
                unsigned e = 0;
                if (c < n_cand) {
                    // first candidate of problem q: the prefix sums are taken again from shared memory (a per-thread copy held over the
                    // tile costs registers the clip needs)
                    int first = 0, end = 0;
#pragma unroll
                    for (int r = 1; r < P; ++r) { end += sm.n_cand[r - 1]; const bool ge = c >= end; q += ge; first = ge ? end : first; }
                    e = pairs_in[(size_t)cap * sm.ei[q] + (c - first)];
                    n0 = start_polygon_zeta(sc, sc.ins[sm.ins[q]], dec_a(e), dec_b(e), sm.cx[q], zr);
                }
                // ---- 2b. block scan of the survivors -> slot numbers in candidate order
                const unsigned alive = __ballot_sync(0xffffffffu, n0 > 0);
                if (lane == 0) sm.warp_tot[wib] = __popc(alive);
                __syncthreads();
                int before = 0, round_total = 0;
#pragma unroll
                for (int w = 0; w < P; ++w) { const int t = sm.warp_tot[w]; if (w < wib) before += t; round_total += t; }
                if (n0 > 0) {
                    const int slot = filled + before + __popc(alive & ((1u << lane) - 1u));
                    if (slot < kTileThreads) {
                        double* z = sm.poly + slot * kPolyStride;
#pragma unroll
                        for (int j = 0; j < 16; ++j)
                            if (j < 4 * n0) z[j] = zr[j];
                        sm.slot_pair[slot] = e; sm.slot_n[slot] = (unsigned char)n0; sm.poly_prob[slot] = (unsigned char)q;
                    } else if (slot == kTileThreads) sm.resume_c = c;   // the slots are full: the next round starts again at this candidate
                }
                __syncthreads();   // slots written, warp_tot read
                if (filled + round_total > kTileThreads) { filled = kTileThreads; c0 = sm.resume_c; }
                else { filled += round_total; c0 += kTileThreads; }
            }
            const bool last = c0 >= n_cand;
            if (filled == 0) { if (last) break; continue; }
            if (filled < kTileThreads && !last) continue;
            const int batch_n = filled;
            // ---- 2c. slot d is clipped in place by thread d, centroid -> a finished PolyRec
            int nv = 0;
            if (tid < batch_n) {
                const int q = sm.poly_prob[tid];
                const unsigned e = sm.slot_pair[tid];
                PolyRec<double>& out = *reinterpret_cast<PolyRec<double>*>(sm.poly + tid * kPolyStride);
                int flags = 0;
                const int n = clip_tet_inplace(reinterpret_cast<double*>(&out), (int)sm.slot_n[tid], flags);
                if (n >= 3) {
                    const InsDev& ins = sc.ins[sm.ins[q]];
                    finish_polygon_slot(n, sc.tets[ins.prim_base2 + dec_b(e)], pair_normal(sc, ins, dec_a(e), dec_b(e), sm.cx[q]), out);
                    nv = n;
                }
                if (flags) atomicOr(&sm.pflags[q], flags);   // rare: non-finite vertex / bad arity
            }
            // ---- 3a. block scan of the vertex counts -> dense (slot, edge) work list, ordered by (problem, pair, edge)
            int incl = nv;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
            if (lane == 31) sm.warp_tot[wib] = incl;
            __syncthreads();
            int before = 0, total = 0;
#pragma unroll
            for (int w = 0; w < P; ++w) { const int t = sm.warp_tot[w]; if (w < wib) before += t; total += t; }
            const int at = before + incl - nv;
            for (int k = 0; k < nv; ++k) sm.items[at + k] = (unsigned short)((tid << 3) | k);
            __syncthreads();
            // ---- 3b. one sub-triangle per thread; 4. sums: the items are ordered by problem, so a warp's 32 items belong to one to three
            // problems: per problem a masked xor-butterfly over the warp, lane j keeps sum j and adds it to the warp's running sum of that
            // problem (fixed item -> lane assignment, fixed tree: bitwise reproducible; no per-item results in shared memory, no barrier)
            for (int i0 = 0; i0 < total; i0 += kTileThreads) {
                const int it = i0 + tid;
                double a6[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
                int npts = 0, q = -1;
                if (it < total) {
                    const int code = sm.items[it];
                    const int slot = code >> 3, k = code & 7;
                    const PolyRec<double>& pr = *reinterpret_cast<const PolyRec<double>*>(sm.poly + slot * kPolyStride);
                    q = sm.poly_prob[slot];
                    const PatchCtx<double>& cx = sm.cx[q];
                    Accum<double, 6> tmp;
                    tmp.fp = sm.fpv[q]; tmp.w_ang = cx.w_ang; tmp.w_lin = cx.w_lin; tmp.dump = nullptr; tmp.dump_cap = 0;
                    tmp.reset(ACC_REGULARIZED);
                    const int kp = (k == 0) ? pr.n - 1 : k - 1;
                    integrate_subtri(pr.v[kp], pr.v[k], pr.cen, pr.nrm, pr.eps_r, cx, tmp);
#pragma unroll
                    for (int j = 0; j < 6; ++j) a6[j] = tmp.a[j];
                    npts = tmp.n_points;
                }
                const unsigned act = __ballot_sync(0xffffffffu, it < total);
                if (act) {   // warp-uniform
                    const int q_first = __shfl_sync(0xffffffffu, q, __ffs(act) - 1), q_last = __shfl_sync(0xffffffffu, q, 31 - __clz(act));
                    for (int qq = q_first; qq <= q_last; ++qq) {
                        const bool mine_q = q == qq;
                        double mine = (double)warp_sum_int(mine_q ? npts : 0);   // lane 6 keeps the point count
#pragma unroll
                        for (int j = 0; j < 6; ++j) { const double t = warp_sum(mine_q ? a6[j] : 0.0); mine = (lane == j) ? t : mine; }
                        if (lane < 7) sm.wtot[wib][qq][lane] += mine;
                    }
                }
            }
            __syncthreads();   // the polygon slots are reused by the next round
            filled = 0;   // (with total == 0 the two barriers of 3a already separate the clip from the next round's slot writes)
            if (last) break;
        }
        // ---- results: the warps' running sums of problem sum_q added in warp order; wrench (zero without contact), flags
        __syncthreads();   // every warp's running sums are final (a tile without candidates comes here straight from the zeroing)
        {
            const long long ei = sm.ei[sum_q];
            if (ei >= 0) {
                double t = 0.0;
                if (lane < 7) {
#pragma unroll
                    for (int w = 0; w < P; ++w) t += sm.wtot[w][sum_q][lane];
                }
                const bool contact = __shfl_sync(0xffffffffu, t, 6) > 0.0;
                if (lane < 6) io.wrench[6 * ei + lane] = contact ? t : 0.0;
                if (lane == 6) io.flags[ei] |= sm.pflags[sum_q] | (contact ? kFlagContact : 0);
            }
        }
        __syncthreads();
        tile = sm.next_tile;
    }
}
