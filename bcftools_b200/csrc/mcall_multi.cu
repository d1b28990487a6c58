/*  mcall_multi.cu -- site kernel of the 3-, 4- and 5-allele classes (int32 PLs, one sample group, every sample diploid,
 *  GT + GQ + trimmed PL all requested, an even sample count that fits the shared-memory copy).
 *
 *  Same algorithm and reference line map as mcall_kernels.cu (set_pdg mcall.c:451-544, mcall_find_best_alleles 591-710,
 *  group combine + QUAL 1546-1567 / 1631-1645, trimming maps 547-570, mcall_call_genotypes 745-886,
 *  mcall_set_ref_genotypes 713-743, mcall_trim_and_update_PLs 1158-1194); what differs is how a site is held and walked:
 *
 *    - ONE small CTA (2-8 warps) owns one site and many CTAs share an SM, so that the serial part of a site (warp 0
 *      comparing the allele sets) overlaps the sample loops of the other CTAs.  HBM sees every PL byte once: phase 1
 *      leaves a byte-packed copy of the site (6 / 10 / 16 bytes per sample for 6 / 10 / 15 genotypes) in shared memory
 *      and the sample's normaliser `sum` (8 bytes) in a per-CTA scratch row that never leaves L2, and phase 2 works
 *      from those -- it neither re-fetches the int32 block nor repeats the G table look-ups per sample.
 *    - every WARP streams its own 64-sample tiles of the int32 block through a private ring of bulk copies
 *      (cp.async.bulk + mbarrier, SASS UBLKCP / SYNCS): no block barrier inside a phase; the first tiles of the CTA's
 *      NEXT site are issued when phase 2 starts, so they land while phase 2 computes.
 *    - each lane takes TWO ADJACENT samples per iteration (coefficient loads are shared, two dependency chains
 *      interleave, the pair's outputs leave in 64/128-bit stores).
 *    - phase 1 keeps ONE plain double product per allele set and thread -- 1 DMUL per set and sample instead of the
 *      exponent-tracked multiply (every factor is >= 1e-27 for PL <= 255, so ten samples cannot underflow); exponents
 *      are split off every fifth iteration and in the warp reduction, which goes through a shared-memory transpose (one
 *      lane per allele set multiplies the 32 partial products).  Samples without data (PL = 0,..,0) are multiplied in
 *      like any other and divided out per site (their factor is a per-site constant).
 *    - a sample with a missing / vector_end value or a PL >= 256 enters the main loop as a no-data sample and its int32
 *      row goes on a per-site list; warp 0 evaluates the list with the general per-sample code (sum of logs) before
 *      the allele sets are compared, and stores the FILLED bytes (mcall.c:495-527) so that phase 2 sees an ordinary sample.
 *    - phase 2 is straight-line code per site type: REF only / a pair {REF,b} / a triple {REF,b,c}, each keeping exactly
 *      the selected alleles.  Everything else (selected set without REF, unseen allele selected, PL >= 256 after the
 *      fill, list overflow) is appended to a fallback list that the general tiled kernel (mcall_kernels.cu) processes.
 *
 *  Numerics: phase 2 is the literal arithmetic of mcall_kernels.cu (bit-exact GT / GQ / PL / AC / AN); phase 1 totals
 *  agree with the reference's sequential sum of logs to ~1e-11 (QUAL within 1e-6 relative, near-ties flagged).
 */

#include "mcall_multi.cuh"

namespace mcb {

#define MM_MAX_NST   4              /* ring stages per warp */
/*  resident threads per SM each instance is compiled for (the register cap is 65536 / threads)  */
#ifndef MM_THREADS3
#define MM_THREADS3 512
#endif
#ifndef MM_THREADS4
#define MM_THREADS4 512
#endif
#ifndef MM_THREADS5
#define MM_THREADS5 256
#endif
template<int NALS> constexpr int mm_threads = NALS==3 ? MM_THREADS3 : (NALS==4 ? MM_THREADS4 : MM_THREADS5);

/*  per-warp shared-memory region: the bulk-copy ring, reused for the warp reduction while no copy is in flight  */
__host__ __device__ constexpr int mm_warp_region(int tile_bytes, int red_bytes, int nst)
{
    return ((nst*tile_bytes > red_bytes ? nst*tile_bytes : red_bytes) + 127) & ~127;
}

template<int NALS, int BLOCK> struct MMShared
{
    using S = Shape<NALS>;
    static constexpr int NW = BLOCK/32, NSET = MMGeom<NALS>::NSET, NACC = NSET + 1;
    double   pl2p[256];
    double   gq_thr[130];
    ScreenTabs scr;                     /* float32 screen of phase 2 (mcall_device.cuh) */
    float    scr_w[8];                  /* its weights of the slots 0..5; [6] != 0: this site stays on the literal path */
    uint64_t bars[NW][MM_MAX_NST];
    MMSetup<NALS> setup[2];
    /* phase-1 partials of every warp: products (mantissa, exponent), integer sums, counts */
    double   red_M[NW][NACC];
    int      red_E[NW][NACC];
    int      red_pls[NW][NALS];
    int      red_cnt[NW];               /* samples without data that went through the main loop (PL = 0,..,0 and the listed ones) */
    /* samples that take the general path: index and int32 row */
    int      nesc;
    unsigned short esc[MM_ESC_CAP];
    int      esc_pl[MM_ESC_CAP][S::G];
    /* site decision record (written by warp 0, read by everybody in phase 2 and by thread 0 at the next site's start) */
    double   max_qual, lk_sum, ref_lk, gap, lse;     /* lse = logsumexp2(lk_sum, ref_lk) */
    double   q[3];
    uint32_t als_new, flags;
    int      path;                      /* 0 nothing to do, 1 REF only, 2 pair {REF,b}, 3 triple {REF,b,c} */
    int      nals_new, ref_gt, site;
    long long out_off;
    int      als_map[NALS];
    int      jgt[6];                    /* byte offset of slot k's genotype in a packed row */
    int      ac[8];
    int4     slot_out[8];               /* triple sites: {gt0, gt1, AC increment lo, hi} of slot k */
};

__device__ __forceinline__ void mm_lds_f64x2(uint32_t a, double &x, double &y)
{
    asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(x), "=d"(y) : "r"(a));
}
__device__ __forceinline__ uint64_t mm_policy_evict_first() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p)); return p; }
__device__ __forceinline__ void mm_ldg_f64x2(const double *p, double &x, double &y, uint64_t pol)
{
    asm volatile("ld.global.cg.L2::cache_hint.v2.f64 {%0,%1}, [%2], %3;" : "=d"(x), "=d"(y) : "l"(p), "l"(pol) : "memory");
}
__device__ __forceinline__ void mm_stg_f64x2(double *p, double x, double y, uint64_t pol)
{
    asm volatile("st.global.cg.L2::cache_hint.v2.f64 [%0], {%1,%2}, %3;" :: "l"(p), "d"(x), "d"(y), "l"(pol) : "memory");
}
__device__ __forceinline__ void mm_bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar, uint64_t pol)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(pol) : "memory");
}
__device__ __forceinline__ int2 mm_lds64i(uint32_t a)
{
    int2 v; asm volatile("ld.shared.v2.s32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a)); return v;
}
__device__ __forceinline__ void mm_sts64(uint32_t a, uint32_t x, uint32_t y) { asm volatile("st.shared.v2.b32 [%0], {%1,%2};" :: "r"(a), "r"(x), "r"(y) : "memory"); }
__device__ __forceinline__ void mm_sts128(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w)
{
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" :: "r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void mm_sts_f64x2(uint32_t a, double x, double y) { asm volatile("st.shared.v2.f64 [%0], {%1,%2};" :: "r"(a), "d"(x), "d"(y) : "memory"); }
__device__ __forceinline__ void mm_sts_f64(uint32_t a, double x) { asm volatile("st.shared.f64 [%0], %1;" :: "r"(a), "d"(x) : "memory"); }


/*  Warp 0 between the phases: the totals of the CTA's warps, then the general-path samples and the decision (mm_decide).  */
template<int NALS, int BLOCK>
static __device__ __noinline__ void mm_epilogue(MMShared<NALS,BLOCK> *shp, const MMSetup<NALS> *su, const KArgs &a, int lane,
                                                uint32_t pl2p_s, uint32_t pack_s, double *sums_g)
{
    constexpr int NSUB = Shape<NALS>::NSUB, NSET = MMGeom<NALS>::NSET, NW = BLOCK/32;
    constexpr double LN2 = 0.693147180559945309417232121458;
    MMShared<NALS,BLOCK> &sh = *shp;
    int n0 = 0;
    #pragma unroll
    for (int w=0; w<NW; w++) n0 += sh.red_cnt[w];
    /* log of the product over all fast-path samples: lane 31 the normalisers, lanes NALS.. the live allele sets */
    double tl = 0;
    if ( lane==31 || (lane>=NALS && lane<NSUB && ((su->live >> (lane-NALS)) & 1u)) )
    {
        const int k = lane==31 ? NSET : lane - NALS;
        double M = 1.0; int E = 0;
        #pragma unroll
        for (int w=0; w<NW; w++) { M = __dmul_rn(M, sh.red_M[w][k]); E += sh.red_E[w][k]; }
        tl = mm_log(M) + (double)E*LN2;
    }
    long long ps = 0;
    if ( lane < NALS )
    {
        #pragma unroll
        for (int w=0; w<NW; w++) ps += sh.red_pls[w][lane];
    }
    const int nesc_raw = sh.nesc;
    const int s = lane < min(nesc_raw, MM_ESC_CAP) ? sh.esc[lane] : 0;
    mm_decide<NALS,12>(&sh, su, a, lane, pl2p_s, pack_s + (uint32_t)(s*MMGeom<NALS>::RS), nesc_raw, sh.esc_pl[lane], sums_g + s, tl, n0, ps);
    if ( lane==0 ) sh.nesc = 0;
}


template<int NALS, int BLOCK>
__global__ void __launch_bounds__(BLOCK, (mm_threads<NALS>/BLOCK > 0 ? mm_threads<NALS>/BLOCK : 1)) mcall_multi_kernel(const KArgs a)
{
    using S = Shape<NALS>;
    using GE = MMGeom<NALS>;
    using SH = MMShared<NALS,BLOCK>;
    constexpr int G = S::G, NPAIR = S::NPAIR, NTRI = S::NTRI, NSET = GE::NSET, NACC = GE::NACC, NW = BLOCK/32, RS = GE::RS;
    constexpr int TILE_BYTES = GE::TILE_BYTES;
    static_assert(offsetof(SH, scr_w) % 16 == 0, "scr_w is read with 128-bit loads");
    static_assert(NACC <= 31 && NW >= 2, "one lane per product in the warp reduction; warp 1 prepares the next site");
    constexpr bool CF_REG = NALS<=3;            /* coefficients of the small shape live in registers */

    SH &sh = *reinterpret_cast<SH*>(mcb_smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nsmpl = a.nsmpl, ntiles = (nsmpl + 63) >> 6, spad = ntiles*64, nst = a.nstage;
    const int ntw = warp < ntiles ? (ntiles - warp + NW - 1)/NW : 0;       /* tiles of this warp: warp, warp+NW, ... */
    const uint32_t sbase = smem_base();
    const uint32_t dyn_s = sbase + (uint32_t)align128(sizeof(SH));
    const int wreg = mm_warp_region(TILE_BYTES, GE::RED_BYTES, nst);       /* per-warp region: bulk-copy ring / warp-reduction scratch */
    const uint32_t ring_s = dyn_s + (uint32_t)(warp*wreg);
    const uint32_t pack_s = dyn_s + (uint32_t)(NW*wreg);
    double *sums_g = a.mm_sums + (size_t)blockIdx.x*spad;                    /* per-CTA row of normalisers: rewritten every site, lives in L2 */
    const uint32_t bars_s = sbase + (uint32_t)offsetof(SH, bars) + (uint32_t)(warp*MM_MAX_NST*8);
    const uint32_t pl2p_s = sbase + (uint32_t)offsetof(SH, pl2p), thr_s = sbase + (uint32_t)offsetof(SH, gq_thr);
    const uint32_t slot_s = sbase + (uint32_t)offsetof(SH, slot_out);
    const int nsites = *a.site_count;

    for (int i=tid; i<256; i+=BLOCK) sh.pl2p[i] = a.tab->pl2p[i];
    for (int i=tid; i<130; i+=BLOCK) sh.gq_thr[i] = i<128 ? a.tab->gq_thr[i] : -1.0;
    screen_tabs_fill(&sh.scr, a.tab, tid, BLOCK);
    const uint32_t plf_s = sbase + (uint32_t)offsetof(SH, scr) + (uint32_t)offsetof(ScreenTabs, plf);
    const uint32_t gqw_s = sbase + (uint32_t)offsetof(SH, scr) + (uint32_t)offsetof(ScreenTabs, gqw);
    const uint32_t q_s = sbase + (uint32_t)offsetof(SH, q), jgt_s = sbase + (uint32_t)offsetof(SH, jgt), scrw_s = sbase + (uint32_t)offsetof(SH, scr_w);
    if ( lane==0 )
    {
        for (int i=0; i<MM_MAX_NST; i++) mbar_init(bars_s + 8*i, 1);
        fence_mbar_init();
    }
    if ( tid==0 )
    {
        sh.setup[0].isite = atomicAdd(a.work_counter, 1);
        sh.nesc = 0;
        for (int j=0; j<8; j++) sh.ac[j] = 0;
        sh.path = 0;
    }
    __syncthreads();
    if ( warp==1 ) mm_setup<NALS>(&sh.setup[0], a, lane, nsites);

    const uint32_t lane_row_s = ring_s + (uint32_t)(lane*2*G*4);
    const uint64_t pol_last = mm_policy_evict_last(), pol_first = mm_policy_evict_first();
    int par = 0;
    /* the ring position of the next tile this warp consumes: the c-th tile a warp pushes through its ring uses stage
       c % nst and completes phase (c / nst) & 1 of that stage's barrier; kept incrementally, across sites */
    uint32_t stage = 0, parity = 0;
    bool prefetched = false;

    /* every tile is 64 samples except the site's last one, which belongs to warp (ntiles-1) % NW as its tile number ntw-1 */
    const uint32_t last_bytes = ((uint32_t)((nsmpl - (ntiles-1)*64)*G*4) + 15u) & ~15u;
    const int j_short = ((ntiles-1) % NW)==warp ? ntw-1 : -1;
    auto issue = [&](const int32_t *site_pl, int j, uint32_t stg)      /* lane 0: tile j of this warp into ring stage stg */
    {
        const uint32_t bytes = j==j_short ? last_bytes : (uint32_t)TILE_BYTES;
        mbar_expect_tx(bars_s + 8*stg, bytes);
        mm_bulk_g2s(ring_s + stg*TILE_BYTES, site_pl + (size_t)(warp + j*NW)*(64*G), bytes, bars_s + 8*stg, pol_first);     /* PL blocks are read once */
    };
    auto issue_first = [&](const int32_t *site_pl)                      /* lane 0: the first tiles of a site, from the current ring position */
    {
        uint32_t stg = stage;
        fence_proxy_async();                    /* the region was written through the generic proxy by the warp reduction */
        for (int j=0; j<nst && j<ntw; j++) { issue(site_pl, j, stg); if ( ++stg==(uint32_t)nst ) stg = 0; }
    };

    for (;;)
    {
        __syncthreads();            /* [A] phase 2 of the previous site is complete, the next set-up is visible */
        if ( tid==0 && sh.path>0 ) { mm_finalize<NALS>(&sh, a); sh.path = 0; }
        const MMSetup<NALS> &su = sh.setup[par];
        if ( su.isite >= nsites ) break;
        const int32_t *site_pl = reinterpret_cast<const int32_t*>(a.pl) + su.pl_off;
        const uint32_t live = su.live;
        const uint32_t su_s = sbase + (uint32_t)offsetof(SH, setup) + (uint32_t)(par*sizeof(MMSetup<NALS>));
        const uint32_t cfp_s = su_s + (uint32_t)offsetof(MMSetup<NALS>, cfp), cft_s = su_s + (uint32_t)offsetof(MMSetup<NALS>, cft);

        if ( !prefetched && lane==0 ) issue_first(site_pl);

        /* =========================== phase 1: site reduction ==================================== */
        double accM[NACC]; int accE[NACC];
        int plsum[NALS];
        int n0 = 0, since = 0;
        #pragma unroll
        for (int k=0; k<NACC; k++) { accM[k] = 1.0; accE[k] = 0; }
        #pragma unroll
        for (int k=0; k<NALS; k++) plsum[k] = 0;
        double cfr[CF_REG ? NPAIR*3 + NTRI*6 : 1];
        if ( CF_REG )
        {
            #pragma unroll
            for (int k=0; k<NPAIR; k++)
                #pragma unroll
                for (int c=0; c<3; c++) cfr[CF_REG ? k*3+c : 0] = lds64(cfp_s + 8u*(uint32_t)(k*4+c));
            #pragma unroll
            for (int k=0; k<NTRI; k++)
                #pragma unroll
                for (int c=0; c<6; c++) cfr[CF_REG ? NPAIR*3+k*6+c : 0] = lds64(cft_s + 8u*(uint32_t)(k*6+c));
        }

        #pragma unroll 1
        for (int j=0; j<ntw; j++)
        {
            mbar_wait(bars_s + 8*stage, parity);
            const int sA = (warp + j*NW)*64 + 2*lane;           /* this lane's samples: sA, sA+1 */
            const bool valid = sA < nsmpl;
            const uint32_t row_s = lane_row_s + stage*TILE_BYTES;
            int x[2*G];
            if ( valid )
            {
                if constexpr ( (2*G*4) % 16 == 0 )
                {
                    #pragma unroll
                    for (int i=0; i<2*G; i+=4) { const int4 v = lds128(row_s + 4u*i); x[i] = v.x; x[i+1] = v.y; x[i+2] = v.z; x[i+3] = v.w; }
                }
                else
                {
                    #pragma unroll
                    for (int i=0; i<2*G; i+=2) { const int2 v = mm_lds64i(row_s + 4u*i); x[i] = v.x; x[i+1] = v.y; }
                }
            }
            else
            {
                #pragma unroll
                for (int i=0; i<2*G; i++) x[i] = 0;
            }
            __syncwarp();
            if ( lane==0 && j+nst < ntw ) { fence_proxy_async(); issue(site_pl, j+nst, stage); }       /* tile j+nst reuses this stage */
            if ( ++stage==(uint32_t)nst ) { stage = 0; parity ^= 1u; }
            if ( !valid ) continue;

            int orA = 0, orB = 0;
            #pragma unroll
            for (int i=0; i<G; i++) { orA |= x[i]; orB |= x[G+i]; }
            if ( (unsigned)(orA | orB) > 255u )
            {
                /* a missing / vector_end value or a PL >= 256: the int32 row goes on warp 0's list and the sample enters the
                   loop below as a no-data sample (its constant factor is divided out with the other no-data samples) */
                if ( (unsigned)orA > 255u )
                {
                    const int pos = atomicAdd(&sh.nesc, 1);
                    if ( pos < MM_ESC_CAP )
                    {
                        sh.esc[pos] = (unsigned short)sA;
                        #pragma unroll
                        for (int i=0; i<G; i++) sh.esc_pl[pos][i] = x[i];
                    }
                    #pragma unroll
                    for (int i=0; i<G; i++) asm volatile("mov.s32 %0, 0;" : "+r"(x[i]));      /* in place: the common path keeps its registers */
                    orA = 0;
                }
                if ( (unsigned)orB > 255u )
                {
                    const int pos = atomicAdd(&sh.nesc, 1);
                    if ( pos < MM_ESC_CAP )
                    {
                        sh.esc[pos] = (unsigned short)(sA+1);
                        #pragma unroll
                        for (int i=0; i<G; i++) sh.esc_pl[pos][i] = x[G+i];
                    }
                    #pragma unroll
                    for (int i=0; i<G; i++) asm volatile("mov.s32 %0, 0;" : "+r"(x[G+i]));
                    orB = 0;
                }
            }
            double pA[G], pB[G];
            #pragma unroll
            for (int i=0; i<G; i++) { pA[i] = lds64c(pl2p_s + 8u*(uint32_t)x[i]); pB[i] = lds64c(pl2p_s + 8u*(uint32_t)x[G+i]); }
            double sumA = pA[0], sumB = pB[0];
            #pragma unroll
            for (int i=1; i<G; i++) { sumA = __dadd_rn(sumA, pA[i]); sumB = __dadd_rn(sumB, pB[i]); }
            /* PL = 0,..,0: no data (mcall.c:529-537).  Such a sample is multiplied in like any other (its factor is a per-site
               constant that warp 0 divides out) and adds nothing to the integer sums. */
            n0 += (orA==0) + (orB==0);
            #pragma unroll
            for (int k=0; k<NALS; k++) plsum[k] += x[hom_idx(k)] + x[G+hom_idx(k)];    /* mcall.c:607-611 */
            accM[NSET] = __dmul_rn(accM[NSET], __dmul_rn(sumA, sumB));
            #pragma unroll
            for (int xx=1; xx<NALS; xx++)
                #pragma unroll
                for (int yy=0; yy<xx; yy++)
                {
                    const int k = pair_idx(xx,yy);
                    if ( live & (1u<<k) )
                    {
                        double c0, c1, c2;
                        if ( CF_REG ) { c0 = cfr[CF_REG ? k*3 : 0]; c1 = cfr[CF_REG ? k*3+1 : 0]; c2 = cfr[CF_REG ? k*3+2 : 0]; }
                        else { mm_lds_f64x2(cfp_s + 32u*(uint32_t)k, c0, c1); c2 = lds64(cfp_s + 32u*(uint32_t)k + 16u); }
                        const double vA = fma(c2, pA[gt_idx(xx,yy)], fma(c1, pA[hom_idx(yy)], c0*pA[hom_idx(xx)]));
                        const double vB = fma(c2, pB[gt_idx(xx,yy)], fma(c1, pB[hom_idx(yy)], c0*pB[hom_idx(xx)]));
                        accM[k] = __dmul_rn(accM[k], __dmul_rn(vA, vB));
                    }
                }
            #pragma unroll
            for (int xx=2; xx<NALS; xx++)
                #pragma unroll
                for (int yy=1; yy<xx; yy++)
                    #pragma unroll
                    for (int zz=0; zz<yy; zz++)
                    {
                        const int k = tri_idx(xx,yy,zz);
                        if ( live & (1u<<(NPAIR+k)) )
                        {
                            double c0, c1, c2, c3, c4, c5;
                            if ( CF_REG )
                            {
                                c0 = cfr[CF_REG ? NPAIR*3+k*6 : 0];   c1 = cfr[CF_REG ? NPAIR*3+k*6+1 : 0]; c2 = cfr[CF_REG ? NPAIR*3+k*6+2 : 0];
                                c3 = cfr[CF_REG ? NPAIR*3+k*6+3 : 0]; c4 = cfr[CF_REG ? NPAIR*3+k*6+4 : 0]; c5 = cfr[CF_REG ? NPAIR*3+k*6+5 : 0];
                            }
                            else
                            {
                                mm_lds_f64x2(cft_s + 48u*(uint32_t)k, c0, c1); mm_lds_f64x2(cft_s + 48u*(uint32_t)k + 16u, c2, c3);
                                mm_lds_f64x2(cft_s + 48u*(uint32_t)k + 32u, c4, c5);
                            }
                            const double vA = fma(c5, pA[gt_idx(yy,zz)], fma(c4, pA[gt_idx(xx,zz)], fma(c3, pA[gt_idx(xx,yy)],
                                              fma(c2, pA[hom_idx(zz)], fma(c1, pA[hom_idx(yy)], c0*pA[hom_idx(xx)])))));
                            const double vB = fma(c5, pB[gt_idx(yy,zz)], fma(c4, pB[gt_idx(xx,zz)], fma(c3, pB[gt_idx(xx,yy)],
                                              fma(c2, pB[hom_idx(zz)], fma(c1, pB[hom_idx(yy)], c0*pB[hom_idx(xx)])))));
                            accM[NPAIR+k] = __dmul_rn(accM[NPAIR+k], __dmul_rn(vA, vB));
                        }
                    }
            /* the byte-packed copy and the normalisers, for phase 2 */
            const uint32_t prow_s = pack_s + (uint32_t)(sA*RS);
            if constexpr ( NALS<=3 )
            {
                mm_sts32(prow_s,      mm_pack4(x[0],x[1],x[2],x[3]));
                mm_sts32(prow_s + 4u, mm_pack4(x[4],x[5],x[6],x[7]));
                mm_sts32(prow_s + 8u, mm_pack4(x[8],x[9],x[10],x[11]));
            }
            else if constexpr ( NALS==4 )
            {
                mm_sts32(prow_s,       mm_pack4(x[0],x[1],x[2],x[3]));
                mm_sts32(prow_s + 4u,  mm_pack4(x[4],x[5],x[6],x[7]));
                mm_sts32(prow_s + 8u,  mm_pack4(x[8],x[9],x[10],x[11]));
                mm_sts32(prow_s + 12u, mm_pack4(x[12],x[13],x[14],x[15]));
                mm_sts32(prow_s + 16u, mm_pack4(x[16],x[17],x[18],x[19]));
            }
            else
            {
                mm_sts128(prow_s,       mm_pack4(x[0],x[1],x[2],x[3]),     mm_pack4(x[4],x[5],x[6],x[7]),     mm_pack4(x[8],x[9],x[10],x[11]),   mm_pack4(x[12],x[13],x[14],0));
                mm_sts128(prow_s + 16u, mm_pack4(x[15],x[16],x[17],x[18]), mm_pack4(x[19],x[20],x[21],x[22]), mm_pack4(x[23],x[24],x[25],x[26]), mm_pack4(x[27],x[28],x[29],0));
            }
            mm_stg_f64x2(sums_g + sA, sumA, sumB, pol_last);
            if ( ++since == MM_RENORM )         /* ten more samples in every product: split the exponents off before anything can underflow */
            {
                #pragma unroll
                for (int k=0; k<NACC; k++) acc_renorm(accM[k], accE[k]);
                since = 0;
            }
        }
        prefetched = false;

        /* ---- warp reduction through a shared-memory transpose (the warp's ring is idle: every tile was consumed, none is in
                flight): lane k multiplies the 32 partial products of accumulator k (mantissa multiply, exponent add) */
        {
            const uint32_t redM_s = ring_s, redE_s = ring_s + (uint32_t)(NACC*256);
            #pragma unroll
            for (int k=0; k<NACC; k++)
            {
                acc_renorm(accM[k], accE[k]);
                mm_sts_f64(redM_s + (uint32_t)(k*256 + lane*8), accM[k]);
                mm_sts32(redE_s + (uint32_t)(k*128 + lane*4), (uint32_t)accE[k]);
            }
            __syncwarp();
            {
                /* lane (k, seg): accumulator k = lane % KPAD, partials [seg*KPAD, (seg+1)*KPAD) -- rotated by k so that the lanes of a
                   segment start in different banks; the 32/KPAD segments are then combined with shuffles */
                constexpr int KPAD = NACC<=8 ? 8 : (NACC<=16 ? 16 : 32);
                const int k = lane & (KPAD-1), seg = lane / KPAD;
                double M0 = 1.0, M1 = 1.0; int E = 0;
                if ( k < NACC )
                {
                    #pragma unroll
                    for (int i=0; i<KPAD; i+=2)
                    {
                        const int c0 = seg*KPAD + ((i + k) & (KPAD-1)), c1 = seg*KPAD + ((i + 1 + k) & (KPAD-1));
                        M0 = __dmul_rn(M0, lds64(redM_s + (uint32_t)((k*32 + c0)*8)));
                        M1 = __dmul_rn(M1, lds64(redM_s + (uint32_t)((k*32 + c1)*8)));
                        E += lds32(redE_s + (uint32_t)((k*32 + c0)*4)) + lds32(redE_s + (uint32_t)((k*32 + c1)*4));
                    }
                }
                double M = __dmul_rn(M0, M1);           /* at most 32 mantissas in [1,2) meet in one product: < 2^32 */
                #pragma unroll
                for (int off=KPAD; off<32; off<<=1)
                {
                    M = __dmul_rn(M, __shfl_xor_sync(0xffffffffu, M, off));
                    E += __shfl_xor_sync(0xffffffffu, E, off);
                }
                if ( lane < NACC )
                {
                    acc_renorm(M, E);
                    sh.red_M[warp][lane] = M; sh.red_E[warp][lane] = E;
                }
            }
            #pragma unroll
            for (int k=0; k<NALS; k++)
            {
                int v = plsum[k];
                #pragma unroll
                for (int off=16; off; off>>=1) v += __shfl_xor_sync(0xffffffffu, v, off);
                if ( lane==0 ) sh.red_pls[warp][k] = v;
            }
            #pragma unroll
            for (int off=16; off; off>>=1) n0 += __shfl_xor_sync(0xffffffffu, n0, off);
            if ( lane==0 ) sh.red_cnt[warp] = n0;
        }
        __syncthreads();            /* [B] */

        if ( warp==0 ) mm_epilogue<NALS,BLOCK>(&sh, &su, a, lane, pl2p_s, pack_s, sums_g);
        else if ( warp==1 )
        {
            if ( lane==0 ) sh.setup[par^1].isite = atomicAdd(a.work_counter, 1);
            mm_setup<NALS>(&sh.setup[par^1], a, lane, nsites);
        }
        __syncthreads();            /* [D] */

        /* =========================== phase 2: per-sample genotypes ============================== */
        {
            /* the first tiles of the CTA's next site land while this phase computes */
            const MMSetup<NALS> &nx = sh.setup[par^1];
            if ( nx.isite < nsites )
            {
                if ( lane==0 ) issue_first(reinterpret_cast<const int32_t*>(a.pl) + nx.pl_off);
                prefetched = true;
            }
        }
        const int path = sh.path;
        const int npair = nsmpl >> 1;
        if ( path==1 )              /* REF only: mcall_set_ref_genotypes (mcall.c:713-743); the PL tag is dropped */
        {
            int2 *out_gt = reinterpret_cast<int2*>(a.gt) + (size_t)sh.site*nsmpl;
            int32_t *out_gq = a.gq + (size_t)sh.site*nsmpl;
            int called = 0;
            double ns0 = 0, ns1 = 0;            /* the normalisers of the next iteration are fetched (from L2) one iteration ahead */
            if ( tid < npair ) mm_ldg_f64x2(sums_g + 2*tid, ns0, ns1, pol_last);
            #pragma unroll 1
            for (int pr=tid; pr<npair; pr+=BLOCK)
            {
                const double s0 = ns0, s1 = ns1;
                if ( pr + BLOCK < npair ) mm_ldg_f64x2(sums_g + 2*(pr + BLOCK), ns0, ns1, pol_last);
                const bool has0 = s0 > 0 && s0 != (double)G, has1 = s1 > 0 && s1 != (double)G;
                const int g0 = has0 ? MCB_GT_UNPHASED(0) : MCB_GT_MISSING, g1 = has1 ? MCB_GT_UNPHASED(0) : MCB_GT_MISSING;
                called += (int)has0 + (int)has1;
                mm_stg128(out_gt + 2*(size_t)pr, g0, g0, g1, g1);
                mm_stg64(out_gq + 2*(size_t)pr, 0, 0);
            }
            #pragma unroll
            for (int off=16; off; off>>=1) called += __shfl_xor_sync(0xffffffffu, called, off);
            if ( lane==0 && called ) atomicAdd(&sh.ac[0], 2*called);
        }
        else if ( path==2 )         /* the pair {REF, b}, both kept: new genotypes 0/0, 0/1, 1/1 are slots 0, 1, 2 */
        {
            int2 *out_gt = reinterpret_cast<int2*>(a.gt) + (size_t)sh.site*nsmpl;
            int32_t *out_gq = a.gq + (size_t)sh.site*nsmpl;
            int32_t *out_pl = a.out_pl + sh.out_off;
            float w0, w1, w2, wn;
            asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(w0), "=f"(w1), "=f"(w2), "=f"(wn) : "r"(scrw_s));
            asm volatile("ld.shared.f32 %0, [%1+24];" : "=f"(wn) : "r"(scrw_s));
            const bool noscr = wn != 0.f;
            const uint32_t j0 = (uint32_t)sh.jgt[0], j1 = (uint32_t)sh.jgt[1], j2 = (uint32_t)sh.jgt[2];
            int f_alt = 0, f_called = 0;
            double ns0 = 0, ns1 = 0;
            if ( tid < npair ) mm_ldg_f64x2(sums_g + 2*tid, ns0, ns1, pol_last);
            #pragma unroll 1
            for (int pr=tid; pr<npair; pr+=BLOCK)
            {
                const uint32_t rA = pack_s + (uint32_t)(pr*2*RS), rB = rA + RS;
                const double s0 = ns0, s1 = ns1;
                if ( pr + BLOCK < npair ) mm_ldg_f64x2(sums_g + 2*(pr + BLOCK), ns0, ns1, pol_last);
                const uint32_t a0 = mm_ldsu8(rA + j0), b0 = mm_ldsu8(rA + j1), c0 = mm_ldsu8(rA + j2);
                const uint32_t a1 = mm_ldsu8(rB + j0), b1 = mm_ldsu8(rB + j1), c1 = mm_ldsu8(rB + j2);
                int k0, k1, g0, g1;
                const bool ok0 = screen2_call(a0, b0, c0, w0, w1, w2, plf_s, gqw_s, k0, g0);
                const bool ok1 = screen2_call(a1, b1, c1, w0, w1, w2, plf_s, gqw_s, k1, g1);
                const bool has0 = s0 > 0 && s0 != (double)G, has1 = s1 > 0 && s1 != (double)G;     /* PL=0,..,0 / all missing: ./. and GQ 0 */
                if ( (!ok0 || noscr) && has0 ) { const int e = mm_fast2_exact(a0, b0, c0, s0, q_s, pl2p_s, thr_s); k0 = e & 255; g0 = e >> 8; }
                if ( (!ok1 || noscr) && has1 ) { const int e = mm_fast2_exact(a1, b1, c1, s1, q_s, pl2p_s, thr_s); k1 = e & 255; g1 = e >> 8; }
                /* new alleles 0 and 1: GT codes 2 and 4, slot index = copies of allele 1 */
                const int x0 = has0 ? (k0==2 ? 4 : 2) : 0, y0 = has0 ? (k0 ? 4 : 2) : 0;
                const int x1 = has1 ? (k1==2 ? 4 : 2) : 0, y1 = has1 ? (k1 ? 4 : 2) : 0;
                f_alt += (has0 ? k0 : 0) + (has1 ? k1 : 0); f_called += (int)has0 + (int)has1;
                mm_stg128(out_gt + 2*(size_t)pr, x0, y0, x1, y1);
                mm_stg64(out_gq + 2*(size_t)pr, has0 ? g0 : 0, has1 ? g1 : 0);
                int32_t *dst = out_pl + 6*(size_t)pr;           /* mcall.c:1158-1194: the kept genotypes are the three slots */
                mm_stg64(dst, (int)a0, (int)b0); mm_stg64(dst + 2, (int)c0, (int)a1); mm_stg64(dst + 4, (int)b1, (int)c1);
                if ( s0 < 0 || s1 < 0 )     /* the int32 row holds sentinels: the output row carries them (same thread: ordered after the stores above) */
                {
                    const int jg[3] = { (int)j0, (int)j1, (int)j2 };
                    if ( s0 < 0 ) mm_raw_pl_row<NALS>(site_pl + (size_t)(2*pr)*G, su.unseen, jg, 3, dst);
                    if ( s1 < 0 ) mm_raw_pl_row<NALS>(site_pl + (size_t)(2*pr+1)*G, su.unseen, jg, 3, dst + 3);
                }
            }
            #pragma unroll
            for (int off=16; off; off>>=1) { f_alt += __shfl_xor_sync(0xffffffffu, f_alt, off); f_called += __shfl_xor_sync(0xffffffffu, f_called, off); }
            if ( lane==0 && f_called ) { atomicAdd(&sh.ac[0], 2*f_called - f_alt); atomicAdd(&sh.ac[1], f_alt); }
        }
        else if ( path==3 )         /* the triple {REF, b, c}, all kept: slot k = new genotype k */
        {
            int2 *out_gt = reinterpret_cast<int2*>(a.gt) + (size_t)sh.site*nsmpl;
            int32_t *out_gq = a.gq + (size_t)sh.site*nsmpl;
            int32_t *out_pl = a.out_pl + sh.out_off;
            float w[6], wn;
            asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(w[0]), "=f"(w[1]), "=f"(w[2]), "=f"(w[3]) : "r"(scrw_s));
            asm volatile("ld.shared.v2.f32 {%0,%1}, [%2+16];" : "=f"(w[4]), "=f"(w[5]) : "r"(scrw_s));
            asm volatile("ld.shared.f32 %0, [%1+24];" : "=f"(wn) : "r"(scrw_s));
            const bool noscr = wn != 0.f;
            uint32_t jg[6];
            #pragma unroll
            for (int k=0; k<6; k++) jg[k] = (uint32_t)sh.jgt[k];
            unsigned long long acc = 0;     /* AC: 12-bit counters, new allele j at bits [12j,12j+12); the launcher keeps samples per thread <= 40 */
            double ns0 = 0, ns1 = 0;
            if ( tid < npair ) mm_ldg_f64x2(sums_g + 2*tid, ns0, ns1, pol_last);
            #pragma unroll 1
            for (int pr=tid; pr<npair; pr+=BLOCK)
            {
                const uint32_t rA = pack_s + (uint32_t)(pr*2*RS), rB = rA + RS;
                const double s0 = ns0, s1 = ns1;
                if ( pr + BLOCK < npair ) mm_ldg_f64x2(sums_g + 2*(pr + BLOCK), ns0, ns1, pol_last);
                uint32_t vA[6], vB[6];
                #pragma unroll
                for (int k=0; k<6; k++) { vA[k] = mm_ldsu8(rA + jg[k]); vB[k] = mm_ldsu8(rB + jg[k]); }
                int32_t *dst = out_pl + 12*(size_t)pr;
                mm_stg128(dst,     (int)vA[0], (int)vA[1], (int)vA[2], (int)vA[3]);
                mm_stg128(dst + 4, (int)vA[4], (int)vA[5], (int)vB[0], (int)vB[1]);
                mm_stg128(dst + 8, (int)vB[2], (int)vB[3], (int)vB[4], (int)vB[5]);
                int k0, k1, g0, g1;
                const bool ok0 = screen3_call(vA, w, plf_s, gqw_s, k0, g0);
                const bool ok1 = screen3_call(vB, w, plf_s, gqw_s, k1, g1);
                const bool has0 = s0 > 0 && s0 != (double)G, has1 = s1 > 0 && s1 != (double)G;
                if ( (!ok0 || noscr) && has0 ) { const int e = mm_fast3_exact(rA, jgt_s, s0, q_s, pl2p_s, thr_s); k0 = e & 255; g0 = e >> 8; }
                if ( (!ok1 || noscr) && has1 ) { const int e = mm_fast3_exact(rB, jgt_s, s1, q_s, pl2p_s, thr_s); k1 = e & 255; g1 = e >> 8; }
                const int4 o0 = lds128(slot_s + 16u*(uint32_t)(has0 ? k0 : 6));
                const int4 o1 = lds128(slot_s + 16u*(uint32_t)(has1 ? k1 : 6));
                acc += ((unsigned long long)(uint32_t)o0.z | ((unsigned long long)(uint32_t)o0.w << 32))
                     + ((unsigned long long)(uint32_t)o1.z | ((unsigned long long)(uint32_t)o1.w << 32));
                mm_stg128(out_gt + 2*(size_t)pr, o0.x, o0.y, o1.x, o1.y);
                mm_stg64(out_gq + 2*(size_t)pr, has0 ? g0 : 0, has1 ? g1 : 0);
                if ( s0 < 0 || s1 < 0 )
                {
                    int jgi[6];
                    #pragma unroll
                    for (int k=0; k<6; k++) jgi[k] = (int)jg[k];
                    if ( s0 < 0 ) mm_raw_pl_row<NALS>(site_pl + (size_t)(2*pr)*G, su.unseen, jgi, 6, dst);
                    if ( s1 < 0 ) mm_raw_pl_row<NALS>(site_pl + (size_t)(2*pr+1)*G, su.unseen, jgi, 6, dst + 6);
                }
            }
            #pragma unroll
            for (int off=16; off; off>>=1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
            if ( lane==0 )
            {
                #pragma unroll
                for (int j=0; j<3; j++)
                {
                    const int c = (int)((acc >> (12*j)) & 0xfff);
                    if ( c ) atomicAdd(&sh.ac[j], c);
                }
            }
        }
        par ^= 1;
    }
}

/* ------------------------------------------------------------------------------------------------
 *  launcher
 * ---------------------------------------------------------------------------------------------- */
template<int NALS, int BLOCK> static size_t mm_smem(int nsmpl, int nst)
{
    const int ntiles = (nsmpl + 63) >> 6, spad = ntiles*64;
    return align128(sizeof(MMShared<NALS,BLOCK>)) + (size_t)(BLOCK/32)*mm_warp_region(MMGeom<NALS>::TILE_BYTES, MMGeom<NALS>::RED_BYTES, nst)
         + align128((size_t)spad*MMGeom<NALS>::RS);
}
template<int NALS, int BLOCK> static cudaError_t mm_launch(const KArgs *a, int nsmpl, int nst, int grid, cudaStream_t st, size_t *smem_out, int *nb)
{
    auto kern = mcall_multi_kernel<NALS,BLOCK>;
    const size_t smem = mm_smem<NALS,BLOCK>(nsmpl, nst);
    if ( smem_out ) *smem_out = smem;
    if ( !a && !nb ) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if ( e!=cudaSuccess ) return e;
    if ( nb ) return cudaOccupancyMaxActiveBlocksPerMultiprocessor(nb, kern, BLOCK, smem);
    kern<<<grid, BLOCK, smem, st>>>(*a);
    return cudaGetLastError();
}
template<int NALS> static cudaError_t mm_dispatch(int block, const KArgs *a, int nsmpl, int nst, int grid, cudaStream_t st, size_t *smem_out, int *nb)
{
    switch ( block )
    {
        case 64:  return mm_launch<NALS,64>(a, nsmpl, nst, grid, st, smem_out, nb);
        case 128: return mm_launch<NALS,128>(a, nsmpl, nst, grid, st, smem_out, nb);
        case 256: return mm_launch<NALS,256>(a, nsmpl, nst, grid, st, smem_out, nb);
    }
    return cudaErrorInvalidValue;
}
static cudaError_t mm_dispatch_nals(int nals, int block, const KArgs *a, int nsmpl, int nst, int grid, cudaStream_t st, size_t *smem_out, int *nb)
{
    switch ( nals )
    {
        case 3: return mm_dispatch<3>(block, a, nsmpl, nst, grid, st, smem_out, nb);
        case 4: return mm_dispatch<4>(block, a, nsmpl, nst, grid, st, smem_out, nb);
        case 5: return mm_dispatch<5>(block, a, nsmpl, nst, grid, st, smem_out, nb);
    }
    return cudaErrorInvalidValue;
}

/*  Smallest CTA size for a sample count: the 12-bit allele counters of phase 2 allow 40 samples per thread.  0: the sample
 *  count is out of this kernel's range (odd, too small to fill two warps, too large for the shared-memory copy).  */
int multi_block_for(int nsmpl)
{
    if ( (nsmpl & 1) || nsmpl < 128 ) return 0;
    if ( nsmpl <= 2560 ) return 64;
    if ( nsmpl <= 5120 ) return 128;
    if ( nsmpl <= 10240 ) return 256;
    return 0;
}
size_t multi_smem_bytes(int nals, int block, int nsmpl, int nst)
{
    size_t smem = 0;
    if ( mm_dispatch_nals(nals, block, nullptr, nsmpl, nst, 0, nullptr, &smem, nullptr)!=cudaSuccess ) return 0;
    return smem;
}
size_t multi_scratch_bytes(int nsmpl, int grid) { return (size_t)grid*(size_t)(((nsmpl + 63) >> 6)*64)*sizeof(double); }
cudaError_t multi_kernel_occupancy(int nals, int block, int nsmpl, int nst, int *blocks_per_sm)
{
    return mm_dispatch_nals(nals, block, nullptr, nsmpl, nst, 0, nullptr, nullptr, blocks_per_sm);
}
cudaError_t launch_multi_kernel(int nals, int block, const KArgs &a, int grid, cudaStream_t st)
{
    return mm_dispatch_nals(nals, block, &a, a.nsmpl, a.nstage, grid, st, nullptr, nullptr);
}

}   // namespace mcb
