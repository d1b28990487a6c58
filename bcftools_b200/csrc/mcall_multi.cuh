/*  mcall_multi.cuh -- what the site kernels of the multi-allelic classes share: the CTA-per-site kernel of the 3-5 allele
 *  classes (mcall_multi.cu) and the warp-per-site kernels of the 3-allele class (mcall_triallelic.cu) and of the 4-allele
 *  class (mcall_multi_warp.cu).  Per-site set-up, the
 *  general path of a sample with missing values, the allele-set decision and the site record, and the literal FP64 calls of
 *  phase 2.  A kernel keeps its decision record in a struct of its own; the templates below read and write it by member name.  */
#pragma once
#include "mcall_device.cuh"

namespace mcb {

#define MM_ESC_CAP   32             /* samples per site that may take the general path (one lane of warp 0 each) */
#define MM_RENORM    5              /* iterations (pairs of samples per lane) between exponent splits of the running products */
#ifndef MM_SCREEN
#define MM_SCREEN    1              /* 1: float32 screen in front of the literal FP64 call of phase 2 (0: every sample takes the literal path) */
#endif

template<int NALS> struct MMGeom
{
    static constexpr int G  = Shape<NALS>::G;
    static constexpr int RS = NALS<=3 ? 6 : (NALS==4 ? 10 : 16);       /* bytes per sample of the packed copy */
    static constexpr int TILE_BYTES = 64*G*4;                           /* one warp tile: 64 samples of int32 PLs */
    static constexpr int NSET = Shape<NALS>::NPAIR + Shape<NALS>::NTRI;
    static constexpr int NACC = NSET + 1;
    static constexpr int RED_BYTES = NACC*32*12;                        /* warp reduction: one (mantissa, exponent) per lane and product */
};

/*  per-site set-up (the CTA kernel double-buffers it: warp 1 writes the NEXT site's while warp 0 evaluates the current one)  */
template<int NALS> struct __align__(16) MMSetup
{
    using S = Shape<NALS>;
    double   cfp[S::NPAIR][4];          /* pair (x>y): fa2 (x/x), fb2 (y/y), 2 fa fb (x/y), unused      mcall.c:629-633 */
    double   cft[S::NTRI][6];           /* triple (x>y>z): fa2 fb2 fc2 2fafb 2fafc 2fbfc                 mcall.c:671-677 */
    double   logv0[MMGeom<NALS>::NSET]; /* log of the set's value for a sample with every PL = 0 */
    float    qf[NALS];
    uint32_t live, flags;
    int      isite, site, unseen;
    long long pl_off;
};

/*  The CTA kernel's row of normalisers is rewritten every site and read back ~50 us later, while PL blocks and results stream
 *  through L2 at several TB/s: without a hint the row is evicted before its reuse (ncu: its reads all went to DRAM).  evict_last keeps it.  */
__device__ __forceinline__ uint64_t mm_policy_evict_last() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p; }
__device__ __forceinline__ void mm_sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t mm_ldsu8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void mm_stg128(void *p, int x, int y, int z, int w)
{
    asm volatile("st.global.cs.v4.s32 [%0], {%1,%2,%3,%4};" :: "l"(p), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");     /* results stream out: evict first */
}
__device__ __forceinline__ void mm_stg64(void *p, int x, int y) { asm volatile("st.global.cs.v2.s32 [%0], {%1,%2};" :: "l"(p), "r"(x), "r"(y) : "memory"); }
__device__ __forceinline__ void mm_stg32(void *p, int x) { asm volatile("st.global.cs.s32 [%0], %1;" :: "l"(p), "r"(x) : "memory"); }
__device__ __forceinline__ uint32_t mm_pack4(int a, int b, int c, int d) { return (uint32_t)a | (uint32_t)b<<8 | (uint32_t)c<<16 | (uint32_t)d<<24; }
/*  byte j of a packed row: a 32-bit shared address, or a generic pointer (the warp kernel of the 4-allele class keeps part
 *  of its packed copy in global memory)  */
__device__ __forceinline__ uint32_t mm_row_u8(uint32_t row_s, uint32_t j) { return mm_ldsu8(row_s + j); }
__device__ __forceinline__ uint32_t mm_row_u8(const uint8_t *row, uint32_t j) { return row[j]; }
__device__ __forceinline__ void mm_row_st8(uint32_t row_s, uint32_t j, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" :: "r"(row_s + j), "r"(v) : "memory"); }
__device__ __forceinline__ void mm_row_st8(uint8_t *row, uint32_t j, uint32_t v) { row[j] = (uint8_t)v; }

static __device__ __noinline__ double mm_log(double x) { return log(x); }
static __device__ __noinline__ double mm_exp(double x) { return exp(x); }
/*  set_pdg's missing-value fill (mcall.c:495-527) on a local copy of one sample's PL vector; returns 0 for "no data"
 *  (same rules as fix_missing in mcall_kernels.cu, including the values it leaves behind when it gives up)  */
static __device__ __noinline__ int mm_fix_missing(int *pl, int nals, int unseen)
{
    const int G = nals*(nals+1)/2;
    int j;
    for (j=0; j<G; j++)
    {
        if ( pl[j]==I32_VEC_END ) return 0;     /* not diploid-shaped: all missing, mcall.c:465-470 */
        if ( pl[j]==I32_MISSING ) break;
    }
    if ( j==0 || j==G ) return 0;               /* first value missing (mcall.c:476-481) / negative garbage that is no sentinel */
    j = 0;
    for (int ia=0; ia<nals; ia++)
        for (int ib=0; ib<=ia; ib++)
        {
            if ( pl[j]==I32_MISSING )
            {
                int k = gt_idx(ia,unseen);
                if ( pl[k]==I32_MISSING ) k = gt_idx(ib,unseen);
                if ( pl[k]==I32_MISSING ) k = gt_idx(unseen,unseen);
                pl[j] = pl[k]==I32_MISSING ? 255 : pl[k];
            }
            else if ( pl[j] < 0 ) return 0;     /* vector_end behind a missing value: undefined in the reference */
            j++;
        }
    return 1;
}

/*  per-lane sums of the samples that took the general path (warp 0 reduces them)  */
template<int NALS> struct MMSlow
{
    double lk[MMGeom<NALS>::NSET];      /* sum of log(val) per allele set, mcall.c:635-645, 680-690 */
    double lnN;                         /* sum of log(sum) */
    long long pls[NALS];                /* sum of PL[a/a], the single-allele sets (mcall.c:607-611) */
    int ndata;
    uint32_t punt;
};

/*  One sample on the general path: takes its int32 row, applies the fill, and -- when the sample has data and every value
 *  fits a byte -- adds its terms to `acc` and stores the filled packed row (and, where the kernel keeps a row of normalisers,
 *  sum_g != nullptr, the normaliser), so that phase 2 treats it like any other sample.  No data: packed zeros; sum = -1 when
 *  the row still holds sentinels (phase 2 then re-derives the output row from the int32 values), +G otherwise.
 *  Returns "the row still holds sentinels and carries no data".  */
template<int NALS, class RowT>
static __device__ __noinline__ bool mm_slow_sample(const int *row, const MMSetup<NALS> *su, uint32_t pl2p_s, RowT dst, double *sum_g, MMSlow<NALS> *acc)
{
    using S = Shape<NALS>;
    constexpr int G = S::G, RS = MMGeom<NALS>::RS;
    int pl[G]; double p[G];
    int orv = 0;
    for (int j=0; j<G; j++) { pl[j] = row[j]; orv |= pl[j]; }
    bool data = orv != 0, raw = false;
    if ( orv < 0 )
    {
        data = mm_fix_missing(pl, NALS, su->unseen);
        raw = !data;
        if ( data ) { orv = 0; for (int j=0; j<G; j++) orv |= pl[j]; data = orv > 0; }
    }
    if ( data && (unsigned)orv > 255u ) { acc->punt = 1; data = false; }    /* PL >= 256: the general kernel owns this site */
    double sum = raw ? -1.0 : (double)G;
    if ( data )
    {
        for (int j=0; j<G; j++) p[j] = lds64(pl2p_s + 8u*(uint32_t)pl[j]);
        sum = p[0];
        for (int j=1; j<G; j++) sum = __dadd_rn(sum, p[j]);
        acc->ndata++;
        acc->lnN += mm_log(sum);
        for (int k=0; k<NALS; k++) acc->pls[k] += pl[hom_idx(k)];
        int k = 0;
        #pragma unroll 1
        for (int x=1; x<NALS; x++)
            #pragma unroll 1
            for (int y=0; y<x; y++, k++)
                if ( su->live & (1u<<k) )
                {
                    const double *c = su->cfp[k];
                    const double val = fma(c[2], p[gt_idx(x,y)], fma(c[1], p[hom_idx(y)], c[0]*p[hom_idx(x)]));
                    acc->lk[k] += mm_log(val);
                }
        #pragma unroll 1
        for (int x=2; x<NALS; x++)
            #pragma unroll 1
            for (int y=1; y<x; y++)
                #pragma unroll 1
                for (int z=0; z<y; z++, k++)
                    if ( su->live & (1u<<k) )
                    {
                        const double *c = su->cft[k - S::NPAIR];
                        const double val = fma(c[5], p[gt_idx(y,z)], fma(c[4], p[gt_idx(x,z)], fma(c[3], p[gt_idx(x,y)],
                                           fma(c[2], p[hom_idx(z)], fma(c[1], p[hom_idx(y)], c[0]*p[hom_idx(x)])))));
                        acc->lk[k] += mm_log(val);
                    }
    }
    for (int j=0; j<RS; j++) mm_row_st8(dst, (uint32_t)j, (data && j<G) ? (uint32_t)pl[j] : 0u);
    if ( sum_g ) asm volatile("st.global.cg.L2::cache_hint.f64 [%0], %1, %2;" :: "l"(sum_g), "d"(sum), "l"(mm_policy_evict_last()) : "memory");
    return raw;
}

/*  qsum (mcall.c:1454-1464), -F prior (1507-1527), normalisation (1530-1535) by lane 0, then the allele-set
 *  coefficients one lane per set: float32 expression then widened (mcall.c:629-630, 671-673).  One warp.  */
template<int NALS>
static __device__ __noinline__ void mm_setup(MMSetup<NALS> *su, const KArgs &a, int lane, int nsites)
{
    using S = Shape<NALS>;
    constexpr int NPAIR = S::NPAIR, NTRI = S::NTRI;
    __syncwarp();
    const int isite = su->isite;
    if ( isite >= nsites ) return;
    const int site = a.site_list[isite];
    const int nsmpl = a.nsmpl;
    if ( lane==0 )
    {
        int nqs = a.nqs ? a.nqs[site] : NALS;
        float q[NALS];
        #pragma unroll
        for (int j=0; j<NALS; j++) q[j] = (a.qs && j<nqs) ? a.qs[(size_t)site*a.max_nals + j] : 0.f;
        uint32_t flags = (a.qs && nqs>0) ? 0 : MCB_SITE_NO_QS;
        if ( a.use_prior && a.prior_an && a.prior_ac )
        {
            int an = a.prior_an[site];
            if ( an!=I32_MISSING && an>0 )
            {
                const int32_t *pac = a.prior_ac + (size_t)site*a.max_nals;
                int ac0 = an;
                for (int j=0; j<NALS-1; j++)
                {
                    if ( pac[j]==I32_VEC_END ) break;
                    if ( pac[j]==I32_MISSING ) continue;
                    ac0 -= pac[j];
                    q[j+1] = (float)( __ddiv_rn(__dadd_rn((double)q[j+1], __dmul_rn(0.5,(double)pac[j])),
                                                __dadd_rn((double)(uint32_t)nsmpl, __dmul_rn(0.5,(double)an))) );
                }
                if ( ac0<0 ) flags |= MCB_SITE_BAD_PRIOR;
                q[0] = (float)( __ddiv_rn(__dadd_rn((double)q[0], __dmul_rn(0.5,(double)ac0)),
                                          __dadd_rn((double)(uint32_t)nsmpl, __dmul_rn(0.5,(double)an))) );
            }
        }
        float qsum = 0;
        #pragma unroll
        for (int j=0; j<NALS; j++) qsum = __fadd_rn(qsum, q[j]);
        if ( qsum != 0 )
        {
            #pragma unroll
            for (int j=0; j<NALS; j++) q[j] = __fdiv_rn(q[j], qsum);
        }
        #pragma unroll
        for (int j=0; j<NALS; j++) su->qf[j] = q[j];
        su->flags = flags;
        su->site = site;
        su->unseen = a.unseen ? a.unseen[site] : 0;
        su->pl_off = a.pl_off[site];
    }
    __syncwarp();
    uint32_t live = 0;
    if ( lane < NPAIR )
    {
        int aa = 1; while ( aa*(aa+1)/2 <= lane ) aa++;     /* pair_idx(aa,bb)==lane */
        int bb = lane - aa*(aa-1)/2;
        float qa = su->qf[aa], qb = su->qf[bb];
        double *cf = su->cfp[lane];
        cf[0] = cf[1] = cf[2] = cf[3] = 0;
        double v0 = 1.0;
        if ( qa!=0 && qb!=0 )
        {
            float den = __fadd_rn(qa,qb);
            double fa = (double)__fdiv_rn(qa,den), fb = (double)__fdiv_rn(qb,den);
            cf[0] = __dmul_rn(fa,fa); cf[1] = __dmul_rn(fb,fb); cf[2] = __dmul_rn(__dmul_rn(2.0,fa),fb);
            v0 = fma(cf[2], 1.0, fma(cf[1], 1.0, cf[0]*1.0));
            live = 1u<<lane;
        }
        su->logv0[lane] = mm_log(v0);
    }
    else if ( lane-NPAIR < NTRI )
    {
        int k = lane-NPAIR;
        int aa = 2; while ( (aa+1)*aa*(aa-1)/6 <= k ) aa++;
        int r = k - aa*(aa-1)*(aa-2)/6;
        int bb = 1; while ( bb*(bb+1)/2 <= r ) bb++;
        int cc = r - bb*(bb-1)/2;
        float qa = su->qf[aa], qb = su->qf[bb], qc = su->qf[cc];
        double *cf = su->cft[k];
        for (int j=0; j<6; j++) cf[j] = 0;
        double v0 = 1.0;
        if ( qa!=0 && qb!=0 && qc!=0 )
        {
            float den = __fadd_rn(__fadd_rn(qa,qb),qc);
            double fa = (double)__fdiv_rn(qa,den), fb = (double)__fdiv_rn(qb,den), fc = (double)__fdiv_rn(qc,den);
            cf[0] = __dmul_rn(fa,fa); cf[1] = __dmul_rn(fb,fb); cf[2] = __dmul_rn(fc,fc);
            cf[3] = __dmul_rn(__dmul_rn(2.0,fa),fb); cf[4] = __dmul_rn(__dmul_rn(2.0,fa),fc); cf[5] = __dmul_rn(__dmul_rn(2.0,fb),fc);
            v0 = fma(cf[5], 1.0, fma(cf[4], 1.0, fma(cf[3], 1.0, fma(cf[2], 1.0, fma(cf[1], 1.0, cf[0]*1.0)))));
            live = 1u<<lane;
        }
        su->logv0[lane] = mm_log(v0);
    }
    #pragma unroll
    for (int off=16; off; off>>=1) live |= __shfl_xor_sync(0xffffffffu, live, off);
    if ( lane==0 ) su->live = live;
    __syncwarp();
}

/*  site record: QUAL (mcall.c:1631-1645), AC/AN (1648-1650).  One thread, after phase 2 of the site has been joined.  */
template<int NALS, class Rec>
static __device__ __noinline__ void mm_finalize(Rec *shp, const KArgs &a)
{
    Rec &sh = *shp;
    const int site = sh.site;
    int nAC = 0;
    if ( !sh.ref_gt ) for (int j=1; j<sh.nals_new && j<8; j++) nAC += sh.ac[j];
    int ret = sh.nals_new;
    if ( !sh.ref_gt && !nAC && (a.flag & MCB_CALL_VARONLY) ) ret = 0;      /* mcall.c:1618 */
    float qual;
    if ( nAC ) qual = (float)sh.max_qual;
    else if ( sh.lk_sum != -CUDART_INF ) qual = (float)(-4.343*(sh.lk_sum - sh.lse));
    else if ( sh.ac[0] ) qual = a.theta ? (float)(-4.343*a.theta) : 0.f;
    else qual = __uint_as_float(MCB_FLOAT_MISSING_BITS);
    a.ret[site] = ret;
    if ( a.als_new ) a.als_new[site] = sh.als_new;
    if ( a.als_map ) for (int j=0; j<a.max_nals; j++) a.als_map[(size_t)site*a.max_nals + j] = j<NALS ? (int8_t)sh.als_map[j] : (int8_t)-1;
    if ( a.qual ) a.qual[site] = qual;
    if ( a.ac ) for (int j=0; j<a.max_nals; j++) a.ac[(size_t)site*a.max_nals + j] = (j<sh.nals_new && j<8) ? sh.ac[j] : 0;
    if ( a.an ) a.an[site] = nAC + sh.ac[0];
    if ( a.site_flags ) a.site_flags[site] = sh.flags;
    if ( a.diag ) { double *d = a.diag + (size_t)site*4; d[0] = sh.max_qual; d[1] = sh.lk_sum; d[2] = sh.ref_lk; d[3] = sh.gap; }
}

/*  Between the phases, one warp: the samples on the general path (lane i takes the i-th listed one: sample esc_s with its
 *  int32 row at esc_row), then lane k <-> allele set k in the reference's enumeration order (mcall.c:600-700), the best set,
 *  QUAL candidates, trimming maps and the phase-2 constants, written to the kernel's record `sh`.  From the main loop:
 *  tl = log of the product over its samples of the lane's allele set (lanes NALS.. with a live set) or of the normalisers
 *  (lane 31), n0 = the samples that went through it without data, ps = sum of PL[lane/lane] (lanes < NALS).
 *  esc_dst: the packed row of the lane's listed sample.  ACB: bits per allele of the AC increments in slot_out.
 *  Returns "the lane's listed sample holds sentinels and no data".  */
template<int NALS, int ACB, class Rec, class RowT>
static __device__ __noinline__ bool mm_decide(Rec *shp, const MMSetup<NALS> *su, const KArgs &a, int lane, uint32_t pl2p_s, RowT esc_dst,
                                              int nesc_raw, const int *esc_row, double *esc_sum, double tl, int n0, long long ps)
{
    using S = Shape<NALS>;
    using GE = MMGeom<NALS>;
    constexpr int G = S::G, NPAIR = S::NPAIR, NSUB = S::NSUB, NSET = GE::NSET;
    constexpr double LN10_10 = 0.2302585092994045684017991454684;
    constexpr double LOG_G = G==6 ? 1.791759469228055000812477358381 : (G==10 ? 2.302585092994045684017991454684 : 2.708050201102210065996004570148);   /* ln 6, ln 10, ln 15 */
    Rec &sh = *shp;
    const int site = su->site, unseen = su->unseen, nsmpl = a.nsmpl;
    const uint32_t live = su->live;

    /* ---- samples on the general path, one per lane ---- */
    MMSlow<NALS> sl;
    for (int k=0; k<NSET; k++) sl.lk[k] = 0;
    for (int k=0; k<NALS; k++) sl.pls[k] = 0;
    sl.lnN = 0; sl.ndata = 0; sl.punt = 0;
    bool raw = false;
    const int nesc = min(nesc_raw, MM_ESC_CAP);
    if ( nesc_raw > MM_ESC_CAP ) sl.punt = 1;
    else if ( lane < nesc ) raw = mm_slow_sample<NALS>(esc_row, su, pl2p_s, esc_dst, esc_sum, &sl);
    if ( __any_sync(0xffffffffu, nesc>0) )
    {
        #pragma unroll 1
        for (int k=0; k<NSET; k++)
        {
            double v = sl.lk[k];
            #pragma unroll
            for (int off=16; off; off>>=1) v += __shfl_xor_sync(0xffffffffu, v, off);
            sl.lk[k] = v;
        }
        #pragma unroll 1
        for (int k=0; k<NALS; k++)
        {
            long long v = sl.pls[k];
            #pragma unroll
            for (int off=16; off; off>>=1) v += __shfl_xor_sync(0xffffffffu, v, off);
            sl.pls[k] = v;
        }
        #pragma unroll
        for (int off=16; off; off>>=1)
        {
            sl.lnN += __shfl_xor_sync(0xffffffffu, sl.lnN, off);
            sl.ndata += __shfl_xor_sync(0xffffffffu, sl.ndata, off);
        }
    }
    const bool punt_esc = __any_sync(0xffffffffu, sl.punt != 0);

    /* ---- totals ---- */
    const int n_all = nsmpl - n0 + sl.ndata;            /* samples with data: every sample went through the main loop, n0 of them as no-data samples */
    /* the normaliser (lane 31, next to the allele sets of the other lanes): samples without data were multiplied in with sum = G exactly */
    double lk = 0; bool cand = false, in_sum = false; uint32_t mask = 0;
    const double lnN_all = n_all ? __shfl_sync(0xffffffffu, tl, 31) - (double)n0*LOG_G + sl.lnN : 0.0;
    if ( lane < NALS )
    {
        long long pss = 0;
        #pragma unroll
        for (int k=0; k<NALS; k++) if ( k==lane ) pss = sl.pls[k];
        ps += pss;
        const bool set = n_all > 0;
        lk = set ? -LN10_10*(double)ps - lnN_all : 0.0;
        if ( lane>0 ) lk += a.theta;
        cand = set; in_sum = set && lane>0; mask = 1u<<lane;
    }
    else if ( lane < NSUB )
    {
        const int k = lane - NALS;                  /* accumulator index: pairs then triples */
        const bool lv = (live >> k) & 1u;
        const bool set = lv && n_all > 0;
        int nonref = 0;
        if ( k < NPAIR )
        {
            int aa = 1; while ( aa*(aa+1)/2 <= k ) aa++;
            int bb = k - aa*(aa-1)/2;
            mask = 1u<<aa | 1u<<bb; nonref = (aa!=0) + (bb!=0);
        }
        else
        {
            int kk = k - NPAIR;
            int aa = 2; while ( (aa+1)*aa*(aa-1)/6 <= kk ) aa++;
            int r = kk - aa*(aa-1)*(aa-2)/6;
            int bb = 1; while ( bb*(bb+1)/2 <= r ) bb++;
            int cc = r - bb*(bb-1)/2;
            mask = 1u<<aa | 1u<<bb | 1u<<cc; nonref = (aa!=0) + (bb!=0) + (cc!=0);
        }
        double slk = 0;
        #pragma unroll 1
        for (int j=0; j<NSET; j++) if ( j==k ) slk = sl.lk[j];
        lk = set ? (tl - (double)n0*su->logv0[k] + slk) - lnN_all : 0.0;
        for (int j=0; j<nonref; j++) lk += a.theta;
        cand = set; in_sum = set;
    }
    /* first strict maximum in enumeration order (UPDATE_MAX_LKs, mcall.c:582-585) */
    double best = cand ? lk : -CUDART_INF; int best_lane = cand ? lane : 64;
    #pragma unroll
    for (int off=16; off; off>>=1)
    {
        double ob = __shfl_xor_sync(0xffffffffu, best, off);
        int    ol = __shfl_xor_sync(0xffffffffu, best_lane, off);
        if ( ob > best || (ob==best && ol < best_lane) ) { best = ob; best_lane = ol; }
    }
    double second = (cand && lane!=best_lane) ? lk : -CUDART_INF;
    #pragma unroll
    for (int off=16; off; off>>=1) second = fmax(second, __shfl_xor_sync(0xffffffffu, second, off));
    /* lk_sum = log sum exp over every evaluated set except {REF} (mcall.c:584, 614), and with it
     *     lse = logsumexp2(lk_sum, ref_lk) = log(1 + exp(lo - hi)) + hi          (mcall.c:573-579, 1554, 1640)
     * With term = sum exp(lk - mx) and R = exp(ref_lk - mx) from the same round of exp(): exp(lo - hi) = min(term/R, R/term),
     * so lanes 0 and 1 take log(term) and log(1 + e) side by side: three transcendental latencies on this warp's critical
     * path (log of the products, exp, log) instead of five.  */
    double mx = in_sum ? lk : -CUDART_INF;
    #pragma unroll
    for (int off=16; off; off>>=1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, off));
    const bool have_sum = mx > -CUDART_INF;
    const double ex = (cand && have_sum) ? mm_exp(lk - mx) : 0.0;
    double term = in_sum ? ex : 0.0;
    #pragma unroll
    for (int off=16; off; off>>=1) term += __shfl_xor_sync(0xffffffffu, term, off);
    const double R = __shfl_sync(0xffffffffu, ex, 0);                   /* lane 0 = {REF} */
    const double e = have_sum ? (term > R ? __ddiv_rn(R, term) : __ddiv_rn(term, R)) : 0.0;
    double lg = 0;
    if ( lane < 2 ) lg = mm_log(lane==0 ? term : __dadd_rn(1.0, e));
    const double grp_lk_sum = have_sum ? mx + __shfl_sync(0xffffffffu, lg, 0) : -CUDART_INF;
    const double grp_ref_lk = __shfl_sync(0xffffffffu, lk, 0);
    const double grp_lse = __shfl_sync(0xffffffffu, lg, 1) + (grp_lk_sum > grp_ref_lk ? grp_lk_sum : grp_ref_lk);
    const uint32_t grp_als = __shfl_sync(0xffffffffu, mask, best_lane & 31);

    if ( lane==0 )
    {
        const bool any = best_lane < 64;
        const uint32_t gals = any ? grp_als : 0;
        uint32_t flags = su->flags;
        double max_qual = -CUDART_INF, lk_sum = -CUDART_INF, ref_lk = -CUDART_INF;
        if ( any )          /* mcall.c:1553-1560 */
        {
            max_qual = -4.343*(grp_ref_lk - grp_lse);
            lk_sum = grp_lk_sum; ref_lk = grp_ref_lk;
        }
        const double gap = any ? best - second : CUDART_INF;
        if ( any && gap < a.tie_eps ) flags |= MCB_SITE_NEAR_TIE;
        uint32_t als_new = gals | 1u;               /* mcall.c:1552, 1564 */
        const int is_variant = als_new!=1;
        const int ret_early = ((a.flag & MCB_CALL_VARONLY) && !is_variant) || (flags & MCB_SITE_NO_QS);
        int nals_new = 0;
        #pragma unroll
        for (int j=0; j<NALS; j++)                  /* mcall.c:1569-1575 (no -A here: the launcher keeps such calls on the general kernel) */
        {
            if ( j>0 && j==unseen ) continue;
            if ( als_new & (1u<<j) ) nals_new++;
        }
        int nout = 0;                               /* mcall.c:547-570 */
        #pragma unroll
        for (int x=0; x<NALS; x++) sh.als_map[x] = (als_new & (1u<<x)) ? nout++ : -1;
        const bool unseen_sel = unseen && (als_new & (1u<<unseen));
        const int pl_dropped = als_new==1;
        const int ref_gt = (als_new==1) || !is_variant;
        int gn = 0;
        #pragma unroll
        for (int j=0; j<NALS; j++) gn += (gals>>j)&1u;
        /* what phase 2 has straight-line code for: REF only / {REF,b} / {REF,b,c}, nothing else kept */
        int path = -1;
        if ( !punt_esc && !unseen_sel && !(a.flag & MCB_CALL_KEEPALT) )
        {
            if ( ret_early ) path = 0;
            else if ( ref_gt ) path = 1;
            else if ( als_new==gals && gn==2 && nals_new==2 ) path = 2;
            else if ( als_new==gals && gn==3 && nals_new==3 ) path = 3;
        }
        if ( path < 0 )             /* the general kernel processes this site from scratch */
        {
            a.fb_list[atomicAdd(a.fb_count, 1)] = site;
            sh.path = 0;
        }
        else if ( path==0 )
        {
            a.ret[site] = 0;
            if ( a.site_flags ) a.site_flags[site] = flags;
            if ( a.pl_off_out ) a.pl_off_out[site] = compact_out_off<false>(a, site, nsmpl, NALS, nals_new, false, flags);
            sh.path = 0;
        }
        else
        {
            long long off = su->pl_off;
            if ( a.pl_off_out )
            {
                off = compact_out_off<false>(a, site, nsmpl, NALS, nals_new, !pl_dropped, flags);
                a.pl_off_out[site] = off;
            }
            if ( pl_dropped ) flags |= MCB_SITE_PL_DROPPED;
            if ( ref_gt ) flags |= MCB_SITE_REF_GT;
            sh.path = path; sh.out_off = off; sh.site = site;
            sh.als_new = als_new; sh.nals_new = nals_new; sh.ref_gt = ref_gt; sh.flags = flags;
            sh.max_qual = max_qual; sh.lk_sum = lk_sum; sh.ref_lk = ref_lk; sh.gap = gap; sh.lse = grp_lse;
            /* selected alleles in ascending order and the genotypes they span: slot k = new genotype k */
            int sel[3] = {0,0,0}, ns = 0;
            #pragma unroll
            for (int j=0; j<NALS; j++) if ( (gals>>j)&1u ) { if ( ns<3 ) sel[ns] = j; ns++; }
            if ( ns>3 ) ns = 3;
            for (int x=0; x<3; x++)
            {
                sh.q[x] = x<ns ? (double)su->qf[sel[x]] : 0.0;
                for (int y=0; y<=x; y++)
                {
                    const int k = x*(x+1)/2 + y;
                    sh.jgt[k] = x<ns ? gt_idx(sel[x], sel[y]) : 0;
                    /* gts[0] = smaller new allele, gts[1] = larger (mcall.c:830-831); AC: one count per allele, ACB-bit fields */
                    const unsigned long long inc = (1ull << (ACB*y)) + (1ull << (ACB*x));
                    sh.slot_out[k] = make_int4(MCB_GT_UNPHASED(y), MCB_GT_UNPHASED(x), (int)(uint32_t)inc, (int)(uint32_t)(inc>>32));
                }
            }
            sh.slot_out[6] = make_int4(MCB_GT_MISSING, MCB_GT_MISSING, 0, 0);
            sh.slot_out[7] = make_int4(MCB_GT_MISSING, MCB_GT_MISSING, 0, 0);
            if ( path>=2 )
            {
                bool scr = MM_SCREEN;
                for (int x=0; x<3; x++)
                    for (int y=0; y<=x; y++)
                        sh.scr_w[x*(x+1)/2 + y] = x<path ? screen_weight(sh.q[x], sh.q[y], x==y ? 1.0 : 2.0, scr) : 0.f;
                sh.scr_w[6] = scr ? 0.f : 1.f;
            }
        }
        for (int j=0; j<8; j++) sh.ac[j] = 0;
    }
    return raw;
}

/*  the literal FP64 call of one sample from its packed bytes and its normaliser: the samples the float32 screen does not accept.
 *  q_s: shared address of the selected alleles' q[3].  Returns slot | GQ << 8.  */
static __device__ __noinline__ int mm_fast2_exact(uint32_t a, uint32_t b, uint32_t c, double sum, uint32_t q_s, uint32_t pl2p_s, uint32_t thr_s)
{
    const double q0 = lds64(q_s), q1 = lds64(q_s + 8u);
    int k, g;
    fast2_call(lds64c(pl2p_s + 8u*a), lds64c(pl2p_s + 8u*b), lds64c(pl2p_s + 8u*c), sum, q0, q1, __dmul_rn(2.0, q1), thr_s, k, g);
    return k | g<<8;
}
template<class RowT>
static __device__ __noinline__ int mm_fast3_exact(RowT row, uint32_t jgt_s, double sum, uint32_t q_s, uint32_t pl2p_s, uint32_t thr_s)
{
    const double q0 = lds64(q_s), q1 = lds64(q_s + 8u), q2 = lds64(q_s + 16u);
    double p[6];
    #pragma unroll
    for (int k=0; k<6; k++) p[k] = lds64c(pl2p_s + 8u*mm_row_u8(row, (uint32_t)lds32(jgt_s + 4u*k)));
    int k, g;
    fast3_call(p, sum, q0, q1, q2, __dmul_rn(2.0, q1), __dmul_rn(2.0, q2), thr_s, k, g);
    return k | g<<8;
}

/*  phase 2, rare: the trimmed PL row of a sample whose int32 row holds sentinels and carries no data (mcall.c:1158-1194
 *  copies whatever set_pdg left in PLs[])  */
template<int NALS>
static __device__ __noinline__ void mm_raw_pl_row(const int32_t *grow, int unseen, const int *jgt, int ngt_new, int32_t *dst)
{
    constexpr int G = Shape<NALS>::G;
    int pl[G];
    for (int j=0; j<G; j++) pl[j] = __ldg(grow + j);
    mm_fix_missing(pl, NALS, unseen);
    for (int k=0; k<ngt_new; k++) mm_stg32(dst + k, pl[jgt[k]]);
}

}   // namespace mcb
