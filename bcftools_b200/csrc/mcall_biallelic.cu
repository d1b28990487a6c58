/*  mcall_biallelic.cu -- warp-per-site kernel for the dominant shape of `call -m`: two alleles (REF + one ALT),
 *  int32 PLs, one sample group, no FORMAT/GP (two instances: every sample diploid / any ploidy vector).
 *
 *  Same algorithm and reference line map as the general site kernel (mcall_kernels.cu); what differs is the mapping:
 *
 *    - ONE WARP owns one site, so there is no block barrier, no cross-warp reduction and no idle warps while a
 *      single lane evaluates the allele sets: warps of a CTA only share the read-only tables.
 *    - phase 1 reads the site's PL block straight from global memory, 4 samples (12 int32 = 3 x 128 bit) per lane and
 *      iteration, and leaves a byte-packed copy (3 bytes per sample: PL <= 255 in the common case) in the warp's
 *      private shared-memory buffer.  A 2504-sample site takes 7.5 KB instead of the 30 KB int32 tile, so ~28 warps
 *      stay resident per SM and HBM still sees every PL byte once.
 *    - phase 2 reads the packed copy, calls the 4 genotypes and writes GT / GQ / trimmed PL with 128-bit stores.
 *    - a sample with a value outside 0..255 (missing, vector_end, PL >= 256) is packed as the escape triple
 *      (255,255,255); both phases send such samples through the general per-sample code on the original int32
 *      values (phase 2 re-reads them; they are rare and hit L2).  A genuine (255,255,255) takes that path too.
 *
 *  Phase 2 arithmetic is the literal one of mcall_kernels.cu (mcall.c:787-878), so GT / GQ / PL / AC / AN are
 *  bit-exact; phase 1 uses the same exponent-tracked products (QUAL within 1e-6 relative).
 */

#include "mcall_device.cuh"

namespace mcb {

#ifndef BW_DYNAMIC
#define BW_DYNAMIC   1                  /* sites claimed from a global counter instead of a static stride */
#endif
#ifndef BW_ROLL1
#define BW_ROLL1     0                  /* 1: phase-1 sample loop rolled (smaller code) */
#endif
#ifndef BW_MAXWARP
#define BW_MAXWARP   14                 /* warps per CTA the kernel is compiled for (2 CTAs per SM => 72 registers, no spills) */
#endif
#ifndef BW_MINCTA
#define BW_MINCTA    2
#endif
#define BW_ESC_CAP   64                 /* escaped samples per site handled lane-parallel after the main loops */
#ifndef BW_PF_NEXT
#define BW_PF_NEXT   0                  /* 128-sample blocks of the warp's next site prefetched into L2 during phase 2 */
#endif
#ifndef BW_PF_DIST
#define BW_PF_DIST   4                  /* L2 prefetch distance of phase 1, in 128-sample iterations */
#endif
#ifndef BW_PF_L1
#define BW_PF_L1     0                  /* 1: the next iteration's 12 lines are also prefetched into L1 (measured: see DESIGN.md 4a) */
#endif
#define BW_REC_BYTES 384                /* per-warp site record in shared memory */

struct BWRec                            /* written by lane 0 after phase 1, read by the whole warp */
{
    int4   slot_out[4];                 /* diploid call of slot k: {gt0, gt1, AC[0] increment, AC[1] increment}; [3] = no call (./., no AC) */
    int4   hap_out[2];                  /* haploid call of selected allele x: {gt0, vector_end, AC[0] increment, AC[1] increment} */
    double q[2];                        /* (double)qsum of the selected alleles, mcall.c:797, 820 */
    double max_qual, lk_sum, ref_lk, gap;
    float  scr_w[4];                    /* float32 screen of phase 2: weights of the slots 0/0, 0/1, 1/1; [3] != 0: the site stays on the literal path */
    float  qf[2];
    uint32_t flags, als_new;
    int    nsel, jgt0, inc_dip, inc_hap, nals_new, ret_early, pl_dropped, ref_gt;
    int    als_map[2];
    long long out_off;
    int    nesc;                        /* samples that need the general path (escape list below; > BW_ESC_CAP: overflowed) */
    unsigned short esc[BW_ESC_CAP];     /* their sample indices */
};
static_assert(sizeof(BWRec) <= BW_REC_BYTES, "BWRec grew past its slot");
static_assert(offsetof(BWRec, scr_w) % 16 == 0, "scr_w is read with one 128-bit load");

/*  the literal FP64 call of one diploid sample of a pair site from its packed bytes: the samples the float32 screen does not accept  */
static __device__ __noinline__ int bw_fast2_exact(uint32_t a, uint32_t b, uint32_t c, double q0, double q1, uint32_t pl2p_s, uint32_t thr_s)      /* slot | GQ << 8 */
{
    const double p0 = lds64c(pl2p_s + 8u*a), p1 = lds64c(pl2p_s + 8u*b), p2 = lds64c(pl2p_s + 8u*c);
    int k, g;
    fast2_call(p0, p1, p2, __dadd_rn(__dadd_rn(p0, p1), p2), q0, q1, __dmul_rn(2.0, q1), thr_s, k, g);
    return k | g<<8;
}

/*  set_pdg's missing-value fill (mcall.c:495-527) on the 3 PLs of a biallelic sample; returns 0 for "no data"  */
__device__ __noinline__ int fix_missing3(int *pl, int unseen)
{
    int j;
    for (j=0; j<3; j++)
    {
        if ( pl[j]==I32_VEC_END ) return 0;         /* not diploid-shaped: all missing, mcall.c:465-470 */
        if ( pl[j]==I32_MISSING ) break;
    }
    if ( j==0 || j==3 ) return 0;                   /* first value missing (mcall.c:476-481) / no sentinel at all */
    j = 0;
    for (int ia=0; ia<2; ia++)
        for (int ib=0; ib<=ia; ib++)
        {
            if ( pl[j]==I32_MISSING )
            {
                int k = gt_idx(ia,unseen);
                if ( pl[k]==I32_MISSING ) k = gt_idx(ib,unseen);
                if ( pl[k]==I32_MISSING ) k = gt_idx(unseen,unseen);
                pl[j] = pl[k]==I32_MISSING ? 255 : pl[k];
            }
            else if ( pl[j] < 0 ) return 0;
            j++;
        }
    return 1;
}

__device__ __noinline__ double bw_big_pl_to_p(const DevTables *tab, int v, uint32_t *flags)
{
    if ( v > 2500 ) *flags |= MCB_SITE_PL_RANGE;
    return (unsigned)v < (unsigned)MCB_PL2P_BIG ? tab->pl2p_big[v] : 0.0;
}

/*  general per-sample load: fills pl[] (missing values filled), p[], sum; returns "sample carries data"  */
__device__ __forceinline__ bool bw_slow_sample(int (&pl)[3], double (&p)[3], double &sum, int unseen, uint32_t pl2p_s,
                                               const DevTables *tab, uint32_t &flags)
{
    int orv = pl[0] | pl[1] | pl[2];
    bool data = orv != 0;
    if ( orv < 0 )
    {
        data = fix_missing3(pl, unseen);
        if ( data ) { orv = pl[0] | pl[1] | pl[2]; data = orv > 0; }
    }
    #pragma unroll
    for (int j=0; j<3; j++)
        p[j] = !data ? 1.0 : ((unsigned)pl[j] < 256u ? lds64(pl2p_s + 8u*(uint32_t)pl[j]) : bw_big_pl_to_p(tab, pl[j], &flags));
    sum = __dadd_rn(__dadd_rn(p[0], p[1]), p[2]);
    return data;
}

/*  libdevice log/exp are ~200 instructions each when inlined; every warp walks the per-site code on its own schedule,
 *  so one shared copy keeps the instruction cache warm  */
__device__ __noinline__ double bw_log(double x) { return log(x); }
__device__ __noinline__ double bw_exp(double x) { return exp(x); }
__device__ __forceinline__ double bw_logsumexp2(double a, double b)       /* mcall.c:573-579 */
{
    const double hi = a>b ? a : b, lo = a>b ? b : a;
    return bw_log(1 + bw_exp(lo - hi)) + hi;
}

struct BWSlow { int pl[3]; double p[3]; double sum; };
__device__ __noinline__ bool bw_slow_sample_ni(BWSlow *w, int unseen, uint32_t pl2p_s, const DevTables *tab, uint32_t *flags)
{
    uint32_t f = 0;
    const bool data = bw_slow_sample(w->pl, w->p, w->sum, unseen, pl2p_s, tab, f);
    if ( f ) *flags |= f;
    return data;
}

/*  mcall_call_genotypes for one HAPLOID sample (mcall.c:793-808, 843-878): lk_x = pdg[s_x/s_x] * q_x over the selected
 *  alleles, GQ over the alleles below grp->nals (inc_hap).  pA = pl2p[PL of s0/s0], pB = of s1/s1.  */
template<bool FAST>
__device__ __forceinline__ int4 bw_call_haploid(double pA, double pB, double sum, const BWConsts &c, uint32_t hap_s, int inc_hap, int &gq)
{
    const double r = FAST ? rcp_shared(sum) : 0.0;
    auto dv = [&](double x) -> double { return FAST ? div_shared(x, sum, r) : __ddiv_rn(x, sum); };
    double best = 0; int bx = 0; bool any_best = false;
    double gv0 = __dmul_rn(dv(pA), c.q0), gv2 = 0;
    if ( best < gv0 ) { best = gv0; bx = 0; any_best = true; }
    if ( c.nsel>1 )
    {
        gv2 = __dmul_rn(dv(pB), c.q1);
        if ( best < gv2 ) { best = gv2; bx = 1; any_best = true; }
    }
    const int4 outc = any_best ? lds128(hap_s + 16u*(uint32_t)bx) : make_int4(MCB_GT_UNPHASED(0), I32_VEC_END, 1, 0);
    gq = 0;
    if ( c.want_gq )
    {
        double gmax = 0, gsum = 0;
        gv0 = (double)__double2float_rn(gv0); gv2 = (double)__double2float_rn(gv2);
        if ( inc_hap & 1 ) { if ( gmax < gv0 ) gmax = gv0; gsum = __dadd_rn(gsum, gv0); }
        if ( inc_hap & 2 ) { if ( gmax < gv2 ) gmax = gv2; gsum = __dadd_rn(gsum, gv2); }
        const double xx = __dadd_rn(1.0, -__ddiv_rn(gmax, gsum));
        if ( !(xx==xx) ) gq = 127;
        else
        {
            int k = __float2int_rz(-3.0102999f*lg2_approx((float)xx));
            k = max(0, min(127, k));
            if ( xx <= lds64c(c.thr_s + 8u*(uint32_t)(k+1)) ) { k++; while ( xx <= lds64c(c.thr_s + 8u*(uint32_t)(k+1)) ) k++; }
            else while ( xx > lds64c(c.thr_s + 8u*(uint32_t)k) ) k--;
            gq = k;
        }
    }
    return outc;
}


#ifndef BW_SCREEN
#define BW_SCREEN    1                  /* 1: float32 screen in front of the literal FP64 call (0: every sample takes the literal path) */
#endif
#ifndef BW_FAST2
#define BW_FAST2     1                  /* 1: straight-line phase 2 for the common variant site, two adjacent samples per lane */
#endif

/*  the sample's call under its ploidy: GT pair + AC increments in the int4, GQ by reference.  `has` = sample carries data.  */
template<bool FAST>
__device__ __forceinline__ int4 bw_call_any(int pld, bool has, bool ref_gt, double p0, double p1, double p2, double sum,
                                            const BWConsts &c, uint32_t hap_s, int inc_hap, int &gq)
{
    gq = 0;
    const int second_missing = pld==2 ? MCB_GT_MISSING : I32_VEC_END;
    if ( !pld || !has ) return make_int4(MCB_GT_MISSING, second_missing, 0, 0);
    if ( ref_gt ) return make_int4(MCB_GT_UNPHASED(0), pld==2 ? MCB_GT_UNPHASED(0) : I32_VEC_END, pld, 0);     /* mcall.c:713-743 */
    if ( pld==2 ) return bw_call_sample<FAST>(p0, p1, p2, sum, c, gq);
    return bw_call_haploid<FAST>(c.jgt0 ? p2 : p0, p2, sum, c, hap_s, inc_hap, gq);
}

__device__ __forceinline__ int4 ldg128(const int4 *p) { return __ldg(p); }
__device__ __forceinline__ void stg128(void *p, int x, int y, int z, int w)
{
    asm volatile("st.global.v4.s32 [%0], {%1,%2,%3,%4};" :: "l"(p), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void stg64(void *p, int x, int y)
{
    asm volatile("st.global.v2.s32 [%0], {%1,%2};" :: "l"(p), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void stg32(void *p, int x)
{
    asm volatile("st.global.s32 [%0], %1;" :: "l"(p), "r"(x) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ldsu32(uint32_t a) { uint32_t v; asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" :: "l"(p)); }
__device__ __forceinline__ void prefetch_l1(const void *p) { asm volatile("prefetch.global.L1 [%0];" :: "l"(p)); }
__device__ __forceinline__ uint32_t ldsu8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t byte_of(uint32_t w, int k) { return (w >> (8*k)) & 0xffu; }

/*  trimmed PL row of one sample (mcall.c:1158-1194) under its ploidy; pl3: both alleles kept  */
__device__ __forceinline__ void bw_store_pl(int32_t *out_pl, bool pl3, int s, int pld, int a, int b, int c)
{
    int v0 = a, v1 = b, v2 = c;
    if ( pld==1 ) { v1 = c; v2 = I32_VEC_END; }                    /* haploid: the homozygous genotypes, then vector_end */
    else if ( pld==0 ) { v0 = I32_MISSING; v1 = v2 = I32_VEC_END; }
    if ( pl3 ) { int32_t *d = out_pl + 3*(size_t)s; stg32(d, v0); stg32(d+1, v1); stg32(d+2, v2); }
    else stg32(out_pl + s, v0);
}

template<bool PLOIDY>
__global__ void __launch_bounds__(BW_MAXWARP*32, BW_MINCTA) mcall_biallelic_warp_kernel(const KArgs a, int warp_bytes)
{
    constexpr double LN2 = 0.693147180559945309417232121458, LN10_10 = 0.2302585092994045684017991454684;
    BWTables &tb = *reinterpret_cast<BWTables*>(mcb_smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = blockDim.x >> 5;
    const uint32_t sbase = smem_base();
    const uint32_t pl2p_s = sbase + (uint32_t)offsetof(BWTables, pl2p), thr_s = sbase + (uint32_t)offsetof(BWTables, gq_thr);
    const uint32_t wbase_s = sbase + (uint32_t)align128(sizeof(BWTables)) + (uint32_t)warp*(uint32_t)warp_bytes;
    const uint32_t buf_s = wbase_s + BW_REC_BYTES;
    BWRec &rec = *reinterpret_cast<BWRec*>(mcb_smem + align128(sizeof(BWTables)) + (size_t)warp*warp_bytes);

    for (int i=tid; i<256; i+=blockDim.x) tb.pl2p[i] = a.tab->pl2p[i];
    for (int i=tid; i<130; i+=blockDim.x) tb.gq_thr[i] = i<128 ? a.tab->gq_thr[i] : -1.0;
    screen_tabs_fill(&tb.scr, a.tab, tid, blockDim.x);
    const uint32_t plf_s = sbase + (uint32_t)offsetof(BWTables, scr) + (uint32_t)offsetof(ScreenTabs, plf);
    const uint32_t gqw_s = sbase + (uint32_t)offsetof(BWTables, scr) + (uint32_t)offsetof(ScreenTabs, gqw);
    __syncthreads();

    const int S = a.nsmpl;
    const int ngrp4 = (S + 3) >> 2, niter = (ngrp4 + 31) >> 5;
    const int nsites = *a.site_count;
    const bool want_gq = a.gq && (a.output_tags & (MCB_CALL_FMT_GQ|MCB_CALL_FMT_GP));

#if BW_DYNAMIC
    /* sites are claimed from a global counter: REF-only sites cost a fraction of a variant site, so a static
       round-robin leaves most warps idle while the unlucky ones finish their last site */
    for (;;)
    {
        int isite = 0;
        if ( lane==0 ) isite = atomicAdd(a.work_counter, 1);
        isite = __shfl_sync(0xffffffffu, isite, 0);
        if ( isite >= nsites ) break;
#else
    for (int isite = blockIdx.x*nwarp + warp; isite < nsites; isite += gridDim.x*nwarp)
    {
#endif
        const int site = a.site_list[isite];
        const int64_t site_off = a.pl_off[site];
        const int32_t *site_pl = reinterpret_cast<const int32_t*>(a.pl) + site_off;
        const int4 *site_pl4 = reinterpret_cast<const int4*>(site_pl);
        const int unseen = a.unseen ? a.unseen[site] : 0;
        const char *site_end = reinterpret_cast<const char*>(site_pl) + (size_t)S*12;
        /* the first blocks of this warp's NEXT site are pulled into L2 while phase 2 of this one runs */
        const char *next_pl = nullptr;
        {
            const int nx = BW_DYNAMIC ? nsites : isite + gridDim.x*nwarp;
            if ( nx < nsites ) next_pl = reinterpret_cast<const char*>(reinterpret_cast<const int32_t*>(a.pl) + a.pl_off[a.site_list[nx]]);
        }
        const uint8_t *ploidy = nullptr;
        if ( PLOIDY )
        {
            int pid = a.ploidy_id ? a.ploidy_id[site] : 0;
            if ( pid >= a.nploidy ) pid = 0;
            ploidy = a.ploidy_tab + (size_t)pid*S;
        }
        if ( lane==0 ) rec.nesc = 0;
        __syncwarp();

        /* ---- site set-up, every lane redundantly: qsum (mcall.c:1454-1464), -F prior (1507-1527), normalisation (1530-1535) */
        float qf0, qf1; uint32_t sflags;
        {
            int nqs = a.nqs ? a.nqs[site] : 2;
            float q[2];
            #pragma unroll
            for (int j=0; j<2; j++) q[j] = (a.qs && j<nqs) ? a.qs[(size_t)site*a.max_nals + j] : 0.f;
            sflags = (a.qs && nqs>0) ? 0 : MCB_SITE_NO_QS;
            if ( a.use_prior && a.prior_an && a.prior_ac )
            {
                int an = a.prior_an[site];
                if ( an!=I32_MISSING && an>0 )
                {
                    const int32_t *pac = a.prior_ac + (size_t)site*a.max_nals;
                    int ac0 = an;
                    if ( pac[0]!=I32_VEC_END && pac[0]!=I32_MISSING )
                    {
                        ac0 -= pac[0];
                        q[1] = (float)( __ddiv_rn(__dadd_rn((double)q[1], __dmul_rn(0.5,(double)pac[0])),
                                                  __dadd_rn((double)(uint32_t)S, __dmul_rn(0.5,(double)an))) );
                    }
                    if ( ac0<0 ) sflags |= MCB_SITE_BAD_PRIOR;
                    q[0] = (float)( __ddiv_rn(__dadd_rn((double)q[0], __dmul_rn(0.5,(double)ac0)),
                                              __dadd_rn((double)(uint32_t)S, __dmul_rn(0.5,(double)an))) );
                }
            }
            float qsum = __fadd_rn(__fadd_rn(0.f, q[0]), q[1]);
            if ( qsum != 0 ) { q[0] = __fdiv_rn(q[0], qsum); q[1] = __fdiv_rn(q[1], qsum); }
            qf0 = q[0]; qf1 = q[1];
        }
        /* the pair {ALT,REF}: float32 expression then widened (mcall.c:629-630) */
        const bool live = qf1!=0 && qf0!=0;
        double cf0 = 0, cf1 = 0, cf2 = 0;      /* fa2 (ALT hom), fb2 (REF hom), 2 fa fb (het) */
        double fa = 0, fb = 0;                 /* haploid samples: fa (ALT), fb (REF), mcall.c:642-643 */
        if ( live )
        {
            const float den = __fadd_rn(qf1, qf0);
            fa = (double)__fdiv_rn(qf1, den); fb = (double)__fdiv_rn(qf0, den);
            cf0 = __dmul_rn(fa,fa); cf1 = __dmul_rn(fb,fb); cf2 = __dmul_rn(__dmul_rn(2.0,fa),fb);
        }

        /* =========================== phase 1: site reduction ==================================== */
        double accP = 1.0, accN = 1.0; int eP = 0, eN = 0;          /* pair product, normaliser product */
        double accC = 1.0; int eC = 0, cnt_called = 0;              /* PLOIDY: normaliser product / count of the samples with ploidy > 0 */
        int nmul = 0, nslow = 0;                                    /* multiplications folded into each product (warp-uniform) / of this lane's overflow samples */
        long long ps0 = 0, ps1 = 0;                                 /* single-allele sets: integer PL sums (mcall.c:607-611) */
        int ps0f = 0, ps1f = 0;                                     /* ... of the iterations with every PL <= 255 */
        int cnt = 0;
        uint32_t tflags = 0;

        auto load_group = [&](int g, int4 &v0, int4 &v1, int4 &v2)
        {
            if ( 4*g + 3 < S ) { v0 = ldg128(site_pl4 + 3*g); v1 = ldg128(site_pl4 + 3*g + 1); v2 = ldg128(site_pl4 + 3*g + 2); }
            else
            {
                int x[12];
                #pragma unroll
                for (int k=0; k<12; k++) x[k] = (4*g + k/3 < S) ? __ldg(site_pl + 12*g + k) : 0;   /* past the end: "no data" */
                v0 = make_int4(x[0],x[1],x[2],x[3]); v1 = make_int4(x[4],x[5],x[6],x[7]); v2 = make_int4(x[8],x[9],x[10],x[11]);
            }
        };
        /*  The 4 samples of an iteration are multiplied together as plain doubles (each factor is in [1e-26, 3]) and enter the
         *  exponent-tracked products once per iteration.  (Measured dead end: packing the 12 raw int32 to bytes first and
         *  issuing the loads of the NEXT iteration before the arithmetic of this one -- the byte extraction and the longer
         *  register lives cost more than the hidden L2 latency gains: class 0.95 -> 1.07 ms.)  */
        const char *pf = reinterpret_cast<const char*>(site_pl) + (size_t)BW_PF_DIST*1536 + 128*lane;
        #pragma unroll 1
        for (int it=0; it<niter; it++)
        {
            const int g = it*32 + lane;
            if ( lane < 12 && pf < site_end ) prefetch_l2(pf);      /* 12 lines of 128 bytes = the 128 samples of iteration it+BW_PF_DIST */
#if BW_PF_L1
            if ( lane < 12 && pf - (BW_PF_DIST-1)*1536 < site_end ) prefetch_l1(pf - (BW_PF_DIST-1)*1536);     /* iteration it+1 into L1 */
#endif
            pf += 1536;
            int4 v0, v1, v2;
            load_group(g, v0, v1, v2);
            const int x[12] = { v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w, v2.x, v2.y, v2.z, v2.w };
            uint32_t pk[3] = {0,0,0};
            double lN = 1.0, lP = 1.0, lC = 1.0;
            #pragma unroll
            for (int j=0; j<4; j++)
            {
                const int pa = x[3*j], pb = x[3*j+1], pc = x[3*j+2];
                const int orv = pa | pb | pc;
                double sum = 1.0, val = 1.0; bool data = false;
                int pld = 2;
                if ( PLOIDY ) pld = (4*g + j < S) ? (int)__ldg(ploidy + 4*g + j) : 2;
                uint32_t tri = 0xffffffu;                               /* escape: the general path goes back to the int32 values */
                if ( (unsigned)orv <= 255u && (pa & pb & pc) != 255 )
                {
                    data = orv != 0;                                    /* PL=0,0,0: no data (mcall.c:529-537) */
                    const double p0 = lds64c(pl2p_s + 8u*(uint32_t)pa), p1 = lds64c(pl2p_s + 8u*(uint32_t)pb), p2 = lds64c(pl2p_s + 8u*(uint32_t)pc);
                    sum = __dadd_rn(__dadd_rn(p0, p1), p2);
                    val = (!PLOIDY || pld==2) ? fma(cf2, p1, fma(cf1, p0, cf0*p2)) : fma(fb, p0, fa*p2);
                    ps0f += pa; ps1f += pc;
                    tri = (uint32_t)pa | (uint32_t)pb<<8 | (uint32_t)pc<<16;
                }
                else
                {
                    const int pos = atomicAdd(&rec.nesc, 1);
                    if ( pos < BW_ESC_CAP ) rec.esc[pos] = (unsigned short)(4*g + j);      /* deferred: one lane per escaped sample */
                    else                                                                    /* list full: right here */
                    {
                        BWSlow w; w.pl[0] = pa; w.pl[1] = pb; w.pl[2] = pc;
                        const bool sdata = bw_slow_sample_ni(&w, unseen, pl2p_s, a.tab, &tflags);
                        if ( sdata ) { ps0 += w.pl[0]; ps1 += w.pl[2]; }
                        const double sval = (!PLOIDY || pld==2) ? fma(cf2, w.p[1], fma(cf1, w.p[0], cf0*w.p[2])) : fma(fb, w.p[0], fa*w.p[2]);
                        /* values of the big-PL table can be tiny: straight into the exponent-tracked products */
                        cnt += sdata;
                        const bool scalled = sdata && (!PLOIDY || pld!=0);
                        acc_mul(accN, eN, sdata ? w.sum : 1.0);
                        if ( PLOIDY ) { cnt_called += scalled; acc_mul(accC, eC, scalled ? w.sum : 1.0); }
                        acc_mul(accP, eP, (scalled && live) ? sval : 1.0);
                        nslow++;
                    }
                }
                cnt += data;                                            /* single-allele sets and N_all: every sample, also ploidy 0 (mcall.c:607-611) */
                const bool called = data && (!PLOIDY || pld!=0);        /* ploidy 0: val stays 0 (mcall.c:639-644) */
                const double fN = data ? sum : 1.0, fP = (called && live) ? val : 1.0, fC = called ? sum : 1.0;
                lN = j ? __dmul_rn(lN, fN) : fN; lP = j ? __dmul_rn(lP, fP) : fP;
                if ( PLOIDY ) { cnt_called += called; lC = j ? __dmul_rn(lC, fC) : fC; }
                /* byte 3j+k of the 12-byte group */
                if ( j==0 ) pk[0] |= tri;
                if ( j==1 ) { pk[0] |= tri<<24; pk[1] |= tri>>8; }
                if ( j==2 ) { pk[1] |= tri<<16; pk[2] |= tri>>16; }
                if ( j==3 ) pk[2] |= tri<<8;
            }
            if ( g < ngrp4 ) { sts32(buf_s + 12u*(uint32_t)g, pk[0]); sts32(buf_s + 12u*(uint32_t)g + 4u, pk[1]); sts32(buf_s + 12u*(uint32_t)g + 8u, pk[2]); }
            acc_mul(accN, eN, lN); acc_mul(accP, eP, lP); if ( PLOIDY ) acc_mul(accC, eC, lC);
            nmul += 1;
            if ( (nmul & 255)==0 ) { acc_renorm(accP, eP); acc_renorm(accN, eN); if ( PLOIDY ) acc_renorm(accC, eC); }
        }
        /*  acc_mul calls made outside the warp-uniform count (escape-list overflow, a handful of samples at most): level
            every lane to the warp's maximum with multiplications by 1.0 so that the exponent bias stays 1023 per call  */
        {
            int mx = nslow;
            #pragma unroll
            for (int off=16; off; off>>=1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, off));
            for (int k=nslow; k<mx; k++) { acc_mul(accN, eN, 1.0); acc_mul(accP, eP, 1.0); if ( PLOIDY ) acc_mul(accC, eC, 1.0); }
            nmul += mx;
        }
        /* ---- the escaped samples, one per lane */
        __syncwarp();
        const int nesc = min(rec.nesc, BW_ESC_CAP);
        const bool esc_overflow = rec.nesc > BW_ESC_CAP;
        #pragma unroll 1
        for (int base=0; base<nesc; base+=32)
        {
            double sum = 1.0, val = 1.0; bool data = false; int pld = 2;
            if ( base + lane < nesc )
            {
                const int s = rec.esc[base + lane];
                if ( PLOIDY ) pld = __ldg(ploidy + s);
                BWSlow w; w.pl[0] = __ldg(site_pl + 3*s); w.pl[1] = __ldg(site_pl + 3*s + 1); w.pl[2] = __ldg(site_pl + 3*s + 2);
                data = bw_slow_sample_ni(&w, unseen, pl2p_s, a.tab, &tflags);
                if ( data ) { ps0 += w.pl[0]; ps1 += w.pl[2]; }
                sum = w.sum;
                val = (!PLOIDY || pld==2) ? fma(cf2, w.p[1], fma(cf1, w.p[0], cf0*w.p[2])) : fma(fb, w.p[0], fa*w.p[2]);
            }
            cnt += data;
            acc_mul(accN, eN, data ? sum : 1.0);
            const bool called = data && (!PLOIDY || pld!=0);
            if ( PLOIDY ) { cnt_called += called; acc_mul(accC, eC, called ? sum : 1.0); }
            acc_mul(accP, eP, (called && live) ? val : 1.0);
            nmul += 1;
        }

        /* ---- warp reduction (mantissa multiply, exponent add) */
        ps0 += ps0f; ps1 += ps1f;
        acc_renorm(accP, eP); acc_renorm(accN, eN); if ( PLOIDY ) acc_renorm(accC, eC);
        #pragma unroll
        for (int off=16; off; off>>=1)
        {
            accP = __dmul_rn(accP, __shfl_xor_sync(0xffffffffu, accP, off)); eP += __shfl_xor_sync(0xffffffffu, eP, off);
            accN = __dmul_rn(accN, __shfl_xor_sync(0xffffffffu, accN, off)); eN += __shfl_xor_sync(0xffffffffu, eN, off);
            ps0 += __shfl_xor_sync(0xffffffffu, ps0, off); ps1 += __shfl_xor_sync(0xffffffffu, ps1, off);
            cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
            tflags |= __shfl_xor_sync(0xffffffffu, tflags, off);
            if ( PLOIDY )
            {
                accC = __dmul_rn(accC, __shfl_xor_sync(0xffffffffu, accC, off)); eC += __shfl_xor_sync(0xffffffffu, eC, off);
                cnt_called += __shfl_xor_sync(0xffffffffu, cnt_called, off);
            }
        }
        acc_renorm(accP, eP); acc_renorm(accN, eN); if ( PLOIDY ) acc_renorm(accC, eC);
        /* every lane multiplied nmul values in (1.0 with biased exponent 1023 for absent samples); acc_renorm removed its own bias */
        const int n_all = cnt, nm = 32*nmul;        /* nmul is warp-uniform */

        /* ---- allele sets in the reference's enumeration order: lane 0 {REF}, lane 1 {ALT}, lane 2 {ALT,REF} ---- */
        {
            const double lnN = n_all ? bw_log(accN) + (double)(eN - 1023*nm)*LN2 : 0.0;
            const int n_called = PLOIDY ? cnt_called : n_all;
            const double lnN_called = PLOIDY ? (n_called ? bw_log(accC) + (double)(eC - 1023*nm)*LN2 : 0.0) : lnN;
            double lk = 0; bool cand = false, in_sum = false; uint32_t mask = 0;
            if ( lane < 2 )
            {
                const bool set = n_all > 0;
                lk = set ? -LN10_10*(double)(lane ? ps1 : ps0) - lnN : 0.0;
                if ( lane>0 ) lk += a.theta;
                cand = set; in_sum = set && lane>0; mask = 1u<<lane;
            }
            else if ( lane==2 )
            {
                const bool set = live && n_called > 0;
                lk = set ? (bw_log(accP) + (double)(eP - 1023*nm)*LN2) - lnN_called : 0.0;
                lk += a.theta;
                cand = set; in_sum = set; mask = 3u;
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
            /* lk_sum = log sum exp over every evaluated set except {REF} (mcall.c:584, 614) */
            double mx = in_sum ? lk : -CUDART_INF;
            #pragma unroll
            for (int off=16; off; off>>=1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, off));
            double term = in_sum ? bw_exp(lk - mx) : 0.0;
            #pragma unroll
            for (int off=16; off; off>>=1) term += __shfl_xor_sync(0xffffffffu, term, off);
            const double grp_lk_sum = mx > -CUDART_INF ? mx + bw_log(term) : -CUDART_INF;
            const double grp_ref_lk = __shfl_sync(0xffffffffu, lk, 0);
            const uint32_t grp_als = __shfl_sync(0xffffffffu, mask, best_lane & 31);

            if ( lane==0 )
            {
                const bool any = best_lane < 64;
                const uint32_t gals = any ? grp_als : 0;
                uint32_t flags = sflags | tflags;
                double max_qual = -CUDART_INF, lk_sum = -CUDART_INF, ref_lk = -CUDART_INF;
                if ( any )          /* mcall.c:1553-1560 */
                {
                    max_qual = -4.343*(grp_ref_lk - bw_logsumexp2(grp_lk_sum, grp_ref_lk));
                    lk_sum = grp_lk_sum; ref_lk = grp_ref_lk;
                }
                const double gap = any ? best - second : CUDART_INF;
                if ( any && gap < a.tie_eps ) flags |= MCB_SITE_NEAR_TIE;
                uint32_t als_new = gals | 1u;               /* mcall.c:1552, 1564 */
                const int is_variant = als_new!=1;
                const int ret_early = ((a.flag & MCB_CALL_VARONLY) && !is_variant) || (flags & MCB_SITE_NO_QS);
                int nals_new = 1;                                                   /* mcall.c:1569-1575: the unseen allele is not counted */
                if ( unseen!=1 )
                {
                    if ( a.flag & MCB_CALL_KEEPALT ) als_new |= 2u;
                    if ( als_new & 2u ) nals_new++;
                }
                int amap[2];
                amap[0] = 0; amap[1] = (als_new & 2u) ? 1 : -1;                    /* mcall.c:547-570 */
                rec.als_map[0] = amap[0]; rec.als_map[1] = amap[1];
                if ( unseen && (als_new & (1u<<unseen)) ) flags |= MCB_SITE_UNSEEN_SEL;
                const int pl_dropped = als_new==1;
                const int ref_gt = (als_new==1) || !is_variant;
                long long off = site_off;
                if ( a.pl_off_out )
                {
                    off = compact_out_off<false>(a, site, S, 2, nals_new, !pl_dropped && !ret_early, flags);
                    a.pl_off_out[site] = off;
                }
                if ( pl_dropped ) flags |= MCB_SITE_PL_DROPPED;
                if ( ref_gt ) flags |= MCB_SITE_REF_GT;
                rec.out_off = off; rec.pl_dropped = pl_dropped; rec.ref_gt = ref_gt;
                rec.als_new = als_new; rec.nals_new = nals_new; rec.ret_early = ret_early; rec.flags = flags;
                rec.max_qual = max_qual; rec.lk_sum = lk_sum; rec.ref_lk = ref_lk; rec.gap = gap;
                rec.qf[0] = qf0; rec.qf[1] = qf1;
                /* phase-2 constants: selected alleles in ascending order and the <=3 genotypes they span */
                const int ngt_new = nals_new*(nals_new+1)/2;
                int sel[2] = {0,0}, ns = 0;
                if ( gals & 1u ) sel[ns++] = 0;
                if ( gals & 2u ) sel[ns++] = 1;
                rec.nsel = ns; rec.jgt0 = ns>0 ? 4*gt_idx(sel[0], sel[0]) : 0;
                int inc_dip = 0, inc_hap = 0;
                const int gn = ns;                                          /* grp->nals: alleles of the selected set */
                for (int xx=0; xx<2; xx++)
                {
                    rec.q[xx] = xx<ns ? (double)(sel[xx] ? qf1 : qf0) : 0.0;
                    const int nx = xx<ns ? amap[sel[xx]] : 0;
                    if ( xx<ns && nx < gn ) inc_hap |= 1<<xx;               /* mcall.c:853 */
                    rec.hap_out[xx] = make_int4(MCB_GT_UNPHASED(nx), I32_VEC_END, nx==0, nx==1);
                    for (int y=0; y<=xx; y++)
                    {
                        const int k = xx*(xx+1)/2 + y;
                        const int ny = y<ns ? amap[sel[y]] : 0;
                        const int ig = gt_idx(nx, ny);
                        if ( xx<ns && ig < ngt_new ) inc_dip |= 1<<k;
                        /* gts[0] = smaller new allele, gts[1] = larger (mcall.c:830-831); AC: one count per allele */
                        rec.slot_out[k] = make_int4(MCB_GT_UNPHASED(ny), MCB_GT_UNPHASED(nx), (ny==0) + (nx==0), (ny==1) + (nx==1));
                    }
                }
                rec.inc_dip = inc_dip; rec.inc_hap = inc_hap;
                {
                    bool scr = ns==2 && BW_SCREEN;
                    rec.scr_w[0] = screen_weight(rec.q[0], rec.q[0], 1.0, scr); rec.scr_w[1] = screen_weight(rec.q[1], rec.q[0], 2.0, scr);
                    rec.scr_w[2] = screen_weight(rec.q[1], rec.q[1], 1.0, scr); rec.scr_w[3] = scr ? 0.f : 1.f;
                }
                rec.slot_out[3] = make_int4(MCB_GT_MISSING, MCB_GT_MISSING, 0, 0);
            }
        }
        __syncwarp();

        /* =========================== phase 2: per-sample genotypes ============================== */
        if ( rec.ret_early )
        {
            if ( lane==0 )
            {
                a.ret[site] = 0;
                if ( a.site_flags ) a.site_flags[site] = rec.flags;
            }
            __syncwarp();
            continue;
        }
        int ac0 = 0, ac1 = 0;
        uint32_t tflags2 = 0;
        {
            const bool ref_gt = rec.ref_gt, pl_dropped = rec.pl_dropped;
            const bool pl3 = rec.nals_new==2;       /* both alleles kept: the PL vector is copied; else (unseen ALT selected) PL[0] only */
            int32_t *out_pl = (a.out_pl && !pl_dropped) ? a.out_pl + rec.out_off : nullptr;
            int32_t *out_gt = a.gt ? a.gt + 2*(size_t)site*S : nullptr;
            int32_t *out_gq = want_gq ? a.gq + (size_t)site*S : nullptr;
            BWConsts c;
            c.q0 = rec.q[0]; c.q1 = rec.q[1]; c.slot_s = wbase_s + (uint32_t)offsetof(BWRec, slot_out); c.thr_s = thr_s;
            c.nsel = rec.nsel; c.jgt0 = rec.jgt0; c.inc_dip = rec.inc_dip; c.want_gq = want_gq;
            const uint32_t hap_s = wbase_s + (uint32_t)offsetof(BWRec, hap_out);
            const int inc_hap = rec.inc_hap;

#if BW_FAST2
            /*  The common variant site -- every sample diploid, {REF,ALT} selected and both kept, GT + GQ + PL all written,
             *  no escape-list overflow, an even sample count (16-byte aligned GT pairs): straight-line code, each lane takes
             *  TWO ADJACENT samples per iteration so that their dependency chains interleave and GT / GQ / PL of the pair
             *  leave as one 128-bit, one 64-bit and three 64-bit stores (a warp still writes contiguous rows).  */
            const bool pair_ok = !ref_gt && c.nsel==2 && c.inc_dip==7 && want_gq && out_pl && pl3 && out_gt && out_gq && !esc_overflow && !(S & 1)
                                 && !((reinterpret_cast<uintptr_t>(out_gt) & 15) | (reinterpret_cast<uintptr_t>(out_gq) & 7) | (reinterpret_cast<uintptr_t>(out_pl) & 7));
            const bool fast2 = !PLOIDY && pair_ok;
            const bool fastp = PLOIDY && pair_ok && inc_hap==3;
            if ( fast2 )
            {
                /* float32 screen (mcall_device.cuh): the arg max and the GQ of a sample far from every decision boundary need no
                   double precision; the few samples it does not accept take the literal sequence */
                float w0, w1, w2, wn;
                asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(w0), "=f"(w1), "=f"(w2), "=f"(wn) : "r"(wbase_s + (uint32_t)offsetof(BWRec, scr_w)));
                const bool noscr = wn != 0.f;
                const int npair = S >> 1;
                #pragma unroll 1
                for (int pr=lane; pr<npair; pr+=32)
                {
                    const uint32_t ad = buf_s + 6u*(uint32_t)pr;
                    const uint32_t pa0 = ldsu8(ad), pb0 = ldsu8(ad + 1u), pc0 = ldsu8(ad + 2u);
                    const uint32_t pa1 = ldsu8(ad + 3u), pb1 = ldsu8(ad + 4u), pc1 = ldsu8(ad + 5u);
                    int32_t *dpl = out_pl + 6*(size_t)pr;       /* escaped samples: placeholders, rewritten after the loop */
                    stg64(dpl, (int)pa0, (int)pb0); stg64(dpl + 2, (int)pc0, (int)pa1); stg64(dpl + 4, (int)pb1, (int)pc1);
                    int k0, k1, q0, q1;
                    const bool ok0 = screen2_call(pa0, pb0, pc0, w0, w1, w2, plf_s, gqw_s, k0, q0);
                    const bool ok1 = screen2_call(pa1, pb1, pc1, w0, w1, w2, plf_s, gqw_s, k1, q1);
                    const bool has0 = (pa0 | pb0 | pc0) != 0, has1 = (pa1 | pb1 | pc1) != 0;     /* PL=0,0,0: no data (mcall.c:529-537) */
                    const bool esc0 = (pa0 & pb0 & pc0) == 255u, esc1 = (pa1 & pb1 & pc1) == 255u;
                    if ( (!ok0 || noscr) && has0 && !esc0 ) { const int e = bw_fast2_exact(pa0, pb0, pc0, c.q0, c.q1, pl2p_s, thr_s); k0 = e & 255; q0 = e >> 8; }
                    if ( (!ok1 || noscr) && has1 && !esc1 ) { const int e = bw_fast2_exact(pa1, pb1, pc1, c.q0, c.q1, pl2p_s, thr_s); k1 = e & 255; q1 = e >> 8; }
                    const int4 o0 = lds128(c.slot_s + 16u*(uint32_t)((has0 && !esc0) ? k0 : 3));
                    const int4 o1 = lds128(c.slot_s + 16u*(uint32_t)((has1 && !esc1) ? k1 : 3));
                    ac0 += o0.z + o1.z; ac1 += o0.w + o1.w;
                    q0 = has0 ? q0 : 0; q1 = has1 ? q1 : 0;
                    if ( !(esc0 | esc1) )
                    {
                        stg128(out_gt + 4*(size_t)pr, o0.x, o0.y, o1.x, o1.y);
                        stg64(out_gq + 2*(size_t)pr, q0, q1);
                    }
                    else            /* on the escape list: called after this loop */
                    {
                        if ( !esc0 ) { stg64(out_gt + 4*(size_t)pr, o0.x, o0.y); stg32(out_gq + 2*(size_t)pr, q0); }
                        if ( !esc1 ) { stg64(out_gt + 4*(size_t)pr + 2, o1.x, o1.y); stg32(out_gq + 2*(size_t)pr + 1, q1); }
                    }
                }
            }
            else if ( fastp )
            {
                /*  The same site under a ploidy vector (chrX): per-sample ploidy 0 / 1 / 2 is folded into the straight-line code with
                 *  selects -- haploid likelihoods are the intermediates of the diploid ones (fast2_call), GT / PL rows take the
                 *  shapes of mcall.c:793-808, 1158-1194 -- so diploid and haploid lanes of a warp do not diverge.  */
                const double q1x2 = __dmul_rn(2.0, c.q1);
                const int npair = S >> 1;
                int nall = 0;
                #pragma unroll 1
                for (int pr=lane; pr<npair; pr+=32)
                {
                    const uint32_t ad = buf_s + 6u*(uint32_t)pr;
                    const uint32_t pa0 = ldsu8(ad), pb0 = ldsu8(ad + 1u), pc0 = ldsu8(ad + 2u);
                    const uint32_t pa1 = ldsu8(ad + 3u), pb1 = ldsu8(ad + 4u), pc1 = ldsu8(ad + 5u);
                    const int pd0 = (int)__ldg(ploidy + 2*pr), pd1 = (int)__ldg(ploidy + 2*pr + 1);
                    int k0, k1, q0, q1;
                    {
                        const double p0 = lds64c(pl2p_s + 8u*pa0), p1 = lds64c(pl2p_s + 8u*pb0), p2 = lds64c(pl2p_s + 8u*pc0);
                        fast2_call(p0, p1, p2, __dadd_rn(__dadd_rn(p0, p1), p2), c.q0, c.q1, q1x2, thr_s, k0, q0, pd0!=2);
                    }
                    {
                        const double p0 = lds64c(pl2p_s + 8u*pa1), p1 = lds64c(pl2p_s + 8u*pb1), p2 = lds64c(pl2p_s + 8u*pc1);
                        fast2_call(p0, p1, p2, __dadd_rn(__dadd_rn(p0, p1), p2), c.q0, c.q1, q1x2, thr_s, k1, q1, pd1!=2);
                    }
                    const bool esc0 = (pa0 & pb0 & pc0) == 255u, esc1 = (pa1 & pb1 & pc1) == 255u;
                    const bool cl0 = (pa0 | pb0 | pc0) != 0 && !esc0 && pd0, cl1 = (pa1 | pb1 | pc1) != 0 && !esc1 && pd1;   /* PL=0,0,0 / ploidy 0: no call */
                    /* trimmed PL rows (mcall.c:1158-1194): diploid a,b,c; haploid the two homozygous values, vector_end; ploidy 0 missing */
                    const int r00 = pd0 ? (int)pa0 : I32_MISSING, r01 = pd0==2 ? (int)pb0 : (pd0 ? (int)pc0 : I32_VEC_END), r02 = pd0==2 ? (int)pc0 : I32_VEC_END;
                    const int r10 = pd1 ? (int)pa1 : I32_MISSING, r11 = pd1==2 ? (int)pb1 : (pd1 ? (int)pc1 : I32_VEC_END), r12 = pd1==2 ? (int)pc1 : I32_VEC_END;
                    int32_t *dpl = out_pl + 6*(size_t)pr;       /* escaped samples: placeholders, rewritten after the loop */
                    stg64(dpl, r00, r01); stg64(dpl + 2, r02, r10); stg64(dpl + 4, r11, r12);
                    /* new alleles 0 and 1 = GT codes 2 and 4; haploid: one allele then vector_end (mcall.c:805-807) */
                    const int x0 = cl0 ? (k0==2 ? 4 : 2) : 0, y0 = pd0==2 ? (cl0 ? (k0 ? 4 : 2) : 0) : I32_VEC_END;
                    const int x1 = cl1 ? (k1==2 ? 4 : 2) : 0, y1 = pd1==2 ? (cl1 ? (k1 ? 4 : 2) : 0) : I32_VEC_END;
                    ac1 += (cl0 ? (pd0==2 ? k0 : (k0>>1)) : 0) + (cl1 ? (pd1==2 ? k1 : (k1>>1)) : 0);
                    nall += (cl0 ? pd0 : 0) + (cl1 ? pd1 : 0);
                    q0 = cl0 ? q0 : 0; q1 = cl1 ? q1 : 0;
                    if ( !(esc0 | esc1) )
                    {
                        stg128(out_gt + 4*(size_t)pr, x0, y0, x1, y1);
                        stg64(out_gq + 2*(size_t)pr, q0, q1);
                    }
                    else            /* on the escape list: called after this loop */
                    {
                        if ( !esc0 ) { stg64(out_gt + 4*(size_t)pr, x0, y0); stg32(out_gq + 2*(size_t)pr, q0); }
                        if ( !esc1 ) { stg64(out_gt + 4*(size_t)pr + 2, x1, y1); stg32(out_gq + 2*(size_t)pr + 1, q1); }
                    }
                }
                ac0 += nall - ac1;          /* ac1 is still this loop's own count here */
            }
            else
#endif
            {
            /* lanes take consecutive samples: GT / GQ / PL rows of a warp are contiguous, every store instruction writes whole sectors */
            const int nit2 = (S + 31) >> 5;
            #pragma unroll 1
            for (int it=0; it<nit2; it++)
            {
                if ( it < BW_PF_NEXT && lane < 12 && next_pl && (it*1536 + 128*lane) < S*12 ) prefetch_l2(next_pl + it*1536 + 128*lane);
                const int s = it*32 + lane;
                if ( s >= S ) continue;
                const uint32_t pa = ldsu8(buf_s + 3u*(uint32_t)s), pb = ldsu8(buf_s + 3u*(uint32_t)s + 1u), pc = ldsu8(buf_s + 3u*(uint32_t)s + 2u);
                const int pld = PLOIDY ? (int)__ldg(ploidy + s) : 2;
                /* mcall.c:1158-1194: both alleles kept, the PL vector is copied.  Escaped samples are rewritten after the loop
                   with their filled int32 values. */
                if ( out_pl ) bw_store_pl(out_pl, pl3, s, pld, (int)pa, (int)pb, (int)pc);
                int4 outc; int q = 0;
                if ( (pa & pb & pc) != 255u )
                {
                    const bool has = (pa | pb | pc) != 0;
                    if ( !PLOIDY )
                    {
                        if ( ref_gt ) outc = make_int4(MCB_GT_UNPHASED(0), MCB_GT_UNPHASED(0), 2, 0);         /* mcall.c:713-743 */
                        else
                        {
                            const double p0 = lds64c(pl2p_s + 8u*pa), p1 = lds64c(pl2p_s + 8u*pb), p2 = lds64c(pl2p_s + 8u*pc);
                            const double sum = __dadd_rn(__dadd_rn(p0, p1), p2);
                            outc = bw_call_sample<true>(p0, p1, p2, sum, c, q);
                        }
                        if ( !has ) { outc = make_int4(MCB_GT_MISSING, MCB_GT_MISSING, 0, 0); q = 0; }
                    }
                    else
                    {
                        const double p0 = lds64c(pl2p_s + 8u*pa), p1 = lds64c(pl2p_s + 8u*pb), p2 = lds64c(pl2p_s + 8u*pc);
                        const double sum = __dadd_rn(__dadd_rn(p0, p1), p2);
                        outc = bw_call_any<true>(pld, has, ref_gt, p0, p1, p2, sum, c, hap_s, inc_hap, q);
                    }
                }
                else if ( !esc_overflow ) continue;     /* on the escape list: called after this loop */
                else                /* list overflowed: general path on the original values, right here */
                {
                    BWSlow w; w.pl[0] = __ldg(site_pl + 3*s); w.pl[1] = __ldg(site_pl + 3*s + 1); w.pl[2] = __ldg(site_pl + 3*s + 2);
                    const bool has = bw_slow_sample_ni(&w, unseen, pl2p_s, a.tab, &tflags2);
                    outc = bw_call_any<false>(pld, has, ref_gt, w.p[0], w.p[1], w.p[2], w.sum, c, hap_s, inc_hap, q);
                    if ( out_pl ) bw_store_pl(out_pl, pl3, s, pld, w.pl[0], w.pl[1], w.pl[2]);
                }
                ac0 += outc.z; ac1 += outc.w;
                if ( out_gt ) stg64(out_gt + 2*(size_t)s, outc.x, outc.y);
                if ( out_gq ) stg32(out_gq + s, q);
            }
            }
            /* ---- the escaped samples, one per lane (their PL rows overwrite the 255s stored above: order the stores) */
            __syncwarp();
            if ( !esc_overflow )
            {
                #pragma unroll 1
                for (int base=0; base<nesc; base+=32)
                {
                    if ( base + lane >= nesc ) continue;
                    const int s = rec.esc[base + lane];
                    const int pld = PLOIDY ? (int)__ldg(ploidy + s) : 2;
                    BWSlow w; w.pl[0] = __ldg(site_pl + 3*s); w.pl[1] = __ldg(site_pl + 3*s + 1); w.pl[2] = __ldg(site_pl + 3*s + 2);
                    const bool has = bw_slow_sample_ni(&w, unseen, pl2p_s, a.tab, &tflags2);
                    int q = 0;
                    const int4 outc = bw_call_any<false>(pld, has, ref_gt, w.p[0], w.p[1], w.p[2], w.sum, c, hap_s, inc_hap, q);
                    ac0 += outc.z; ac1 += outc.w;
                    if ( out_gt ) stg64(out_gt + 2*(size_t)s, outc.x, outc.y);
                    if ( out_gq ) stg32(out_gq + s, q);
                    if ( out_pl ) bw_store_pl(out_pl, pl3, s, pld, w.pl[0], w.pl[1], w.pl[2]);
                }
            }
        }
        #pragma unroll
        for (int off=16; off; off>>=1)
        {
            ac0 += __shfl_xor_sync(0xffffffffu, ac0, off); ac1 += __shfl_xor_sync(0xffffffffu, ac1, off);
            tflags2 |= __shfl_xor_sync(0xffffffffu, tflags2, off);
        }

        /* ---- site record: QUAL (mcall.c:1631-1645), AC/AN (1648-1650) ---------------------------------- */
        if ( lane==0 )
        {
            const int nals_new = rec.nals_new;
            int nAC = 0;
            if ( !rec.ref_gt && nals_new>1 ) nAC = ac1;
            int ret = nals_new;
            if ( !rec.ref_gt && !nAC && (a.flag & MCB_CALL_VARONLY) ) ret = 0;      /* mcall.c:1618 */
            float qual;
            if ( nAC ) qual = (float)rec.max_qual;
            else if ( rec.lk_sum != -CUDART_INF ) qual = (float)(-4.343*(rec.lk_sum - bw_logsumexp2(rec.lk_sum, rec.ref_lk)));
            else if ( ac0 ) qual = a.theta ? (float)(-4.343*a.theta) : 0.f;
            else qual = __uint_as_float(MCB_FLOAT_MISSING_BITS);
            a.ret[site] = ret;
            if ( a.als_new ) a.als_new[site] = rec.als_new;
            if ( a.als_map ) for (int j=0; j<a.max_nals; j++) a.als_map[(size_t)site*a.max_nals + j] = j<2 ? (int8_t)rec.als_map[j] : (int8_t)-1;
            if ( a.qual ) a.qual[site] = qual;
            if ( a.ac ) for (int j=0; j<a.max_nals; j++) a.ac[(size_t)site*a.max_nals + j] = j==0 ? ac0 : ((j==1 && nals_new>1) ? ac1 : 0);
            if ( a.an ) a.an[site] = nAC + ac0;
            if ( a.site_flags ) a.site_flags[site] = rec.flags | tflags2;
            if ( a.diag ) { double *d = a.diag + (size_t)site*4; d[0] = rec.max_qual; d[1] = rec.lk_sum; d[2] = rec.ref_lk; d[3] = rec.gap; }
        }
        __syncwarp();
    }
}

/* ------------------------------------------------------------------------------------------------
 *  launcher
 * ---------------------------------------------------------------------------------------------- */
size_t biallelic_warp_bytes(int nsmpl)
{
    return BW_REC_BYTES + (((size_t)3*(((size_t)nsmpl + 3) & ~(size_t)3) + 15) & ~(size_t)15) ;
}
size_t biallelic_smem_bytes(int nsmpl, int nwarp)
{
    return align128(sizeof(BWTables)) + (size_t)nwarp*biallelic_warp_bytes(nsmpl);
}
int biallelic_max_warps() { return BW_MAXWARP; }
int biallelic_ctas_per_sm() { return BW_MINCTA; }

cudaError_t launch_biallelic_warp_kernel(const KArgs &a, bool ploidy, int grid, int nwarp, cudaStream_t st)
{
    const size_t smem = biallelic_smem_bytes(a.nsmpl, nwarp);
    auto kern = ploidy ? mcall_biallelic_warp_kernel<true> : mcall_biallelic_warp_kernel<false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if ( e != cudaSuccess ) return e;
    kern<<<grid, nwarp*32, smem, st>>>(a, (int)biallelic_warp_bytes(a.nsmpl));
    return cudaGetLastError();
}

}   // namespace mcb
