/*  mcall_kernels.cu -- the fused site kernel (phase 1 site reduction + phase 2 per-sample genotype).
 *  See mcall_kernels.cuh for the design summary and the reference line map.
 */

#include "mcall_device.cuh"

#ifndef MCB_UNROLL1
#define MCB_UNROLL1 1       /* unroll factor of the phase-1 sample loop */
#endif
#ifndef MCB_UNROLL2
#define MCB_UNROLL2 1       /* unroll factor of the phase-2 sample loop */
#endif
#ifndef MCB_FAST2_N2
#define MCB_FAST2_N2 1      /* the same path in the two-allele instances of this kernel (int32 PLs, S > 8,192: the biobank shape) */
#endif
#ifndef MCB_FAST2
#define MCB_FAST2 0         /* 1: straight-line phase 2 for pair sites INSIDE the 3-5 allele instances (measured slower: instruction fetch; mcall_multi.cu is the fast path of those classes) */
#endif

namespace mcb {

constexpr int kUnroll1 = MCB_UNROLL1, kUnroll2 = MCB_UNROLL2;

/*  per-site constants of phase 2: the group's selected alleles s0<s1<s2 span at most 6 genotypes ("slots"),
 *  kept in the output (igt) order  k: 0=(s0,s0) 1=(s1,s0) 2=(s1,s1) 3=(s2,s0) 4=(s2,s1) 5=(s2,s2)        */
struct Phase2Consts
{
    int4   slot_out[6];     /* diploid call of slot k: {gt0, gt1, AC increment lo, hi} (12-bit counters per new allele) */
    int4   hap_out[3];      /* haploid call of allele s_x: {gt0, vector_end, AC increment lo, hi} */
    double q[3];            /* (double)qsum[s_x], mcall.c:797, 820 */
    int    nsel;            /* number of selected alleles, 1..3 */
    int    jgt4[6];         /* byte offset of the slot's genotype in the ORIGINAL PL vector */
    int    igt[6];          /* genotype index in the trimmed vector (GP) */
    int    hap_new[3];      /* new allele index of s_x */
    uint32_t inc_dip;       /* bit k: slot k lies below nmax=ngt_new (mcall.c:852) */
    uint32_t inc_hap;       /* bit x: als_map[s_x] < grp->nals (mcall.c:853) */
};

template<int NALS, int BLOCK> struct Shared
{
    using S = Shape<NALS>;
    static constexpr int NW = BLOCK/32;
    double   pl2p[256];
    double   gq_thr[130];                            /* [128],[129] = -1: never reached */
    uint64_t bars[MAX_STAGE];
    /* per-site coefficients of the allele sets (mcall.c:629-633, 671-677) */
    double   cf_pair[(S::NPAIR ? S::NPAIR : 1)*5];   /* fa2 fb2 fab | fa fb */
    double   cf_tri[(S::NTRI ? S::NTRI : 1)*9];      /* fa2 fb2 fc2 fab fac fbc | fa fb fc */
    uint32_t live;                                   /* bit k: pair k evaluated; bit NPAIR+k: triple k evaluated */
    /* cross-warp reduction scratch */
    double   red_M[NW][S::NACC];
    int      red_E[NW][S::NACC];
    long long red_pls[NW][NALS];
    int      red_cnt[NW][2];
    /* site decision record */
    float    qf[NALS];
    double   max_qual, lk_sum, ref_lk, gap;
    uint32_t grp_als, als_new, flags;
    int      grp_nals, nals_new, is_variant, ret_early, pl_dropped, ref_gt;
    long long out_off;       /* where this site's trimmed PL / GP block goes */
    int      als_map[NALS];
    int      pl_map[S::G];
    int      ac[8];
    int      next_site;
    Phase2Consts p2;
};

/* ------------------------------------------------------------------------------------------------
 *  set_pdg for one sample (mcall.c:460-543), the rare part: missing / vector_end values present.
 *  `row` indexes the sample's PL vector inside the ring; the fill of mcall.c:495-527 is written back
 *  because the filled values are what gets trimmed and output later.  Returns 0 when the sample has
 *  no data (all missing).
 * ---------------------------------------------------------------------------------------------- */
template<typename PT>
__device__ __noinline__ int fix_missing(uint32_t row_s, int nals, int unseen)
{
    using P = PLType<PT>;
    const int G = nals*(nals+1)/2;
    auto PL = [&](int j) -> int { return P::widen(P::ld(row_s + (uint32_t)(P::ES*j))); };
    int j;
    for (j=0; j<G; j++)
    {
        const int v = PL(j);
        if ( v==I32_VEC_END ) return 0;         /* not diploid-shaped: all missing, mcall.c:465-470 */
        if ( v==I32_MISSING ) break;
    }
    if ( j==0 ) return 0;                       /* first value missing: all missing, mcall.c:476-481 */
    if ( j==G ) return 0;                       /* negative garbage that is no sentinel: undefined in the reference */
    j = 0;
    for (int ia=0; ia<nals; ia++)
        for (int ib=0; ib<=ia; ib++)
        {
            const int v = PL(j);
            if ( v==I32_MISSING )
            {
                int k = gt_idx(ia,unseen);
                if ( PL(k)==I32_MISSING ) k = gt_idx(ib,unseen);
                if ( PL(k)==I32_MISSING ) k = gt_idx(unseen,unseen);
                const int w = PL(k)==I32_MISSING ? 255 : PL(k);
                P::st(row_s + (uint32_t)(P::ES*j), w);
            }
            else if ( v < 0 ) return 0;         /* vector_end behind a missing value: undefined in the reference */
            j++;
        }
    return 1;
}

/*  PL >= 256 (mcall.c:472): host-built table in global memory, 0 beyond the double range  */
__device__ __noinline__ double big_pl_to_p(const DevTables *tab, int v, uint32_t *flags)
{
    if ( v > 2500 ) *flags |= MCB_SITE_PL_RANGE;
    return (unsigned)v < (unsigned)MCB_PL2P_BIG ? tab->pl2p_big[v] : 0.0;
}

/*  One sample per lane, called by ALL 32 lanes of a warp: PLs, likelihoods p[j] = pl2p[PL[j]] and their sum in
 *  index order (mcall.c:462-474).  The rare cases -- missing / vector_end values, PL >= 256 -- are detected with
 *  one warp vote so that the common path is straight-line code; `fast` (warp-uniform) tells the caller that every
 *  valid lane has all PLs in 0..255.  Lanes with valid==false must pass the address of some readable row.
 *  Returns true when the lane's sample carries data.                                                          */
template<int NALS, typename PT>
__device__ __forceinline__ bool load_sample_w(uint32_t row_s, uint32_t pl2p_s, bool valid, int unseen, const DevTables *tab,
                                              int (&pl)[Shape<NALS>::G], double (&p)[Shape<NALS>::G], double &sum, bool &fast, uint32_t &flags)
{
    constexpr int G = Shape<NALS>::G;
    int orv = 0;
    #pragma unroll
    for (int j=0; j<G; j++) { pl[j] = PLType<PT>::ld(row_s + (uint32_t)(PLType<PT>::ES*j)); orv |= pl[j]; }
    /* negative (sentinels) or >= 256.  Lanes past the end of the tile re-read the last row: they must vote too, or an
       all-idle warp would index the table with that row's sentinel. */
    const bool special = (unsigned)orv > 255u;
    fast = !__any_sync(0xffffffffu, special);
    bool data = valid && orv!=0;            /* PL=0,..,0: sum==n_gt, no data (mcall.c:529-537) */
    if ( fast )
    {
        #pragma unroll
        for (int j=0; j<G; j++) p[j] = lds64c(pl2p_s + 8u*(uint32_t)pl[j]);
    }
    else
    {
        if ( valid && orv<0 )
        {
            data = fix_missing<PT>(row_s, NALS, unseen);
            if ( data )
            {
                orv = 0;
                #pragma unroll
                for (int j=0; j<G; j++) { pl[j] = PLType<PT>::widen(PLType<PT>::ld(row_s + (uint32_t)(PLType<PT>::ES*j))); orv |= pl[j]; }
                data = orv>0;
            }
        }
        #pragma unroll
        for (int j=0; j<G; j++)
            p[j] = !data ? 1.0 : ((unsigned)pl[j] < 256u ? lds64(pl2p_s + 8u*(uint32_t)pl[j]) : big_pl_to_p(tab, pl[j], &flags));
    }
    sum = p[0];
    #pragma unroll
    for (int j=1; j<G; j++) sum = __dadd_rn(sum, p[j]);
    return data;
}

/* ------------------------------------------------------------------------------------------------
 *  the fused kernel
 * ---------------------------------------------------------------------------------------------- */
template<int NALS, int BLOCK> struct MinBlocks
{
#ifndef MCB_MINB2
#define MCB_MINB2 4         /* CTAs of 256 threads per SM the 1-2 allele kernels are compiled for (register cap 65536/(256*n)) */
#endif
    static constexpr int per256 = NALS<=2 ? MCB_MINB2 : (NALS==3 ? 2 : 1);
    #ifndef MCB_MINB3
#define MCB_MINB3 6
#endif
#ifndef MCB_MINB4
#define MCB_MINB4 4
#endif
#ifndef MCB_MINB5
#define MCB_MINB5 3
#endif
    static constexpr int per128 = NALS<=2 ? 2*MCB_MINB2 : (NALS==3 ? MCB_MINB3 : (NALS==4 ? MCB_MINB4 : MCB_MINB5));
    static constexpr int value  = BLOCK==256 ? per256 : (BLOCK==128 ? per128 : (BLOCK==64 ? (2*per128 > 32 ? 32 : 2*per128) : (4*per128 > 32 ? 32 : 4*per128)));
};

template<int NALS, bool PLOIDY, int BLOCK, typename PT, bool GPOUT>
__global__ void __launch_bounds__(BLOCK, (MinBlocks<NALS,BLOCK>::value)) mcall_site_kernel(const KArgs a)
{
    using PLT = PLType<PT>;
    constexpr int ES = PLT::ES;                 /* bytes per PL element in the slab and in the tile ring */
    using S = Shape<NALS>;
    constexpr int G = S::G, NPAIR = S::NPAIR, NTRI = S::NTRI, NSUB = S::NSUB, NACC = S::NACC;
    constexpr int MAXSEL = S::MAXSEL, NSLOT = S::NSLOT, NW = BLOCK/32;
    constexpr double LN2 = 0.693147180559945309417232121458, LN10_10 = 0.2302585092994045684017991454684;

    using SH = Shared<NALS,BLOCK>;
    SH &sh = *reinterpret_cast<SH*>(mcb_smem);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nsmpl = a.nsmpl, TS = a.tile_smpl, nstage = a.nstage;
    const int tile_ints = TS*G;
    const int ntiles = (nsmpl + TS - 1)/TS;
    const bool resident = ntiles <= nstage;
    const int total_visits = resident ? ntiles : 2*ntiles;
    const uint32_t sbase = smem_base();
    const uint32_t ring_s = sbase + (uint32_t)align128(sizeof(SH)), bars_s = sbase + (uint32_t)offsetof(SH, bars);
    const uint32_t pl2p_s = sbase + (uint32_t)offsetof(SH, pl2p), thr_s = sbase + (uint32_t)offsetof(SH, gq_thr);
    const uint32_t slot_s = sbase + (uint32_t)(offsetof(SH, p2) + offsetof(Phase2Consts, slot_out));
    const uint32_t hap_s  = sbase + (uint32_t)(offsetof(SH, p2) + offsetof(Phase2Consts, hap_out));

    for (int i=tid; i<256; i+=BLOCK) sh.pl2p[i] = a.tab->pl2p[i];
    for (int i=tid; i<130; i+=BLOCK) sh.gq_thr[i] = i<128 ? a.tab->gq_thr[i] : -1.0;
    if ( tid==0 )
    {
        for (int i=0; i<nstage; i++) mbar_init(bars_s + 8*i, 1);
        fence_mbar_init();
    }
    __syncthreads();

    uint32_t phase_bits = 0;
    const int nsites = *a.site_count;

#ifndef MCB_DYNAMIC
#define MCB_DYNAMIC 1       /* CTAs claim sites from a global counter (REF-only sites are cheap: a static stride leaves a long tail) */
#endif
#if MCB_DYNAMIC
    for (;;)
    {
        if ( tid==0 ) sh.next_site = atomicAdd(a.work_counter, 1);
        __syncthreads();
        const int isite = sh.next_site;
        if ( isite >= nsites ) break;
#else
    for (int isite = blockIdx.x; isite < nsites; isite += gridDim.x)
    {
#endif
        const int site = a.site_list[isite];
        const int64_t site_off = a.pl_off[site];
        const PT *site_pl = reinterpret_cast<const PT*>(a.pl) + site_off;
        const int unseen = a.unseen ? a.unseen[site] : 0;
        const uint8_t *ploidy = nullptr;
        if ( PLOIDY )
        {
            int pid = a.ploidy_id ? a.ploidy_id[site] : 0;
            if ( pid >= a.nploidy ) pid = 0;
            ploidy = a.ploidy_tab + (size_t)pid*nsmpl;
        }

        auto issue = [&](int v)
        {
            int t = v % ntiles, stage = v % nstage;
            int n = min(TS, nsmpl - t*TS);
            uint32_t bytes = ((uint32_t)(n*G*ES) + 15u) & ~15u;
            mbar_expect_tx(bars_s + 8*stage, bytes);
            bulk_g2s(ring_s + (uint32_t)(ES*stage*tile_ints), site_pl + (size_t)t*tile_ints, bytes, bars_s + 8*stage);
        };
        if ( tid==0 )
            for (int v=0; v<nstage && v<total_visits; v++) issue(v);

        /* ---- site set-up by thread 0: qsum (mcall.c:1454-1464), -F prior (1507-1527), normalisation (1530-1535) */
        if ( tid==0 )
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
            for (int j=0; j<NALS; j++) sh.qf[j] = q[j];
            sh.flags = flags;
            for (int j=0; j<8; j++) sh.ac[j] = 0;
        }
        __syncthreads();
        /* ---- allele-set coefficients, one lane per set.  float32 expression then widened (mcall.c:629-630, 671-673) */
        if ( warp==0 )
        {
            uint32_t live = 0;
            if ( lane < NPAIR )
            {
                int aa = 1; while ( aa*(aa+1)/2 <= lane ) aa++;     /* pair_idx(aa,bb)==lane */
                int bb = lane - aa*(aa-1)/2;
                float qa = sh.qf[aa], qb = sh.qf[bb];
                double *cf = sh.cf_pair + lane*5;
                if ( qa!=0 && qb!=0 )
                {
                    float den = __fadd_rn(qa,qb);
                    double fa = (double)__fdiv_rn(qa,den), fb = (double)__fdiv_rn(qb,den);
                    cf[0] = __dmul_rn(fa,fa); cf[1] = __dmul_rn(fb,fb); cf[2] = __dmul_rn(__dmul_rn(2.0,fa),fb);
                    cf[3] = fa; cf[4] = fb;
                    live = 1u<<lane;
                }
                else { cf[0] = cf[1] = cf[2] = cf[3] = cf[4] = 0; }
            }
            else if ( lane-NPAIR < NTRI )
            {
                int k = lane-NPAIR;
                int aa = 2; while ( (aa+1)*aa*(aa-1)/6 <= k ) aa++;
                int r = k - aa*(aa-1)*(aa-2)/6;
                int bb = 1; while ( bb*(bb+1)/2 <= r ) bb++;
                int cc = r - bb*(bb-1)/2;
                float qa = sh.qf[aa], qb = sh.qf[bb], qc = sh.qf[cc];
                double *cf = sh.cf_tri + k*9;
                if ( qa!=0 && qb!=0 && qc!=0 )
                {
                    float den = __fadd_rn(__fadd_rn(qa,qb),qc);
                    double fa = (double)__fdiv_rn(qa,den), fb = (double)__fdiv_rn(qb,den), fc = (double)__fdiv_rn(qc,den);
                    cf[0] = __dmul_rn(fa,fa); cf[1] = __dmul_rn(fb,fb); cf[2] = __dmul_rn(fc,fc);
                    cf[3] = __dmul_rn(__dmul_rn(2.0,fa),fb); cf[4] = __dmul_rn(__dmul_rn(2.0,fa),fc); cf[5] = __dmul_rn(__dmul_rn(2.0,fb),fc);
                    cf[6] = fa; cf[7] = fb; cf[8] = fc;
                    live = 1u<<lane;
                }
                else { for (int j=0; j<9; j++) cf[j] = 0; }
            }
            #pragma unroll
            for (int off=16; off; off>>=1) live |= __shfl_xor_sync(0xffffffffu, live, off);
            if ( lane==0 ) sh.live = live;
        }
        __syncthreads();
        const uint32_t live = sh.live;

        /* =========================== phase 1: site reduction ==================================== */
        double accM[NACC]; int accE[NACC];
        int plsum32[NALS]; long long plsum[NALS];
        int cnt_all = 0, cnt_called = 0, since_renorm = 0;
        uint32_t tflags = 0;
        #pragma unroll
        for (int k=0; k<NACC; k++) { accM[k] = 1.0; accE[k] = 0; }
        #pragma unroll
        for (int k=0; k<NALS; k++) { plsum[k] = 0; plsum32[k] = 0; }
        /* coefficients of the small shapes live in registers; larger shapes read them from shared memory */
        constexpr bool CF_REG = NALS<=2;
        double cfp[CF_REG ? (NPAIR ? NPAIR : 1)*5 : 1], cft[CF_REG ? (NTRI ? NTRI : 1)*9 : 1];
        if ( CF_REG )
        {
            #pragma unroll
            for (int k=0; k<NPAIR*5; k++) cfp[k] = sh.cf_pair[k];
            #pragma unroll
            for (int k=0; k<NTRI*9; k++) cft[k] = sh.cf_tri[k];
        }
        const uint32_t cfp_s = sbase + (uint32_t)offsetof(SH, cf_pair), cft_s = sbase + (uint32_t)offsetof(SH, cf_tri);
        auto CP = [&](int k, int c) -> double { return CF_REG ? cfp[CF_REG ? k*5+c : 0] : lds64(cfp_s + 8u*(uint32_t)(k*5+c)); };
        auto CT = [&](int k, int c) -> double { return CF_REG ? cft[CF_REG ? k*9+c : 0] : lds64(cft_s + 8u*(uint32_t)(k*9+c)); };

        for (int t=0; t<ntiles; t++)
        {
            const int stage = t % nstage;
            mbar_wait(bars_s + 8*stage, (phase_bits>>stage)&1u);
            phase_bits ^= 1u<<stage;
            const uint32_t tile_s = ring_s + (uint32_t)(ES*stage*tile_ints);
            const int s0 = t*TS, n = min(TS, nsmpl - s0);
            /* pass 0: normalisers, single-allele sums, pairs (+ triples unless SPLIT); pass 1 (SPLIT): triples */
            #pragma unroll 1
            for (int pass=0; pass<(S::SPLIT ? 2 : 1); pass++)
            {
                const bool do_pairs = pass==0, do_tri = S::SPLIT ? pass==1 : true;
                #pragma unroll (kUnroll1)
                for (int sb=0; sb<n; sb+=BLOCK)         /* uniform trip count: the loader votes across the warp */
                {
                    const int s = min(sb + tid, n-1);
                    const bool valid = sb + tid < n;
                    int pl[G]; double p[G]; double sum; bool fast;
                    if ( !load_sample_w<NALS,PT>(tile_s + (uint32_t)(s*G*ES), pl2p_s, valid, unseen, a.tab, pl, p, sum, fast, tflags) ) continue;
                    int pld = 2;
                    if ( PLOIDY ) pld = __ldg(ploidy + s0 + s);
                    if ( pass==0 )
                    {
                        /* single-allele sets: log(pdg[aa]) = -PL*ln10/10 - log(sum), every sample incl. ploidy 0 (mcall.c:607-611) */
                        if ( !fast )
                        {
                            #pragma unroll
                            for (int k=0; k<NALS; k++) plsum[k] += pl[hom_idx(k)];
                        }
                        else
                        {
                            #pragma unroll
                            for (int k=0; k<NALS; k++) plsum32[k] += pl[hom_idx(k)];
                        }
                        cnt_all++;
                        acc_mul(accM[NACC-2], accE[NACC-2], sum);
                        if ( PLOIDY && pld!=0 ) { cnt_called++; acc_mul(accM[NACC-1], accE[NACC-1], sum); }
                    }
                    if ( PLOIDY && pld==0 ) continue;       /* ploidy 0: val stays 0 (mcall.c:639-644) */
                    if ( !PLOIDY || pld==2 )
                    {
                        if ( do_pairs )
                        {
                            #pragma unroll
                            for (int x=1; x<NALS; x++)
                                #pragma unroll
                                for (int y=0; y<x; y++)
                                {
                                    const int k = pair_idx(x,y);
                                    if ( live & (1u<<k) )
                                    {
                                        double val = fma(CP(k,2), p[gt_idx(x,y)], fma(CP(k,1), p[hom_idx(y)], CP(k,0)*p[hom_idx(x)]));
                                        acc_mul(accM[k], accE[k], val);
                                    }
                                }
                        }
                        if ( do_tri )
                        {
                            #pragma unroll
                            for (int x=2; x<NALS; x++)
                                #pragma unroll
                                for (int y=1; y<x; y++)
                                    #pragma unroll
                                    for (int z=0; z<y; z++)
                                    {
                                        const int k = tri_idx(x,y,z);
                                        if ( live & (1u<<(NPAIR+k)) )
                                        {
                                            double val = fma(CT(k,5), p[gt_idx(y,z)], fma(CT(k,4), p[gt_idx(x,z)], fma(CT(k,3), p[gt_idx(x,y)],
                                                         fma(CT(k,2), p[hom_idx(z)], fma(CT(k,1), p[hom_idx(y)], CT(k,0)*p[hom_idx(x)])))));
                                            acc_mul(accM[NPAIR+k], accE[NPAIR+k], val);
                                        }
                                    }
                        }
                    }
                    else    /* haploid (mcall.c:642-643, 687-688) */
                    {
                        if ( do_pairs )
                        {
                            #pragma unroll
                            for (int x=1; x<NALS; x++)
                                #pragma unroll
                                for (int y=0; y<x; y++)
                                {
                                    const int k = pair_idx(x,y);
                                    if ( live & (1u<<k) )
                                    {
                                        double val = fma(CP(k,4), p[hom_idx(y)], CP(k,3)*p[hom_idx(x)]);
                                        acc_mul(accM[k], accE[k], val);
                                    }
                                }
                        }
                        if ( do_tri )
                        {
                            #pragma unroll
                            for (int x=2; x<NALS; x++)
                                #pragma unroll
                                for (int y=1; y<x; y++)
                                    #pragma unroll
                                    for (int z=0; z<y; z++)
                                    {
                                        const int k = tri_idx(x,y,z);
                                        if ( live & (1u<<(NPAIR+k)) )
                                        {
                                            double val = fma(CT(k,8), p[hom_idx(z)], fma(CT(k,7), p[hom_idx(y)], CT(k,6)*p[hom_idx(x)]));
                                            acc_mul(accM[NPAIR+k], accE[NPAIR+k], val);
                                        }
                                    }
                        }
                    }
                }
            }
            #pragma unroll
            for (int k=0; k<NALS; k++) { plsum[k] += plsum32[k]; plsum32[k] = 0; }
            since_renorm += (TS + BLOCK - 1)/BLOCK;
            if ( since_renorm >= 256 )
            {
                #pragma unroll
                for (int k=0; k<NACC; k++) acc_renorm(accM[k], accE[k]);
                since_renorm = 0;
            }
            if ( !resident )
            {
                fence_proxy_async();
                __syncthreads();
                if ( tid==0 && t+nstage < total_visits ) issue(t+nstage);
            }
        }
        if ( !PLOIDY ) cnt_called = cnt_all;

        /* ---- block reduction of the products (mantissa multiply, exponent add) and the integer sums */
        #pragma unroll
        for (int k=0; k<NACC; k++)
        {
            if ( !PLOIDY && k==NACC-1 ) continue;
            acc_renorm(accM[k], accE[k]);
            #pragma unroll
            for (int off=16; off; off>>=1)
            {
                accM[k] = __dmul_rn(accM[k], __shfl_xor_sync(0xffffffffu, accM[k], off));
                accE[k] += __shfl_xor_sync(0xffffffffu, accE[k], off);
            }
            acc_renorm(accM[k], accE[k]);
        }
        #pragma unroll
        for (int k=0; k<NALS; k++)
            #pragma unroll
            for (int off=16; off; off>>=1) plsum[k] += __shfl_xor_sync(0xffffffffu, plsum[k], off);
        #pragma unroll
        for (int off=16; off; off>>=1)
        {
            cnt_all    += __shfl_xor_sync(0xffffffffu, cnt_all, off);
            cnt_called += __shfl_xor_sync(0xffffffffu, cnt_called, off);
            tflags     |= __shfl_xor_sync(0xffffffffu, tflags, off);
        }
        if ( lane==0 )
        {
            #pragma unroll
            for (int k=0; k<NACC; k++) { sh.red_M[warp][k] = accM[k]; sh.red_E[warp][k] = accE[k]; }
            #pragma unroll
            for (int k=0; k<NALS; k++) sh.red_pls[warp][k] = plsum[k];
            sh.red_cnt[warp][0] = cnt_all; sh.red_cnt[warp][1] = cnt_called;
            if ( tflags ) atomicOr(&sh.flags, tflags);
        }
        __syncthreads();

        /* ---- epilogue, warp 0: lane k <-> allele set k in the reference's enumeration order ------------- */
        if ( warp==0 )
        {
            int n_all = 0, n_called = 0;
            #pragma unroll
            for (int w=0; w<NW; w++) { n_all += sh.red_cnt[w][0]; n_called += sh.red_cnt[w][1]; }
            auto total_log = [&](int k, int n) -> double
            {
                double M = 1.0; int E = 0;
                #pragma unroll
                for (int w=0; w<NW; w++) { M = __dmul_rn(M, sh.red_M[w][k]); E += sh.red_E[w][k]; }
                return site_log(M) + (double)(E - 1023*n)*LN2;
            };
            const double lnN_all    = n_all ? total_log(NACC-2, n_all) : 0.0;
            const double lnN_called = PLOIDY ? (n_called ? total_log(NACC-1, n_called) : 0.0) : lnN_all;

            double lk = 0; bool cand = false, in_sum = false; uint32_t mask = 0;
            if ( lane < NALS )
            {
                long long ps = 0;
                #pragma unroll
                for (int w=0; w<NW; w++) ps += sh.red_pls[w][lane];
                bool set = n_all > 0;
                lk = set ? -LN10_10*(double)ps - lnN_all : 0.0;
                if ( lane>0 ) lk += a.theta;
                cand = set; in_sum = set && lane>0; mask = 1u<<lane;
            }
            else if ( lane < NSUB )
            {
                int k = lane - NALS;                    /* accumulator index: pairs then triples */
                bool lv = (live >> k) & 1u;
                bool set = lv && n_called > 0;
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
                lk = set ? total_log(k, n_called) - lnN_called : 0.0;
                for (int j=0; j<nonref; j++) lk += a.theta;
                cand = set; in_sum = set;
            }
            if ( a.exact_phase1 )       /* near-tie adjudication: the literal sample-sequential sums of logs instead */
            {
                bool is_set = false;
                uint32_t xflags = 0;
                const double xlk = exact_set_lk<NALS,PLOIDY,PT>(site_pl, nullptr, nsmpl, unseen, ploidy, pl2p_s, a.tab, lane, sh.cf_pair, sh.cf_tri, live, a.theta, &is_set, &xflags);
                if ( lane < NSUB )
                {
                    lk = xlk; cand = is_set;
                    in_sum = is_set && lane != 0;           /* UPDATE_MAX_LKs(1<<ia, ia>0 && lk_tot_set) / (..., lk_tot_set) */
                    if ( lane==0 && !is_set ) lk = 0;       /* ref_lk = lk_tot of {REF}, also when nothing was added */
                }
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
            double term = in_sum ? site_exp(lk - mx) : 0.0;
            #pragma unroll
            for (int off=16; off; off>>=1) term += __shfl_xor_sync(0xffffffffu, term, off);
            double grp_lk_sum = mx > -CUDART_INF ? mx + site_log(term) : -CUDART_INF;
            if ( a.exact_phase1 )       /* ... and lk_sum as the reference's running logsumexp2 in enumeration order (mcall.c:573-585) */
                grp_lk_sum = exact_lk_sum(lk, in_sum, NSUB, -CUDART_INF);
            const double grp_ref_lk = __shfl_sync(0xffffffffu, lk, 0);
            const uint32_t grp_als = __shfl_sync(0xffffffffu, mask, best_lane & 31);

            if ( lane==0 )
            {
                const bool any = best_lane < 64;
                uint32_t gals = any ? grp_als : 0;
                uint32_t flags = sh.flags;
                double max_qual = -CUDART_INF, lk_sum = -CUDART_INF, ref_lk = -CUDART_INF;
                if ( any )          /* mcall.c:1553-1560 */
                {
                    max_qual = -4.343*(grp_ref_lk - logsumexp2_dev(grp_lk_sum, grp_ref_lk));
                    lk_sum = grp_lk_sum; ref_lk = grp_ref_lk;
                }
                double gap = any ? best - second : CUDART_INF;
                if ( any && gap < a.tie_eps ) flags |= MCB_SITE_NEAR_TIE;
                if ( a.adj_pass ) flags |= MCB_SITE_NEAR_TIE | MCB_SITE_ADJUDICATED;
                uint32_t als_new = gals | 1u;               /* mcall.c:1552, 1564 */
                int is_variant = als_new!=1;
                int ret_early = ((a.flag & MCB_CALL_VARONLY) && !is_variant) || (flags & MCB_SITE_NO_QS);
                int nals_new = 0;
                #pragma unroll
                for (int j=0; j<NALS; j++)                  /* mcall.c:1569-1575 */
                {
                    if ( j>0 && j==unseen ) continue;
                    if ( a.flag & MCB_CALL_KEEPALT ) als_new |= 1u<<j;
                    if ( als_new & (1u<<j) ) nals_new++;
                }
                int nout = 0, kk = 0, l = 0;                /* mcall.c:547-570 */
                int amap[NALS];
                #pragma unroll
                for (int x=0; x<NALS; x++) { amap[x] = (als_new & (1u<<x)) ? nout++ : -1; sh.als_map[x] = amap[x]; }
                #pragma unroll
                for (int x=0; x<NALS; x++)
                    #pragma unroll
                    for (int y=0; y<=x; y++) { if ( (als_new & (1u<<x)) && (als_new & (1u<<y)) ) { if ( kk<G ) sh.pl_map[kk] = l; kk++; } l++; }
                for (; kk<G; kk++) sh.pl_map[kk] = 0;
                if ( unseen && (als_new & (1u<<unseen)) ) flags |= MCB_SITE_UNSEEN_SEL;
                sh.pl_dropped = als_new==1;
                sh.ref_gt = (als_new==1) || !is_variant;
                {
                    long long off = site_off;
                    if ( a.pl_off_out )
                    {
                        off = compact_out_off<true>(a, site, nsmpl, NALS, nals_new, !sh.pl_dropped && !ret_early, flags);
                        a.pl_off_out[site] = off;
                    }
                    sh.out_off = off;
                }
                if ( sh.pl_dropped ) flags |= MCB_SITE_PL_DROPPED;
                if ( sh.ref_gt ) flags |= MCB_SITE_REF_GT;
                int gn = 0;
                #pragma unroll
                for (int j=0; j<NALS; j++) gn += (gals>>j)&1u;
                sh.grp_als = gals; sh.grp_nals = gn; sh.als_new = als_new; sh.nals_new = nals_new;
                sh.is_variant = is_variant; sh.ret_early = ret_early; sh.flags = flags;
                sh.max_qual = max_qual; sh.lk_sum = lk_sum; sh.ref_lk = ref_lk; sh.gap = gap;
                /* phase-2 constants: selected alleles in ascending order and the <=6 genotypes they span */
                {
                    Phase2Consts &c = sh.p2;
                    const int ngt_new = nals_new*(nals_new+1)/2;
                    int sel[3] = {0,0,0}, ns = 0;
                    #pragma unroll
                    for (int j=0; j<NALS; j++) if ( (gals>>j)&1u ) { if ( ns<3 ) sel[ns] = j; ns++; }
                    if ( ns>3 ) ns = 3;
                    c.nsel = ns; c.inc_dip = 0; c.inc_hap = 0;
                    for (int x=0; x<3; x++)
                    {
                        c.q[x] = x<ns ? (double)sh.qf[sel[x]] : 0.0;
                        int nx = x<ns ? amap[sel[x]] : 0;
                        c.hap_new[x] = nx;
                        if ( x<ns && nx < gn ) c.inc_hap |= 1u<<x;
                        unsigned long long hinc = 1ull << (12*min(nx,4));
                        c.hap_out[x] = make_int4(MCB_GT_UNPHASED(nx), I32_VEC_END, (int)(uint32_t)hinc, (int)(uint32_t)(hinc>>32));
                        for (int y=0; y<=x; y++)
                        {
                            int k = x*(x+1)/2 + y;
                            int ny = y<ns ? amap[sel[y]] : 0;
                            c.jgt4[k] = (x<ns) ? ES*gt_idx(sel[x], sel[y]) : 0;
                            int ig = gt_idx(nx, ny);
                            c.igt[k] = ig;
                            if ( x<ns && ig < ngt_new ) c.inc_dip |= 1u<<k;
                            /* gts[0] = smaller new allele, gts[1] = larger (mcall.c:830-831); AC: one count per allele */
                            unsigned long long inc = (1ull << (12*min(ny,4))) + (1ull << (12*min(nx,4)));
                            c.slot_out[k] = make_int4(MCB_GT_UNPHASED(ny), MCB_GT_UNPHASED(nx), (int)(uint32_t)inc, (int)(uint32_t)(inc>>32));
                        }
                    }
                }
            }
        }
        __syncthreads();

        /* =========================== phase 2: per-sample genotypes ============================== */
        if ( sh.ret_early )
        {
            if ( tid==0 )
            {
                a.ret[site] = 0;
                if ( a.site_flags ) a.site_flags[site] = sh.flags;
            }
            /* drain the phase-2 tiles already in flight for this site (streaming mode): they hit L2 */
            if ( !resident )
                for (int v=ntiles; v<ntiles+nstage && v<total_visits; v++)
                {
                    const int stage = v % nstage;
                    mbar_wait(bars_s + 8*stage, (phase_bits>>stage)&1u);
                    phase_bits ^= 1u<<stage;
                }
            __syncthreads();
            continue;
        }
        {
            const int nals_new = sh.nals_new, ngt_new = nals_new*(nals_new+1)/2, grp_nals = sh.grp_nals;
            const bool ref_gt = sh.ref_gt, pl_dropped = sh.pl_dropped;
            const bool want_gq = a.gq && (a.output_tags & (MCB_CALL_FMT_GQ|MCB_CALL_FMT_GP));
            /* FORMAT/GP is compiled into its own instances: its code in the sample loop costs the GP-less kernels 2-6 % */
            const bool want_gp = GPOUT && a.gp && (a.output_tags & MCB_CALL_FMT_GP) && !ref_gt;
            const bool want_gqm = want_gq || want_gp;       /* the max/sum arithmetic is shared by GQ and GP */
            int32_t *out_pl = (a.out_pl && !pl_dropped) ? a.out_pl + sh.out_off : nullptr;
            float   *out_gp = want_gp ? a.gp + sh.out_off : nullptr;
            int2 *out_gt = a.gt ? reinterpret_cast<int2*>(a.gt) + (size_t)site*nsmpl : nullptr;
            int32_t *out_gq = want_gq ? a.gq + (size_t)site*nsmpl : nullptr;
            /* per-site constants into registers */
            const int nsel = sh.p2.nsel;
            const double q0 = sh.p2.q[0], q1 = sh.p2.q[1], q2 = sh.p2.q[2];
            int jgt4[NSLOT];
            #pragma unroll
            for (int k=0; k<NSLOT; k++) jgt4[k] = sh.p2.jgt4[k];
            const uint32_t inc_dip = sh.p2.inc_dip, inc_hap = sh.p2.inc_hap;
            const uint32_t full_dip = nsel>=3 ? 0x3fu : (nsel==2 ? 0x7u : 0x1u), full_hap = (1u<<nsel) - 1u;
            const bool inc_full = (inc_dip & full_dip)==full_dip && (inc_hap & full_hap)==full_hap;
            constexpr int NPLM = G<6 ? G : 6;
            int plm4[NPLM];
            #pragma unroll
            for (int k=0; k<NPLM; k++) plm4[k] = ES*sh.pl_map[k];
            const uint32_t oflags = (out_gt ? 1u : 0u) | (out_gq ? 2u : 0u) | (out_pl ? 4u : 0u) | (out_gp ? 8u : 0u);
            /*  fast2: every sample diploid, the selected set is a pair s0<s1 whose alleles are exactly the kept ones (new alleles
             *  0 and 1, all three new genotypes below ngt_new), GT + GQ + PL all written, int32 PLs, an even sample count
             *  and 16-byte aligned outputs (pairs of samples leave in vector stores).  CTA-uniform.  */
            constexpr bool PAIR_OK = !PLOIDY && !GPOUT && ES==4 && NALS>=2;
            constexpr bool FAST2 = PAIR_OK && (MCB_FAST2 || (MCB_FAST2_N2 && NALS==2));     /* two alleles (S > 8,192, the biobank shape): the small kernel takes the extra path without fetch misses */
            const bool pair_site = PAIR_OK && !ref_gt && nsel==2 && (inc_dip & 7u)==7u && nals_new==2 && sh.als_new==sh.grp_als && want_gq
                               && oflags==7u && !(nsmpl & 1)
                               && !((reinterpret_cast<uintptr_t>(out_gt) & 15) | (reinterpret_cast<uintptr_t>(out_gq) & 7) | (reinterpret_cast<uintptr_t>(out_pl) & 7));
            /* two-allele instances: measured +16 % at 100,000 samples (C4), -4..-9 % at 1,000-2,504 (where the warp kernel of
               mcall_biallelic.cu is the default path anyway) */
            const bool fast2 = FAST2 && pair_site && !(TS & 1) && (MCB_FAST2 || nsmpl > 8192);
            const double fq0 = q0, fq1 = q1, fq1x2 = __dmul_rn(2.0, q1);
            const int fj0 = jgt4[0], fj1 = jgt4[NSLOT>1 ? 1 : 0], fj2 = jgt4[NSLOT>2 ? 2 : 0];
            int f_alt = 0, f_called = 0;
            unsigned long long acc = 0;     /* AC: 12-bit counters, new allele j at bits [12j,12j+12) */
            int acc_n = 0;
            uint32_t tflags2 = 0;
            auto flush_ac = [&]()           /* called by all threads of the block together */
            {
                unsigned long long v = acc;     /* <= 2*60 per lane and field: no carry between the 12-bit fields within a warp */
                #pragma unroll
                for (int off=16; off; off>>=1) v += __shfl_xor_sync(0xffffffffu, v, off);
                if ( lane==0 )
                {
                    #pragma unroll
                    for (int j=0; j<5; j++)
                    {
                        int c = (int)((v >> (12*j)) & 0xfff);
                        if ( c ) atomicAdd(&sh.ac[j], c);
                    }
                }
                acc = 0; acc_n = 0;
            };

            for (int t=0; t<ntiles; t++)
            {
                const int v = resident ? t : ntiles + t, stage = v % nstage;
                if ( !resident )
                {
                    mbar_wait(bars_s + 8*stage, (phase_bits>>stage)&1u);
                    phase_bits ^= 1u<<stage;
                }
                const uint32_t tile_s = ring_s + (uint32_t)(ES*stage*tile_ints);
                const int s0 = t*TS, n = min(TS, nsmpl - s0);
                const int per_tile = 2*((TS + 2*BLOCK - 1)/(2*BLOCK));     /* samples of a tile per thread */
                if ( acc_n + per_tile > 63 ) flush_ac();                    /* uniform across the block: safe to shuffle */
                acc_n += per_tile;
                #pragma unroll 1
                for (int sb=0; sb<n; sb+=2*BLOCK)       /* uniform trip count: the loaders vote across the warp */
                {
                const int wb = sb + 64*warp;            /* a warp owns 64 consecutive samples per iteration */
                bool done = false;
                if constexpr ( FAST2 ) if ( fast2 )
                {
                    /*  The common variant site (see fast2 above): each lane takes TWO ADJACENT samples, straight-line code
                     *  (fast2_call), GT / GQ / PL of the pair leave as one 128-bit and four 64-bit stores.  A warp whose 64
                     *  samples hold a missing value or a PL >= 256 votes itself onto the general path below.  */
                    const int sp = wb + 2*lane;
                    const bool valid = sp < n;
                    const uint32_t row_s = tile_s + (uint32_t)((valid ? sp : 0)*G*4);
                    int pl2[2*G];
                    if constexpr ( (G & 1)==0 )
                    {
                        #pragma unroll
                        for (int j=0; j<2*G; j+=4) { const int4 v = lds128(row_s + 4u*j); pl2[j] = v.x; pl2[j+1] = v.y; pl2[j+2] = v.z; pl2[j+3] = v.w; }
                    }
                    else
                    {
                        #pragma unroll
                        for (int j=0; j<2*G; j+=2) { pl2[j] = lds32(row_s + 4u*j); pl2[j+1] = lds32(row_s + 4u*j + 4u); }
                    }
                    int orv0 = 0, orv1 = 0;
                    #pragma unroll
                    for (int j=0; j<G; j++) { orv0 |= pl2[j]; orv1 |= pl2[G+j]; }
                    if ( !__any_sync(0xffffffffu, (unsigned)(orv0 | orv1) > 255u) )
                    {
                        done = true;
                        if ( valid )
                        {
                            int k0, k1, g0, g1;
                            const int a0 = lds32(row_s + (uint32_t)fj0), b0 = lds32(row_s + (uint32_t)fj1), c0 = lds32(row_s + (uint32_t)fj2);
                            const int a1 = lds32(row_s + (uint32_t)(4*G) + (uint32_t)fj0), b1 = lds32(row_s + (uint32_t)(4*G) + (uint32_t)fj1), c1 = lds32(row_s + (uint32_t)(4*G) + (uint32_t)fj2);
                            {
                                double sum = lds64c(pl2p_s + 8u*(uint32_t)pl2[0]);
                                #pragma unroll
                                for (int j=1; j<G; j++) sum = __dadd_rn(sum, lds64c(pl2p_s + 8u*(uint32_t)pl2[j]));
                                fast2_call(lds64c(pl2p_s + 8u*(uint32_t)a0), lds64c(pl2p_s + 8u*(uint32_t)b0), lds64c(pl2p_s + 8u*(uint32_t)c0),
                                           sum, fq0, fq1, fq1x2, thr_s, k0, g0);
                            }
                            {
                                double sum = lds64c(pl2p_s + 8u*(uint32_t)pl2[G]);
                                #pragma unroll
                                for (int j=1; j<G; j++) sum = __dadd_rn(sum, lds64c(pl2p_s + 8u*(uint32_t)pl2[G+j]));
                                fast2_call(lds64c(pl2p_s + 8u*(uint32_t)a1), lds64c(pl2p_s + 8u*(uint32_t)b1), lds64c(pl2p_s + 8u*(uint32_t)c1),
                                           sum, fq0, fq1, fq1x2, thr_s, k1, g1);
                            }
                            const bool has0 = orv0 != 0, has1 = orv1 != 0;      /* PL=0,..,0: no data (mcall.c:529-537) */
                            /* new alleles 0 and 1: GT codes 2 and 4, slot index = copies of allele 1; no data: ./. and GQ 0 */
                            const int x0 = has0 ? (k0==2 ? 4 : 2) : 0, y0 = has0 ? (k0 ? 4 : 2) : 0;
                            const int x1 = has1 ? (k1==2 ? 4 : 2) : 0, y1 = has1 ? (k1 ? 4 : 2) : 0;
                            f_alt += (has0 ? k0 : 0) + (has1 ? k1 : 0); f_called += (int)has0 + (int)has1;
                            const size_t sg = (size_t)(s0 + sp);
                            asm volatile("st.global.v4.s32 [%0], {%1,%2,%3,%4};" :: "l"(out_gt + sg), "r"(x0), "r"(y0), "r"(x1), "r"(y1) : "memory");
                            asm volatile("st.global.v2.s32 [%0], {%1,%2};" :: "l"(out_gq + sg), "r"(has0 ? g0 : 0), "r"(has1 ? g1 : 0) : "memory");
                            const int32_t *dst = out_pl + 3*sg;             /* mcall.c:1158-1194: the kept genotypes are the three slots */
                            asm volatile("st.global.v2.s32 [%0], {%1,%2};" :: "l"(dst), "r"(a0), "r"(b0) : "memory");
                            asm volatile("st.global.v2.s32 [%0+8], {%1,%2};" :: "l"(dst), "r"(c0), "r"(a1) : "memory");
                            asm volatile("st.global.v2.s32 [%0+16], {%1,%2};" :: "l"(dst), "r"(b1), "r"(c1) : "memory");
                        }
                    }
                }
                if ( !done )
                #pragma unroll 1
                for (int half=0; half<2; half++)
                {
                    const int sidx = wb + 32*half + lane;
                    const int s = min(sidx, n-1);
                    const bool valid = sidx < n;
                    int pl[G]; double p[G]; double sum = 1; bool fast;
                    const uint32_t row_s = tile_s + (uint32_t)(s*G*ES);
                    const bool has = load_sample_w<NALS,PT>(row_s, pl2p_s, valid, unseen, a.tab, pl, p, sum, fast, tflags2);
                    const int pld = PLOIDY ? __ldg(ploidy + s0 + s) : 2;
                    int4 outc = make_int4(MCB_GT_MISSING, pld==2 ? MCB_GT_MISSING : I32_VEC_END, 0, 0);
                    int gq = 0;
                    bool called = false;
                    double gsum = 0;
                    double gv[NSLOT];
                    if ( !pld || !has ) { }
                    else if ( ref_gt )          /* mcall.c:713-743 */
                    {
                        outc = make_int4(MCB_GT_UNPHASED(0), pld==2 ? MCB_GT_UNPHASED(0) : I32_VEC_END, pld, 0);
                    }
                    else                        /* mcall.c:787-840, literal arithmetic */
                    {
                        called = true;
                        const double r = fast ? rcp_shared(sum) : 0.0;     /* `fast` is warp-uniform */
                        auto pdg_of = [&](int k) -> double
                        {
                            double pk;
                            if ( NALS==1 ) pk = p[0];
                            else if ( NALS==2 ) pk = k==1 ? p[1] : (k==2 ? p[2] : (jgt4[0] ? p[2] : p[0]));
                            else
                            {
                                const int v = PLT::ld(row_s + (uint32_t)jgt4[k<NSLOT?k:0]);
                                pk = (fast || v<256) ? lds64(pl2p_s + 8u*(uint32_t)(v & 255)) : big_pl_to_p(a.tab, v, &tflags2);
                            }
                            return fast ? div_shared(pk, sum, r) : __ddiv_rn(pk, sum);
                        };
                        double best = 0; int bk = 0;        /* default 0/0 when every lk is 0 (mcall.c:787-789) */
                        bool any_best = false;
                        #pragma unroll
                        for (int k=0; k<NSLOT; k++) gv[k] = 0;
                        /* homozygous / haploid, a ascending (mcall.c:793-808) */
                        {
                            const double pdg = pdg_of(0);
                            const double lk = pld==2 ? __dmul_rn(__dmul_rn(pdg,q0),q0) : __dmul_rn(pdg,q0);
                            gv[0] = lk;
                            if ( best < lk ) { best = lk; bk = 0; any_best = true; }
                        }
                        if constexpr ( MAXSEL>1 ) if ( nsel>1 )
                        {
                            const double pdg = pdg_of(2);
                            const double lk = pld==2 ? __dmul_rn(__dmul_rn(pdg,q1),q1) : __dmul_rn(pdg,q1);
                            gv[2] = lk;
                            if ( best < lk ) { best = lk; bk = 2; any_best = true; }
                        }
                        if constexpr ( MAXSEL>2 ) if ( nsel>2 )
                        {
                            const double pdg = pdg_of(5);
                            const double lk = pld==2 ? __dmul_rn(__dmul_rn(pdg,q2),q2) : __dmul_rn(pdg,q2);
                            gv[5] = lk;
                            if ( best < lk ) { best = lk; bk = 5; any_best = true; }
                        }
                        if ( pld==2 )
                        {
                            /* heterozygous: (s1,s0), (s2,s0), (s2,s1)  (mcall.c:812-834) */
                            if constexpr ( MAXSEL>1 ) if ( nsel>1 )
                            {
                                const double lk = __dmul_rn(__dmul_rn(__dmul_rn(2.0,pdg_of(1)),q1),q0);
                                gv[1] = lk;
                                if ( best < lk ) { best = lk; bk = 1; any_best = true; }
                            }
                            if constexpr ( MAXSEL>2 ) if ( nsel>2 )
                            {
                                const double lk = __dmul_rn(__dmul_rn(__dmul_rn(2.0,pdg_of(3)),q2),q0);
                                gv[3] = lk;
                                if ( best < lk ) { best = lk; bk = 3; any_best = true; }
                                const double lk2 = __dmul_rn(__dmul_rn(__dmul_rn(2.0,pdg_of(4)),q2),q1);
                                gv[4] = lk2;
                                if ( best < lk2 ) { best = lk2; bk = 4; any_best = true; }
                            }
                            /* nothing beat 0: the reference keeps its 0/0 default, i.e. NEW allele 0 (mcall.c:788) */
                            outc = any_best ? lds128(slot_s + 16u*(uint32_t)bk) : make_int4(MCB_GT_UNPHASED(0), MCB_GT_UNPHASED(0), 2, 0);
                        }
                        else
                        {
                            const int bx = bk==0 ? 0 : (bk==2 ? 1 : 2);
                            outc = any_best ? lds128(hap_s + 16u*(uint32_t)bx) : make_int4(MCB_GT_UNPHASED(0), I32_VEC_END, 1, 0);
                        }
                        if ( want_gqm )         /* mcall.c:843-878: max and sum over the float32 gps[0..nmax) in index order */
                        {
                            double gmax;
                            #pragma unroll
                            for (int k=0; k<NSLOT; k++) gv[k] = (double)__double2float_rn(gv[k]);
                            if ( inc_full )
                            {
                                /* float rounding is monotone: max of the rounded values = rounded max */
                                gmax = (double)__double2float_rn(best);
                                gsum = gv[0];
                                #pragma unroll
                                for (int k=1; k<NSLOT; k++) gsum = __dadd_rn(gsum, gv[k]);     /* absent slots hold +0 */
                            }
                            else
                            {
                                gmax = 0;
                                const uint32_t inc = pld==2 ? inc_dip : ((inc_hap&1u) | ((inc_hap&2u)<<1) | ((inc_hap&4u)<<3));
                                #pragma unroll
                                for (int k=0; k<NSLOT; k++)
                                    if ( inc & (1u<<k) )
                                    {
                                        if ( gmax < gv[k] ) gmax = gv[k];
                                        gsum = __dadd_rn(gsum, gv[k]);
                                    }
                            }
                            const double xx = __dadd_rn(1.0, -__ddiv_rn(gmax, gsum));
                            if ( !(xx==xx) ) gq = 127;      /* NaN (0/0): `max<=INT8_MAX` is false => INT8_MAX */
                            else
                            {
                                /* (int)(-4.34294*log(x)) from host-libm thresholds: float estimate, exact fix-up */
                                int k = __float2int_rz(-3.0102999f*lg2_approx((float)xx));
                                k = max(0, min(127, k));
                                if ( xx <= lds64c(thr_s + 8u*(uint32_t)(k+1)) ) { k++; while ( xx <= lds64c(thr_s + 8u*(uint32_t)(k+1)) ) k++; }
                                else while ( xx > lds64c(thr_s + 8u*(uint32_t)k) ) k--;
                                gq = k;
                            }
                        }
                    }
                    if ( !valid ) continue;
                    acc += (unsigned long long)(uint32_t)outc.z | ((unsigned long long)(uint32_t)outc.w << 32);
                    const int sg = s0 + s;
                    /* stores: one address computation per output array, explicit PTX so that it is not rebuilt per value */
                    if ( oflags & 1u )
                    {
                        const int2 *p2 = out_gt + sg;
                        asm volatile("st.global.v2.s32 [%0], {%1,%2};" :: "l"(p2), "r"(outc.x), "r"(outc.y) : "memory");
                    }
                    if ( oflags & 2u )
                    {
                        const int32_t *p1 = out_gq + sg;
                        asm volatile("st.global.s32 [%0], %1;" :: "l"(p1), "r"(gq) : "memory");
                    }
                    if ( oflags & 4u )          /* mcall.c:1158-1194; the ring row holds the filled PLs */
                    {
                        const int32_t *dst = out_pl + (size_t)sg*ngt_new;
                        if ( G<=3 || ngt_new<=3 )       /* at most 3 values: the common, fully unrolled case */
                        {
                            int v0, v1 = I32_VEC_END, v2 = I32_VEC_END;
                            if ( pld==2 )
                            {
                                v0 = PLT::widen(PLT::ld(row_s + (uint32_t)plm4[0]));
                                if ( G>1 ) { v1 = PLT::widen(PLT::ld(row_s + (uint32_t)plm4[G>1?1:0])); v2 = PLT::widen(PLT::ld(row_s + (uint32_t)plm4[G>2?2:0])); }
                            }
                            else if ( pld==1 )
                            {
                                v0 = PLT::widen(PLT::ld(row_s + (uint32_t)plm4[0]));                   /* hom_idx(0) = 0 */
                                if ( G>1 && nals_new>1 ) v1 = PLT::widen(PLT::ld(row_s + (uint32_t)plm4[G>2?2:0]));  /* hom_idx(1) = 2 */
                            }
                            else v0 = I32_MISSING;
                            asm volatile("st.global.s32 [%0], %1;" :: "l"(dst), "r"(v0) : "memory");
                            if ( ngt_new>1 )
                            {
                                asm volatile("st.global.s32 [%0+4], %1;" :: "l"(dst), "r"(v1) : "memory");
                                asm volatile("st.global.s32 [%0+8], %1;" :: "l"(dst), "r"(v2) : "memory");
                            }
                        }
                        else
                        {
                            #pragma unroll
                            for (int k=0; k<G; k++)
                            {
                                if ( k>=ngt_new ) continue;
                                int v;
                                if ( pld==2 ) v = PLT::widen(PLT::ld(row_s + (uint32_t)(k<NPLM ? plm4[k<NPLM?k:0] : ES*sh.pl_map[k])));
                                else if ( pld==1 ) v = k<nals_new ? PLT::widen(PLT::ld(row_s + (uint32_t)(ES*sh.pl_map[hom_idx(k)]))) : I32_VEC_END;
                                else v = k==0 ? I32_MISSING : I32_VEC_END;
                                asm volatile("st.global.s32 [%0], %1;" :: "l"(dst + k), "r"(v) : "memory");
                            }
                        }
                    }
                    if ( oflags & 8u )          /* FORMAT/GP, mcall.c:859-884 (gv[] holds the float32-rounded values) */
                    {
                        float *dst = out_gp + (size_t)sg*ngt_new;
                        const int nmax = pld==2 ? ngt_new : (pld==1 ? grp_nals : 0);
                        if ( !called )
                        {
                            for (int k=0; k<ngt_new; k++) dst[k] = 0.f;
                            if ( nmax==0 ) { dst[0] = __uint_as_float(MCB_FLOAT_MISSING_BITS); if ( 1<ngt_new ) dst[1] = __uint_as_float(MCB_FLOAT_VECTOR_END_BITS); }
                            else if ( nmax<ngt_new ) dst[nmax] = __uint_as_float(MCB_FLOAT_VECTOR_END_BITS);
                        }
                        else
                        {
                            const float zero = (float)__ddiv_rn(0.0, gsum);
                            for (int k=0; k<ngt_new; k++) dst[k] = k<nmax ? zero : __uint_as_float(MCB_FLOAT_VECTOR_END_BITS);
                            if ( pld==2 )
                            {
                                #pragma unroll
                                for (int k=0; k<NSLOT; k++)
                                    if ( inc_dip & (1u<<k) ) dst[sh.p2.igt[k]] = (float)__ddiv_rn(gv[k], gsum);
                            }
                            else
                            {
                                #pragma unroll
                                for (int x=0; x<MAXSEL; x++)
                                    if ( inc_hap & (1u<<x) ) dst[sh.p2.hap_new[x]] = (float)__ddiv_rn(gv[x*(x+3)/2], gsum);
                            }
                        }
                    }
                }
                }
                if ( !resident )
                {
                    fence_proxy_async();
                    __syncthreads();
                    if ( tid==0 && v+nstage < total_visits ) issue(v+nstage);
                }
            }
            flush_ac();
            if constexpr ( FAST2 ) if ( fast2 )
            {
                #pragma unroll
                for (int off=16; off; off>>=1) { f_alt += __shfl_xor_sync(0xffffffffu, f_alt, off); f_called += __shfl_xor_sync(0xffffffffu, f_called, off); }
                if ( lane==0 && f_called ) { atomicAdd(&sh.ac[0], 2*f_called - f_alt); atomicAdd(&sh.ac[1], f_alt); }
            }
            if ( tflags2 ) atomicOr(&sh.flags, tflags2);
        }
        __syncthreads();

        /* ---- site record: QUAL (mcall.c:1631-1645), AC/AN (1648-1650) ---------------------------------- */
        if ( tid==0 )
        {
            int nAC = 0;
            if ( !sh.ref_gt ) for (int j=1; j<sh.nals_new && j<8; j++) nAC += sh.ac[j];
            int ret = sh.nals_new;
            if ( !sh.ref_gt && !nAC && (a.flag & MCB_CALL_VARONLY) ) ret = 0;      /* mcall.c:1618 */
            float qual;
            if ( nAC ) qual = (float)sh.max_qual;
            else if ( sh.lk_sum != -CUDART_INF ) qual = (float)(-4.343*(sh.lk_sum - logsumexp2_dev(sh.lk_sum, sh.ref_lk)));
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
        __syncthreads();
    }
}

/* ------------------------------------------------------------------------------------------------
 *  division self-test: div_shared(a, b, rcp_shared(b)) must be bit-identical to a/b on the table domain
 * ---------------------------------------------------------------------------------------------- */
__global__ void selftest_div_kernel(const DevTables *tab, int mode, unsigned long long n, unsigned long long seed, unsigned long long *mismatch)
{
    unsigned long long bad = 0;
    const unsigned long long stride = (unsigned long long)gridDim.x*blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x*blockDim.x + threadIdx.x; i<n; i += stride)
    {
        double num[15]; int g;
        if ( mode==0 )      /* exhaustive biallelic: i encodes three PLs */
        {
            g = 3;
            num[0] = tab->pl2p[i & 255]; num[1] = tab->pl2p[(i>>8) & 255]; num[2] = tab->pl2p[(i>>16) & 255];
        }
        else                /* random G = 6, 10 or 15 */
        {
            unsigned long long x = (i + 1)*0x9E3779B97F4A7C15ull ^ seed;
            g = mode;
            for (int j=0; j<g; j++)
            {
                x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;
                /* skew towards small PLs like real data, but cover all 256 values */
                int v = (x & 3) ? (int)((x>>8) & 255) : (int)((x>>8) & 15);
                num[j] = tab->pl2p[v];
            }
        }
        double sum = num[0];
        for (int j=1; j<g; j++) sum = __dadd_rn(sum, num[j]);
        const double r = rcp_shared(sum);
        for (int j=0; j<g; j++)
        {
            double q1 = div_shared(num[j], sum, r), q2 = __ddiv_rn(num[j], sum);
            if ( __double_as_longlong(q1) != __double_as_longlong(q2) ) bad++;
        }
    }
    if ( bad ) atomicAdd(mismatch, bad);
}
/*  float32 screen self-test (mcall_device.cuh): every accepted sample must carry the slot and GQ of the literal FP64 sequence.
 *  mode 20/21: pair sites, all 256^3 PL triples, q1 = 10^(-seed/8), q0 = 1 - q1 (as floats): 20 counts accepted samples that
 *  differ, 21 counts rejected ones.  mode 22/23: triple sites, n random PL sextuples, q1 and q2 from the seed.  */
__global__ void selftest_screen_kernel(const DevTables *tab, int mode, unsigned long long n, unsigned long long seed, unsigned long long *count)
{
    __shared__ ScreenTabs st;
    __shared__ double s_pl2p[256], s_thr[130];
    for (int i=threadIdx.x; i<256; i+=blockDim.x) s_pl2p[i] = tab->pl2p[i];
    for (int i=threadIdx.x; i<130; i+=blockDim.x) s_thr[i] = i<128 ? tab->gq_thr[i] : -1.0;
    screen_tabs_fill(&st, tab, threadIdx.x, blockDim.x);
    __syncthreads();
    const uint32_t plf_s = smem_u32(st.plf), gqw_s = smem_u32(st.gqw), thr_s = smem_u32(s_thr);
    const bool triple = mode >= 22;
    const float q1f = (float)exp10(-(double)(seed & 63)/8.0), q2f = triple ? (float)exp10(-(double)((seed >> 6) & 63)/8.0) : 0.f;
    float q0f = 1.f - q1f - q2f;
    const float qs = q0f + q1f + q2f;
    const double q0 = (double)(q0f/qs), q1 = (double)(q1f/qs), q2 = (double)(q2f/qs);
    bool scr = true;
    float w[6];
    w[0] = screen_weight(q0, q0, 1.0, scr); w[1] = screen_weight(q1, q0, 2.0, scr); w[2] = screen_weight(q1, q1, 1.0, scr);
    if ( triple ) { w[3] = screen_weight(q2, q0, 2.0, scr); w[4] = screen_weight(q2, q1, 2.0, scr); w[5] = screen_weight(q2, q2, 1.0, scr); }
    unsigned long long bad = 0;
    const unsigned long long stride = (unsigned long long)gridDim.x*blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x*blockDim.x + threadIdx.x; i<n; i += stride)
    {
        int ks, gs, ke, ge; bool ok;
        if ( !triple )
        {
            const uint32_t a = i & 255, b = (i>>8) & 255, c = (i>>16) & 255;
            ok = screen2_call(a, b, c, w[0], w[1], w[2], plf_s, gqw_s, ks, gs) && scr;
            const double p0 = s_pl2p[a], p1 = s_pl2p[b], p2 = s_pl2p[c];
            fast2_call(p0, p1, p2, __dadd_rn(__dadd_rn(p0, p1), p2), q0, q1, __dmul_rn(2.0, q1), thr_s, ke, ge);
        }
        else
        {
            unsigned long long x = (i + 1)*0x9E3779B97F4A7C15ull ^ (seed*0xD1B54A32D192ED03ull);
            uint32_t v[6]; double p[6];
            for (int j=0; j<6; j++)
            {
                x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;
                v[j] = (x & 3) ? (uint32_t)((x>>8) & 255) : (uint32_t)((x>>8) & 15);
                p[j] = s_pl2p[v[j]];
            }
            /* the normaliser of a multi-allelic sample also covers genotypes outside the triple */
            double sum = p[0];
            for (int j=1; j<6; j++) sum = __dadd_rn(sum, p[j]);
            sum = __dadd_rn(sum, s_pl2p[(x>>40) & 255]);
            ok = screen3_call(v, w, plf_s, gqw_s, ks, gs) && scr;
            fast3_call(p, sum, q0, q1, q2, __dmul_rn(2.0, q1), __dmul_rn(2.0, q2), thr_s, ke, ge);
        }
        if ( mode & 1 ) bad += !ok;
        else bad += ok && (ks != ke || gs != ge);
    }
    if ( bad ) atomicAdd(count, bad);
}
cudaError_t launch_selftest_div(const DevTables *tab, int mode, unsigned long long n, unsigned long long seed, unsigned long long *mismatch, cudaStream_t st)
{
    if ( mode >= 20 )
    {
        selftest_screen_kernel<<<148*8, 256, 0, st>>>(tab, mode, n, seed, mismatch);
        return cudaGetLastError();
    }
    selftest_div_kernel<<<148*8, 256, 0, st>>>(tab, mode, n, seed, mismatch);
    return cudaGetLastError();
}

/* ------------------------------------------------------------------------------------------------
 *  site classification: one list of site indices per allele count (1..5), one for everything else
 * ---------------------------------------------------------------------------------------------- */
__global__ void classify_sites_kernel(const uint8_t *nals, int nsites, int32_t *lists, int32_t *counts, int list_stride,
                                      int max_nals, int32_t *ret, uint32_t *site_flags, int64_t *pl_off_out)
{
    int i = blockIdx.x*blockDim.x + threadIdx.x;
    if ( i >= nsites ) return;
    int n = nals[i];
    if ( n > max_nals && n <= MCB_MAX_NALS )
    {
        /* more alleles than the stride of the per-site allele arrays (qs, prior_ac, ac, als_map): no kernel may index them */
        ret[i] = 0;
        if ( site_flags ) site_flags[i] = MCB_SITE_UNSUPPORTED;
        if ( pl_off_out ) pl_off_out[i] = -1;
        return;
    }
    int cls = (n>=1 && n<=5) ? n : 0;
    int pos = atomicAdd(&counts[cls], 1);
    lists[(size_t)cls*list_stride + pos] = i;
}

/*  In-call adjudication: the sites the first evaluation flagged MCB_SITE_NEAR_TIE, one list per allele-count class (the
 *  layout of classify_sites_kernel).  Runs after every site kernel of the call; the hot kernels append to no list.  */
__global__ void collect_near_ties_kernel(const uint8_t *nals, int nsites, const uint32_t *site_flags, int32_t *lists, int32_t *counts, int list_stride)
{
    for (int i = blockIdx.x*blockDim.x + threadIdx.x; i < nsites; i += gridDim.x*blockDim.x)
    {
        if ( !(site_flags[i] & MCB_SITE_NEAR_TIE) ) continue;
        const int n = nals[i], cls = (n>=1 && n<=5) ? n : 0;
        const int pos = atomicAdd(&counts[cls], 1);
        lists[(size_t)cls*list_stride + pos] = i;
    }
}

/*  sites the templated kernels do not cover (n_allele 0 or >5): reported as skipped for now  */
__global__ void unsupported_sites_kernel(const int32_t *list, const int32_t *count, int32_t *ret, uint32_t *site_flags, const uint8_t *nals, int64_t *pl_off_out)
{
    int n = *count;
    for (int i = blockIdx.x*blockDim.x + threadIdx.x; i<n; i += gridDim.x*blockDim.x)
    {
        int site = list[i];
        ret[site] = 0;
        if ( site_flags ) site_flags[site] = nals[site] > 32 ? MCB_SITE_TOO_MANY_ALS : MCB_SITE_UNSUPPORTED;
        if ( pl_off_out ) pl_off_out[site] = -1;
    }
}

template<int NALS, bool PLOIDY, int BLOCK, typename PT, bool GPOUT>
static cudaError_t launch_one(const KArgs &a, int grid, size_t ring_bytes, cudaStream_t st)
{
    auto kern = mcall_site_kernel<NALS,PLOIDY,BLOCK,PT,GPOUT>;
    const size_t smem = align128(sizeof(Shared<NALS,BLOCK>)) + ring_bytes;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if ( e!=cudaSuccess ) return e;
    kern<<<grid, BLOCK, smem, st>>>(a);
    return cudaGetLastError();
}
template<int NALS, bool PLOIDY, int BLOCK, typename PT, bool GPOUT>
static cudaError_t occ_one(size_t ring_bytes, int *nb)
{
    auto kern = mcall_site_kernel<NALS,PLOIDY,BLOCK,PT,GPOUT>;
    const size_t smem = align128(sizeof(Shared<NALS,BLOCK>)) + ring_bytes;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if ( e!=cudaSuccess ) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(nb, kern, BLOCK, smem);
}
/*  one dispatcher for launch (nb==NULL) and occupancy query (nb!=NULL)  */
template<int NALS>
static cudaError_t dispatch(bool ploidy, bool gp, int block, int pl_es, const KArgs *a, int grid, size_t ring_bytes, cudaStream_t st, int *nb)
{
#define MCB_CASE(P,B,T,GP) return nb ? occ_one<NALS,P,B,T,GP>(ring_bytes, nb) : launch_one<NALS,P,B,T,GP>(*a, grid, ring_bytes, st)
    if ( gp )               /* FORMAT/GP: one instance per shape and element type (any ploidy, 128-thread CTAs) */
    {
        if ( pl_es==4 ) MCB_CASE(true,128,int32_t,true);
        if ( pl_es==2 ) MCB_CASE(true,128,int16_t,true);
        return cudaErrorInvalidValue;
    }
    if ( pl_es==4 )
    {
        if ( block==32 )  { if ( ploidy ) MCB_CASE(true,32,int32_t,false);  MCB_CASE(false,32,int32_t,false); }
        if ( block==64 )  { if ( ploidy ) MCB_CASE(true,64,int32_t,false);  MCB_CASE(false,64,int32_t,false); }
        if ( block==128 ) { if ( ploidy ) MCB_CASE(true,128,int32_t,false); MCB_CASE(false,128,int32_t,false); }
        if ( block==256 ) { if ( ploidy ) MCB_CASE(true,256,int32_t,false); MCB_CASE(false,256,int32_t,false); }
    }
    if ( pl_es==2 )         /* BCF int16 typed vectors: 128-thread CTAs only */
    {
        if ( ploidy ) MCB_CASE(true,128,int16_t,false); MCB_CASE(false,128,int16_t,false);
    }
#undef MCB_CASE
    return cudaErrorInvalidValue;
}
static cudaError_t dispatch_nals(int nals, bool ploidy, bool gp, int block, int pl_es, const KArgs *a, int grid, size_t ring_bytes, cudaStream_t st, int *nb)
{
    switch ( nals )
    {
        case 1: return dispatch<1>(ploidy, gp, block, pl_es, a, grid, ring_bytes, st, nb);
        case 2: return dispatch<2>(ploidy, gp, block, pl_es, a, grid, ring_bytes, st, nb);
        case 3: return dispatch<3>(ploidy, gp, block, pl_es, a, grid, ring_bytes, st, nb);
        case 4: return dispatch<4>(ploidy, gp, block, pl_es, a, grid, ring_bytes, st, nb);
        case 5: return dispatch<5>(ploidy, gp, block, pl_es, a, grid, ring_bytes, st, nb);
    }
    return cudaErrorInvalidValue;
}
cudaError_t launch_site_kernel(int nals, bool ploidy, bool gp, int block, int pl_es, const KArgs &a, int grid, size_t ring_bytes, cudaStream_t st)
{
    return dispatch_nals(nals, ploidy, gp, gp ? 128 : block, pl_es, &a, grid, ring_bytes, st, nullptr);
}
cudaError_t site_kernel_occupancy(int nals, bool ploidy, bool gp, int block, int pl_es, size_t ring_bytes, int *nb)
{
    return dispatch_nals(nals, ploidy, gp, gp ? 128 : block, pl_es, nullptr, 0, ring_bytes, nullptr, nb);
}

cudaError_t launch_classify(const uint8_t *nals, int nsites, int32_t *lists, int32_t *counts, int list_stride, int max_nals, int32_t *ret, uint32_t *site_flags, int64_t *pl_off_out, cudaStream_t st)
{
    if ( nsites<=0 ) return cudaSuccess;
    classify_sites_kernel<<<(nsites+255)/256, 256, 0, st>>>(nals, nsites, lists, counts, list_stride, max_nals, ret, site_flags, pl_off_out);
    return cudaGetLastError();
}
cudaError_t launch_collect_near_ties(const uint8_t *nals, int nsites, const uint32_t *site_flags, int32_t *lists, int32_t *counts, int list_stride, cudaStream_t st)
{
    if ( nsites<=0 ) return cudaSuccess;
    collect_near_ties_kernel<<<(nsites+255)/256 < 1024 ? (nsites+255)/256 : 1024, 256, 0, st>>>(nals, nsites, site_flags, lists, counts, list_stride);
    return cudaGetLastError();
}
cudaError_t launch_unsupported(const int32_t *list, const int32_t *count, int32_t *ret, uint32_t *site_flags, const uint8_t *nals, int64_t *pl_off_out, cudaStream_t st)
{
    unsupported_sites_kernel<<<64, 256, 0, st>>>(list, count, ret, site_flags, nals, pl_off_out);
    return cudaGetLastError();
}

}   // namespace mcb
