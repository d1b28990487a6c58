/*  mcall_groups.cu -- site kernel for grouped calling (`call -m -G`, call->nsmpl_grp > 1; mcall.c:250-349, 1466-1504,
 *  1546-1561, 1608-1614).  Correctness-first: one CTA per site, 1..5 alleles.
 *
 *    phase A  one WARP per sample group, lane k <-> allele set k (<= 25 sets): the group's quality sums from
 *             FORMAT/AD in float32, sequential in group order exactly like mcall.c:1478-1503 (lane a <-> allele a);
 *             then the group's samples are walked sequentially, every lane accumulating its own set as an
 *             exponent-tracked product (same numerics as the pooled kernel); the set epilogue is the pooled one.
 *             KArgs.exact_phase1 (options exact_phase1 / adjudicate): every group takes the sample-parallel path and lane k
 *             then walks the group's member list once more with the literal sums of logs (exact_set_lk, mcall_device.cuh).
 *    phase B  thread 0 combines the groups: als_new = OR of the groups' sets | REF, the QUAL candidate of the group
 *             with the largest QUAL (mcall.c:1546-1575), trimming maps (mcall.c:547-570).
 *    phase C  one THREAD per sample: literal mcall_call_genotypes() with the sample's own group record
 *             (mcall.c:745-886), GQ/GP, PL trimming, AC.
 *
 *  PLs are read from global memory directly (L2 serves the second read); the per-group records live in a global
 *  scratch area owned by the CTA.
 */
#include "mcall_device.cuh"

namespace mcb {

#ifndef GBLOCK
#define GBLOCK 160          /* five warps: the five super-population groups of a 1000G-shaped call take one round of phase A */
#endif
#define GNW    (GBLOCK/32)
/*  resident CTAs per SM the instances are compiled for (register cap 65536 / (GBLOCK * n)): up to three alleles 64 registers,
 *  four alleles 96, five alleles 200 (no spills; a batch holds few such sites).  Sweeps: profiles/r02_groups_cta_regcap_sweep.log  */
#ifndef GMINB
#define GMINB 2
#endif
#ifndef GMINB3
#define GMINB3 6
#endif
#ifndef GMINB4
#define GMINB4 4
#endif
#ifndef BIG_GROUP
#define BIG_GROUP 64        /* groups of at least this many samples are reduced by the whole CTA, sample-parallel */
#endif

struct GroupRec
{
    double q[5];            /* (double)(float)qsum, normalised (mcall.c:1530-1535) */
    double qual, ref_lk, lk_sum;
    uint32_t als;           /* grp->als */
    int nals, has_max, pad;
};

#define GS_NODATA  (-2.0)
#define GS_GENERIC (-1.0)
__host__ __device__ inline size_t groups_rec_bytes(int ngroups) { return ((size_t)ngroups*sizeof(GroupRec) + 15) & ~(size_t)15; }
__host__ __device__ inline size_t groups_cta_bytes(int ngroups, int nsmpl) { return groups_rec_bytes(ngroups) + (((size_t)nsmpl*sizeof(double) + 15) & ~(size_t)15); }

struct GSite                /* site decision record, shared memory */
{
    double max_qual, lk_sum, ref_lk;
    uint32_t als_new, flags;
    int nals_new, is_variant, ret_early, pl_dropped, ref_gt;
    long long out_off;
    int als_map[5], pl_map[15], ac[8];
};

/*  set_pdg's missing-value fill (mcall.c:495-527) on a thread-local PL row  */
__device__ __noinline__ int fix_missing_local(int *pl, int nals, int unseen)
{
    const int G = nals*(nals+1)/2;
    int j;
    for (j=0; j<G; j++)
    {
        if ( pl[j]==I32_VEC_END ) return 0;
        if ( pl[j]==I32_MISSING ) break;
    }
    if ( j==0 || j==G ) return 0;
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
            else if ( pl[j] < 0 ) return 0;
            j++;
        }
    return 1;
}

__device__ __forceinline__ double pl_to_p_dev(const double *s_pl2p, const DevTables *tab, int v, uint32_t *flags)
{
    if ( (unsigned)v < 256u ) return s_pl2p[v];
    if ( v > 2500 ) *flags |= MCB_SITE_PL_RANGE;
    return (unsigned)v < (unsigned)MCB_PL2P_BIG ? tab->pl2p_big[v] : 0.0;
}

/*  GQ from the largest and the sum of the genotype posteriors (mcall.c:843-878): phred of 1 - max/sum through the
 *  threshold table, 127 when the ratio is not a number  */
__device__ __forceinline__ int groups_gq(double gmax, double gsum, const double *s_thr)
{
    const double xx = __dadd_rn(1.0, -__ddiv_rn(gmax, gsum));
    if ( !(xx==xx) ) return 127;
    int k = __float2int_rz(-3.0102999f*lg2_approx((float)xx));
    k = max(0, min(127, k));
    if ( xx <= s_thr[k+1] ) { k++; while ( xx <= s_thr[k+1] ) k++; }
    else while ( xx > s_thr[k] ) k--;
    return k;
}

template<int NALS>
__global__ void __launch_bounds__(GBLOCK, (NALS<=3 ? GMINB3 : (NALS==4 ? GMINB4 : GMINB))) mcall_groups_kernel(const KArgs a, GroupRec *scratch)
{
    using S = Shape<NALS>;
    constexpr int G = S::G, NPAIR = S::NPAIR, NSUB = S::NSUB;
    constexpr double LN2 = 0.693147180559945309417232121458;

    __shared__ double s_pl2p[256];
    __shared__ double s_thr[130];
    __shared__ double s_p[GNW][16];
    __shared__ int    s_chunk[GNW][32][16];     /* PL rows of 32 samples of the group, fetched together: one global round trip per 32 samples */
    __shared__ float  s_adc[GNW][32][5];        /* per-sample AD fractions of the chunk */
    __shared__ unsigned char s_pld[GNW][32];
    __shared__ int    s_sid[GNW][32];
    /* block-wide path for big groups (>= BIG_GROUP samples): same data flow as phase 1 of the pooled kernel */
    constexpr int NTRI = S::NTRI, NACC = S::NACC;
    __shared__ float  s_qf[GNW][NALS];
    __shared__ double s_cfp[GNW][(NPAIR ? NPAIR : 1)*5], s_cft[GNW][(NTRI ? NTRI : 1)*9];
    __shared__ uint32_t s_live[GNW];
    __shared__ double s_redM[GNW][NACC];
    __shared__ int    s_redE[GNW][NACC];
    __shared__ long long s_redP[GNW][NALS];
    __shared__ int    s_redC[GNW][2];
    __shared__ GSite  st;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nsmpl = a.nsmpl, ngrp = a.ngroups;
    char *cta_scratch = reinterpret_cast<char*>(scratch) + (size_t)blockIdx.x*groups_cta_bytes(ngrp, nsmpl);
    GroupRec *grec = reinterpret_cast<GroupRec*>(cta_scratch);
    /* per-sample normaliser sum_j p[j] written by phase A and read by phase C (the site's samples are partitioned by the
       groups, mcall_abi.cu checks it): > 0 the sum, GS_NODATA a row of zeros, GS_GENERIC a row with missing values */
    double *ssum = reinterpret_cast<double*>(cta_scratch + groups_rec_bytes(ngrp));

    for (int i=tid; i<256; i+=GBLOCK) s_pl2p[i] = a.tab->pl2p[i];
    for (int i=tid; i<130; i+=GBLOCK) s_thr[i] = i<128 ? a.tab->gq_thr[i] : -1.0;
    __syncthreads();

    const int nsites = *a.site_count;
    for (int isite = blockIdx.x; isite < nsites; isite += gridDim.x)
    {
        const int site = a.site_list[isite];
        const int64_t site_off = a.pl_off[site];
        const int32_t *site_pl = reinterpret_cast<const int32_t*>(a.pl) + site_off;     /* int32 only in the grouped kernel */
        const int unseen = a.unseen ? a.unseen[site] : 0;
        int pid = a.ploidy_id ? a.ploidy_id[site] : 0;
        if ( pid >= a.nploidy ) pid = 0;
        const uint8_t *ploidy = a.ploidy_tab + (size_t)pid*nsmpl;
        const int nad = a.nad ? a.nad[site] : 0;
        const int32_t *site_ad = a.ad ? a.ad + a.ad_off[site] : nullptr;
        if ( tid==0 ) { st.flags = (site_ad && nad>0) ? 0 : MCB_SITE_NO_QS; for (int j=0; j<8; j++) st.ac[j] = 0; }
        __syncthreads();

        /* =========================== phase A: one warp per group =============================== */
        for (int g=warp; g<ngrp; g+=GNW)
        {
            const int beg = a.grp_off[g], end = a.grp_off[g+1];
            if ( end-beg >= BIG_GROUP || a.exact_phase1 ) continue;     /* handled below (the literal phase 1 always is) */
            /* ---- quality sums from FORMAT/AD: float32, sequential over the group's samples (mcall.c:1484-1501) */
            float qa = 0;
            if ( site_ad )
                for (int base=beg; base<end; base+=32)
                {
                    /* every lane: the fractions AD[a]/sum of ONE sample (independent per sample) ... */
                    const int i = base + lane;
                    float frac[5] = {0,0,0,0,0};
                    if ( i<end )
                    {
                        const int32_t *ptr = site_ad + (size_t)a.grp_smpl[i]*nad;
                        int adv[5]; float sum = 0; int e = nad<5 ? nad : 5;
                        #pragma unroll
                        for (int j=0; j<5; j++) adv[j] = j<nad ? ptr[j] : I32_VEC_END;
                        #pragma unroll
                        for (int j=0; j<5; j++)
                        {
                            if ( j>=e ) break;
                            if ( adv[j]==I32_VEC_END ) { e = j; break; }
                            if ( adv[j]!=I32_MISSING ) sum = __fadd_rn(sum, (float)adv[j]);
                        }
                        if ( sum!=0 )
                        {
                            #pragma unroll
                            for (int j=0; j<5; j++) if ( j<e && adv[j]!=I32_MISSING ) frac[j] = __fdiv_rn((float)adv[j], sum);
                        }
                    }
                    #pragma unroll
                    for (int j=0; j<5; j++) s_adc[warp][lane][j] = frac[j];
                    __syncwarp();
                    /* ... lane a: the float32 running sum in group order (adding +0 for non-contributing samples is exact) */
                    if ( lane<NALS )
                    {
                        const int n = min(32, end-base);
                        for (int k=0; k<n; k++) qa = __fadd_rn(qa, s_adc[warp][k][lane]);
                    }
                    __syncwarp();
                }
            float qf[NALS];
            #pragma unroll
            for (int j=0; j<NALS; j++) qf[j] = __shfl_sync(0xffffffffu, qa, j);
            /* ---- -F prior (mcall.c:1507-1527) with this group's sample count, then normalisation (1530-1535) */
            if ( a.use_prior && a.prior_an && a.prior_ac )
            {
                const int an = a.prior_an[site];
                if ( an!=I32_MISSING && an>0 )
                {
                    const int32_t *pac = a.prior_ac + (size_t)site*a.max_nals;
                    const double den = __dadd_rn((double)(uint32_t)(end-beg), __dmul_rn(0.5,(double)an));
                    int ac0 = an;
                    for (int j=0; j<NALS-1; j++)
                    {
                        if ( pac[j]==I32_VEC_END ) break;
                        if ( pac[j]==I32_MISSING ) continue;
                        ac0 -= pac[j];
                        qf[j+1] = (float)__ddiv_rn(__dadd_rn((double)qf[j+1], __dmul_rn(0.5,(double)pac[j])), den);
                    }
                    if ( ac0<0 && lane==0 ) atomicOr(&st.flags, MCB_SITE_BAD_PRIOR);
                    qf[0] = (float)__ddiv_rn(__dadd_rn((double)qf[0], __dmul_rn(0.5,(double)ac0)), den);
                }
            }
            {
                float qs = 0;
                #pragma unroll
                for (int j=0; j<NALS; j++) qs = __fadd_rn(qs, qf[j]);
                if ( qs!=0 )
                {
                    #pragma unroll
                    for (int j=0; j<NALS; j++) qf[j] = __fdiv_rn(qf[j], qs);
                }
            }
            /* ---- lane k: its allele set, in the reference's enumeration order (mcall.c:601-698) */
            int sa = 0, sb = -1, sc = -1;       /* alleles of the set, sa > sb > sc */
            bool live = false;
            if ( lane < NALS ) { sa = lane; live = true; }
            else if ( lane < NALS+NPAIR )
            {
                int k = lane-NALS; sa = 1; while ( sa*(sa+1)/2 <= k ) sa++;
                sb = k - sa*(sa-1)/2;
            }
            else if ( lane < NSUB )
            {
                int k = lane-NALS-NPAIR; sa = 2; while ( (sa+1)*sa*(sa-1)/6 <= k ) sa++;
                int r = k - sa*(sa-1)*(sa-2)/6; sb = 1; while ( sb*(sb+1)/2 <= r ) sb++;
                sc = r - sb*(sb-1)/2;
            }
            auto QF = [&](int j) -> float { float v = 0; for (int t=0; t<NALS; t++) if ( t==j ) v = qf[t]; return v; };
            /* terms: up to 3 homozygous (diploid coefficient cd, haploid ch) then up to 3 heterozygous (cd only) */
            int tix[6] = {0,0,0,0,0,0}; double cd[6] = {0,0,0,0,0,0}, ch[3] = {0,0,0};
            uint32_t mask = 0; int nonref = 0;
            if ( lane < NALS ) { tix[0] = hom_idx(sa); cd[0] = 1; ch[0] = 1; mask = 1u<<sa; nonref = sa!=0; }
            else if ( lane < NALS+NPAIR )
            {
                const float fqa = QF(sa), fqb = QF(sb);
                mask = 1u<<sa | 1u<<sb; nonref = (sa!=0) + (sb!=0);
                if ( fqa!=0 && fqb!=0 )
                {
                    live = true;
                    const float den = __fadd_rn(fqa,fqb);
                    const double fa = (double)__fdiv_rn(fqa,den), fb = (double)__fdiv_rn(fqb,den);
                    tix[0] = hom_idx(sa); tix[1] = hom_idx(sb); tix[3] = gt_idx(sa,sb);
                    cd[0] = __dmul_rn(fa,fa); cd[1] = __dmul_rn(fb,fb); cd[3] = __dmul_rn(__dmul_rn(2.0,fa),fb);
                    ch[0] = fa; ch[1] = fb;
                }
            }
            else if ( lane < NSUB )
            {
                const float fqa = QF(sa), fqb = QF(sb), fqc = QF(sc);
                mask = 1u<<sa | 1u<<sb | 1u<<sc; nonref = (sa!=0) + (sb!=0) + (sc!=0);
                if ( fqa!=0 && fqb!=0 && fqc!=0 )
                {
                    live = true;
                    const float den = __fadd_rn(__fadd_rn(fqa,fqb),fqc);
                    const double fa = (double)__fdiv_rn(fqa,den), fb = (double)__fdiv_rn(fqb,den), fc = (double)__fdiv_rn(fqc,den);
                    tix[0] = hom_idx(sa); tix[1] = hom_idx(sb); tix[2] = hom_idx(sc);
                    tix[3] = gt_idx(sa,sb); tix[4] = gt_idx(sa,sc); tix[5] = gt_idx(sb,sc);
                    cd[0] = __dmul_rn(fa,fa); cd[1] = __dmul_rn(fb,fb); cd[2] = __dmul_rn(fc,fc);
                    cd[3] = __dmul_rn(__dmul_rn(2.0,fa),fb); cd[4] = __dmul_rn(__dmul_rn(2.0,fa),fc); cd[5] = __dmul_rn(__dmul_rn(2.0,fb),fc);
                    ch[0] = fa; ch[1] = fb; ch[2] = fc;
                }
            }
            const bool single = lane < NALS;

            /* ---- walk the group's samples; lane k accumulates prod val_s and prod sum_s of ITS set */
            double M = 1, MN = 1; int E = 0, EN = 0, cnt = 0, since = 0;
            uint32_t wflags = 0;
            for (int base=beg; base<end; base+=32)
            {
                {
                    const int i = base + lane;
                    if ( i<end )
                    {
                        const int s = a.grp_smpl[i];
                        #pragma unroll
                        for (int j=0; j<G; j++) s_chunk[warp][lane][j] = site_pl[(size_t)s*G + j];
                        s_pld[warp][lane] = ploidy[s];
                        s_sid[warp][lane] = s;
                    }
                }
                __syncwarp();
                const int nchunk = min(32, end-base);
                for (int k=0; k<nchunk; k++)
                {
                    int *row = s_chunk[warp][k];
                    int v = lane<G ? row[lane] : 0;
                    bool data = true;
                    const bool neg = __any_sync(0xffffffffu, v<0);
                    if ( neg )
                    {
                        int ok = 0;
                        if ( lane==0 ) ok = fix_missing_local(row, NALS, unseen);
                        ok = __shfl_sync(0xffffffffu, ok, 0);
                        __syncwarp();
                        if ( lane<G ) v = row[lane];
                        data = ok && !__any_sync(0xffffffffu, v<0);
                    }
                    if ( !__any_sync(0xffffffffu, v!=0) ) data = false;      /* PL=0,..,0: no data (mcall.c:529-537) */
                    if ( lane==0 && (neg || !data) ) ssum[s_sid[warp][k]] = neg ? GS_GENERIC : GS_NODATA;
                    if ( !data ) continue;
                    if ( lane<G ) s_p[warp][lane] = pl_to_p_dev(s_pl2p, a.tab, v, &wflags);
                    __syncwarp();
                    double sum = s_p[warp][0];
                    #pragma unroll
                    for (int j=1; j<G; j++) sum = __dadd_rn(sum, s_p[warp][j]);
                    if ( lane==0 && !neg ) ssum[s_sid[warp][k]] = sum > 0 ? sum : GS_GENERIC;
                    const int pld = s_pld[warp][k];
                    if ( live && lane<NSUB )
                    {
                        double val = 0; bool use = false;
                        if ( single ) { val = s_p[warp][tix[0]]; use = true; }     /* every sample, also ploidy 0 (mcall.c:607-611) */
                        else if ( pld==2 )
                        {
                            val = cd[0]*s_p[warp][tix[0]];
                            val = fma(cd[1], s_p[warp][tix[1]], val);
                            if ( sc>=0 ) val = fma(cd[2], s_p[warp][tix[2]], val);
                            val = fma(cd[3], s_p[warp][tix[3]], val);
                            if ( sc>=0 ) { val = fma(cd[4], s_p[warp][tix[4]], val); val = fma(cd[5], s_p[warp][tix[5]], val); }
                            use = true;
                        }
                        else if ( pld==1 )
                        {
                            val = ch[0]*s_p[warp][tix[0]];
                            val = fma(ch[1], s_p[warp][tix[1]], val);
                            if ( sc>=0 ) val = fma(ch[2], s_p[warp][tix[2]], val);
                            use = true;
                        }
                        if ( use && val!=0 ) { acc_mul(M, E, val); acc_mul(MN, EN, sum); cnt++; }
                    }
                    if ( ++since >= 256 ) { acc_renorm(M, E); acc_renorm(MN, EN); since = 0; }
                    __syncwarp();
                }
                __syncwarp();
            }
            /* ---- set totals and the group's best set (same epilogue as the pooled kernel) */
            double lk = 0;
            const bool cand = live && lane<NSUB && cnt>0;
            if ( cand ) lk = (log(M) + (double)(E - 1023*cnt)*LN2) - (log(MN) + (double)(EN - 1023*cnt)*LN2);
            if ( lane<NSUB ) for (int j=0; j<nonref; j++) lk += a.theta;
            const bool in_sum = cand && !(single && sa==0);
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
            double mx = in_sum ? lk : -CUDART_INF;
            #pragma unroll
            for (int off=16; off; off>>=1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, off));
            double term = in_sum ? exp(lk - mx) : 0.0;
            #pragma unroll
            for (int off=16; off; off>>=1) term += __shfl_xor_sync(0xffffffffu, term, off);
            #pragma unroll
            for (int off=16; off; off>>=1) wflags |= __shfl_xor_sync(0xffffffffu, wflags, off);
            const double g_lk_sum = mx > -CUDART_INF ? mx + log(term) : -CUDART_INF;
            const double g_ref_lk = __shfl_sync(0xffffffffu, lk, 0);
            const uint32_t g_als = __shfl_sync(0xffffffffu, mask, best_lane & 31);
            if ( lane==0 )
            {
                const bool any = best_lane < 64;
                GroupRec &r = grec[g];
                #pragma unroll
                for (int j=0; j<NALS; j++) r.q[j] = (double)qf[j];
                r.als = any ? g_als : 0;
                int n = 0;
                for (int j=0; j<NALS; j++) n += (r.als>>j)&1u;
                r.nals = n; r.has_max = any;
                r.ref_lk = g_ref_lk; r.lk_sum = g_lk_sum;
                r.qual = any ? -4.343*(g_ref_lk - logsumexp2_dev(g_lk_sum, g_ref_lk)) : -CUDART_INF;
                uint32_t f = wflags;
                if ( any && best - second < a.tie_eps ) f |= MCB_SITE_NEAR_TIE;
                if ( f ) atomicOr(&st.flags, f);
            }
        }
        __threadfence_block();
        __syncthreads();
        /* =========================== phase A, big groups: one WARP per group, one lane per SAMPLE =======
         *  Every warp takes its own groups from start to end -- quality sums, coefficients, the sample-parallel products,
         *  the set comparison -- with warp-level synchronisation only.  (The first version ran the groups one after the
         *  other on the whole CTA: warp 0's sequential AD sums and set comparisons were 40 % of all instructions and the
         *  other three warps spent more than half of their time at the barriers behind them, profiles/r02_ncu_groups_*.)  */
        for (int g=0, big_i=0; g<ngrp; g++)
        {
            const int beg = a.grp_off[g], end = a.grp_off[g+1], ng = end-beg;
            if ( ng < BIG_GROUP && !a.exact_phase1 ) continue;
            if ( (big_i++ % GNW) != warp ) continue;
            {
                /* quality sums (float32, group order), -F prior, normalisation: as in the warp path above */
                float qa = 0;
                if ( site_ad )
                    for (int base=beg; base<end; base+=32)
                    {
                        const int i = base + lane;
                        float frac[5] = {0,0,0,0,0};
                        if ( i<end )
                        {
                            const int32_t *ptr = site_ad + (size_t)a.grp_smpl[i]*nad;
                            int adv[5]; float sum = 0; int e = nad<5 ? nad : 5;
                            #pragma unroll
                            for (int j=0; j<5; j++) adv[j] = j<nad ? ptr[j] : I32_VEC_END;
                            #pragma unroll
                            for (int j=0; j<5; j++)
                            {
                                if ( j>=e ) break;
                                if ( adv[j]==I32_VEC_END ) { e = j; break; }
                                if ( adv[j]!=I32_MISSING ) sum = __fadd_rn(sum, (float)adv[j]);
                            }
                            if ( sum!=0 )
                            {
                                #pragma unroll
                                for (int j=0; j<5; j++) if ( j<e && adv[j]!=I32_MISSING ) frac[j] = __fdiv_rn((float)adv[j], sum);
                            }
                        }
                        #pragma unroll
                        for (int j=0; j<5; j++) s_adc[warp][lane][j] = frac[j];
                        __syncwarp();
                        if ( lane<NALS )
                        {
                            const int n = min(32, end-base);
                            for (int k=0; k<n; k++) qa = __fadd_rn(qa, s_adc[warp][k][lane]);
                        }
                        __syncwarp();
                    }
                float qf[NALS];
                #pragma unroll
                for (int j=0; j<NALS; j++) qf[j] = __shfl_sync(0xffffffffu, qa, j);
                if ( a.use_prior && a.prior_an && a.prior_ac )
                {
                    const int an = a.prior_an[site];
                    if ( an!=I32_MISSING && an>0 )
                    {
                        const int32_t *pac = a.prior_ac + (size_t)site*a.max_nals;
                        const double den = __dadd_rn((double)(uint32_t)ng, __dmul_rn(0.5,(double)an));
                        int ac0 = an;
                        for (int j=0; j<NALS-1; j++)
                        {
                            if ( pac[j]==I32_VEC_END ) break;
                            if ( pac[j]==I32_MISSING ) continue;
                            ac0 -= pac[j];
                            qf[j+1] = (float)__ddiv_rn(__dadd_rn((double)qf[j+1], __dmul_rn(0.5,(double)pac[j])), den);
                        }
                        if ( ac0<0 && lane==0 ) atomicOr(&st.flags, MCB_SITE_BAD_PRIOR);
                        qf[0] = (float)__ddiv_rn(__dadd_rn((double)qf[0], __dmul_rn(0.5,(double)ac0)), den);
                    }
                }
                {
                    float qs = 0;
                    #pragma unroll
                    for (int j=0; j<NALS; j++) qs = __fadd_rn(qs, qf[j]);
                    if ( qs!=0 )
                    {
                        #pragma unroll
                        for (int j=0; j<NALS; j++) qf[j] = __fdiv_rn(qf[j], qs);
                    }
                }
                if ( lane==0 )
                {
                    #pragma unroll
                    for (int j=0; j<NALS; j++) { s_qf[warp][j] = qf[j]; grec[g].q[j] = (double)qf[j]; }
                }
                __syncwarp();
                /* allele-set coefficients, one lane per set (mcall.c:629-633, 671-677) */
                uint32_t live = 0;
                if ( lane < NPAIR )
                {
                    int aa = 1; while ( aa*(aa+1)/2 <= lane ) aa++;
                    int bb = lane - aa*(aa-1)/2;
                    float fqa = s_qf[warp][aa], fqb = s_qf[warp][bb];
                    double *cf = s_cfp[warp] + lane*5;
                    if ( fqa!=0 && fqb!=0 )
                    {
                        float den = __fadd_rn(fqa,fqb);
                        double fa = (double)__fdiv_rn(fqa,den), fb = (double)__fdiv_rn(fqb,den);
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
                    float fqa = s_qf[warp][aa], fqb = s_qf[warp][bb], fqc = s_qf[warp][cc];
                    double *cf = s_cft[warp] + k*9;
                    if ( fqa!=0 && fqb!=0 && fqc!=0 )
                    {
                        float den = __fadd_rn(__fadd_rn(fqa,fqb),fqc);
                        double fa = (double)__fdiv_rn(fqa,den), fb = (double)__fdiv_rn(fqb,den), fc = (double)__fdiv_rn(fqc,den);
                        cf[0] = __dmul_rn(fa,fa); cf[1] = __dmul_rn(fb,fb); cf[2] = __dmul_rn(fc,fc);
                        cf[3] = __dmul_rn(__dmul_rn(2.0,fa),fb); cf[4] = __dmul_rn(__dmul_rn(2.0,fa),fc); cf[5] = __dmul_rn(__dmul_rn(2.0,fb),fc);
                        cf[6] = fa; cf[7] = fb; cf[8] = fc;
                        live = 1u<<lane;
                    }
                    else { for (int j=0; j<9; j++) cf[j] = 0; }
                }
                #pragma unroll
                for (int off=16; off; off>>=1) live |= __shfl_xor_sync(0xffffffffu, live, off);
                if ( lane==0 ) s_live[warp] = live;
            }
            __syncwarp();
            const uint32_t live = s_live[warp];
            /* ---- sample-parallel accumulation (pooled kernel, phase 1) over the group's sample list */
            double accM[NACC]; int accE[NACC]; long long plsum[NALS];
            int cnt_all = 0, cnt_called = 0, since = 0;
            uint32_t bflags = 0;
            #pragma unroll
            for (int k=0; k<NACC; k++) { accM[k] = 1.0; accE[k] = 0; }
            #pragma unroll
            for (int k=0; k<NALS; k++) plsum[k] = 0;
            for (int i=lane; i<ng; i+=32)
            {
                const int smp = a.grp_smpl[beg+i];
                int pl[G]; double p[G];
                int orv = 0;
                #pragma unroll
                for (int j=0; j<G; j++) { pl[j] = site_pl[(size_t)smp*G + j]; orv |= pl[j]; }
                const bool neg = orv<0;
                if ( neg )
                {
                    ssum[smp] = GS_GENERIC;
                    int tmp[16];
                    #pragma unroll
                    for (int j=0; j<G; j++) tmp[j] = pl[j];
                    const int ok = fix_missing_local(tmp, NALS, unseen);
                    orv = 0;
                    #pragma unroll
                    for (int j=0; j<G; j++) { if ( ok ) pl[j] = tmp[j]; orv |= pl[j]; }
                    if ( !ok || orv<0 ) continue;
                }
                if ( orv==0 ) { if ( !neg ) ssum[smp] = GS_NODATA; continue; }
                #pragma unroll
                for (int j=0; j<G; j++) p[j] = pl_to_p_dev(s_pl2p, a.tab, pl[j], &bflags);
                double sum = p[0];
                #pragma unroll
                for (int j=1; j<G; j++) sum = __dadd_rn(sum, p[j]);
                if ( !neg ) ssum[smp] = sum > 0 ? sum : GS_GENERIC;
                const int pld = ploidy[smp];
                #pragma unroll
                for (int k=0; k<NALS; k++) plsum[k] += pl[hom_idx(k)];
                cnt_all++;
                acc_mul(accM[NACC-2], accE[NACC-2], sum);
                if ( pld==0 ) continue;
                cnt_called++;
                acc_mul(accM[NACC-1], accE[NACC-1], sum);
                if ( pld==2 )
                {
                    #pragma unroll
                    for (int x=1; x<NALS; x++)
                        #pragma unroll
                        for (int y=0; y<x; y++)
                        {
                            const int k = pair_idx(x,y);
                            if ( live & (1u<<k) )
                            {
                                const double *cf = s_cfp[warp] + k*5;
                                double val = fma(cf[2], p[gt_idx(x,y)], fma(cf[1], p[hom_idx(y)], cf[0]*p[hom_idx(x)]));
                                acc_mul(accM[k], accE[k], val);
                            }
                        }
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
                                    const double *cf = s_cft[warp] + k*9;
                                    double val = fma(cf[5], p[gt_idx(y,z)], fma(cf[4], p[gt_idx(x,z)], fma(cf[3], p[gt_idx(x,y)],
                                                 fma(cf[2], p[hom_idx(z)], fma(cf[1], p[hom_idx(y)], cf[0]*p[hom_idx(x)])))));
                                    acc_mul(accM[NPAIR+k], accE[NPAIR+k], val);
                                }
                            }
                }
                else
                {
                    #pragma unroll
                    for (int x=1; x<NALS; x++)
                        #pragma unroll
                        for (int y=0; y<x; y++)
                        {
                            const int k = pair_idx(x,y);
                            if ( live & (1u<<k) )
                            {
                                const double *cf = s_cfp[warp] + k*5;
                                double val = fma(cf[4], p[hom_idx(y)], cf[3]*p[hom_idx(x)]);
                                acc_mul(accM[k], accE[k], val);
                            }
                        }
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
                                    const double *cf = s_cft[warp] + k*9;
                                    double val = fma(cf[8], p[hom_idx(z)], fma(cf[7], p[hom_idx(y)], cf[6]*p[hom_idx(x)]));
                                    acc_mul(accM[NPAIR+k], accE[NPAIR+k], val);
                                }
                            }
                }
                if ( ++since >= 256 )
                {
                    #pragma unroll
                    for (int k=0; k<NACC; k++) acc_renorm(accM[k], accE[k]);
                    since = 0;
                }
            }
            /* ---- CTA reduction (mantissa multiply, exponent add) */
            #pragma unroll
            for (int k=0; k<NACC; k++)
            {
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
                bflags     |= __shfl_xor_sync(0xffffffffu, bflags, off);
            }
            if ( lane==0 )
            {
                #pragma unroll
                for (int k=0; k<NACC; k++) { s_redM[warp][k] = accM[k]; s_redE[warp][k] = accE[k]; }
                #pragma unroll
                for (int k=0; k<NALS; k++) s_redP[warp][k] = plsum[k];
                s_redC[warp][0] = cnt_all; s_redC[warp][1] = cnt_called;
                if ( bflags ) atomicOr(&st.flags, bflags);
            }
            __syncwarp();
            /* ---- set totals and the group's best set: lane k <-> allele set k */
            {
                constexpr double LN10_10 = 0.2302585092994045684017991454684;
                int n_all = 0, n_called = 0;
                #pragma unroll
                { const int w = warp; n_all += s_redC[w][0]; n_called += s_redC[w][1]; }
                auto total_log = [&](int k, int n) -> double
                {
                    double M = 1.0; int E = 0;
                    #pragma unroll
                    { const int w = warp; M = __dmul_rn(M, s_redM[w][k]); E += s_redE[w][k]; }
                    return log(M) + (double)(E - 1023*n)*LN2;
                };
                const double lnN_all = n_all ? total_log(NACC-2, n_all) : 0.0;
                const double lnN_called = n_called ? total_log(NACC-1, n_called) : 0.0;
                double lk = 0; bool cand = false, in_sum = false; uint32_t mask = 0;
                if ( lane < NALS )
                {
                    long long ps = 0;
                    #pragma unroll
                    ps += s_redP[warp][lane];
                    const bool set = n_all > 0;
                    lk = set ? -LN10_10*(double)ps - lnN_all : 0.0;
                    if ( lane>0 ) lk += a.theta;
                    cand = set; in_sum = set && lane>0; mask = 1u<<lane;
                }
                else if ( lane < NSUB )
                {
                    const int k = lane - NALS;
                    const bool lv = (live >> k) & 1u;
                    const bool set = lv && n_called > 0;
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
                if ( a.exact_phase1 )
                {
                    /* literal phase 1 (options exact_phase1 / adjudicate): lane k walks the group's member list strictly in
                       order with the reference's pdg, val and log (mcall.c:601-698); the products above still filled ssum[] */
                    bool is_set = false;
                    uint32_t xflags = 0;
                    const double xlk = exact_set_lk<NALS,true,int32_t>(site_pl, a.grp_smpl + beg, ng, unseen, ploidy, smem_u32(s_pl2p), a.tab, lane,
                                                                       s_cfp[warp], s_cft[warp], live, a.theta, &is_set, &xflags);
                    if ( lane < NSUB )
                    {
                        lk = xlk; cand = is_set;
                        in_sum = is_set && lane != 0;
                        if ( lane==0 && !is_set ) lk = 0;
                    }
                }
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
                double mx = in_sum ? lk : -CUDART_INF;
                #pragma unroll
                for (int off=16; off; off>>=1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, off));
                double term = in_sum ? exp(lk - mx) : 0.0;
                #pragma unroll
                for (int off=16; off; off>>=1) term += __shfl_xor_sync(0xffffffffu, term, off);
                double g_lk_sum = mx > -CUDART_INF ? mx + log(term) : -CUDART_INF;
                if ( a.exact_phase1 ) g_lk_sum = exact_lk_sum(lk, in_sum, NSUB, -CUDART_INF);     /* running logsumexp2 in enumeration order */
                const double g_ref_lk = __shfl_sync(0xffffffffu, lk, 0);
                const uint32_t g_als = __shfl_sync(0xffffffffu, mask, best_lane & 31);
                if ( lane==0 )
                {
                    const bool any = best_lane < 64;
                    GroupRec &r = grec[g];
                    r.als = any ? g_als : 0;
                    int n = 0;
                    for (int j=0; j<NALS; j++) n += (r.als>>j)&1u;
                    r.nals = n; r.has_max = any;
                    r.ref_lk = g_ref_lk; r.lk_sum = g_lk_sum;
                    r.qual = any ? -4.343*(g_ref_lk - logsumexp2_dev(g_lk_sum, g_ref_lk)) : -CUDART_INF;
                    if ( any && best - second < a.tie_eps ) atomicOr(&st.flags, MCB_SITE_NEAR_TIE);
                }
            }
            __syncwarp();
        }
        __threadfence_block();
        __syncthreads();

        /* =========================== phase B: combine the groups (mcall.c:1546-1577) ============= */
        if ( tid==0 )
        {
            uint32_t als_new = 0, flags = st.flags;
            if ( a.adj_pass ) flags |= MCB_SITE_NEAR_TIE | MCB_SITE_ADJUDICATED;
            double ref_lk = -CUDART_INF, lk_sum = -CUDART_INF, max_qual = -CUDART_INF;
            for (int g=0; g<ngrp; g++)
            {
                const GroupRec &r = grec[g];
                als_new |= r.als;
                if ( !r.has_max ) continue;
                if ( max_qual < r.qual ) { max_qual = r.qual; lk_sum = r.lk_sum; ref_lk = r.ref_lk; }
            }
            als_new |= 1u;
            const int is_variant = als_new!=1;
            st.ret_early = ((a.flag & MCB_CALL_VARONLY) && !is_variant) || (flags & MCB_SITE_NO_QS);
            int nals_new = 0;
            for (int j=0; j<NALS; j++)
            {
                if ( j>0 && j==unseen ) continue;
                if ( a.flag & MCB_CALL_KEEPALT ) als_new |= 1u<<j;
                if ( als_new & (1u<<j) ) nals_new++;
            }
            int nout = 0, kk = 0, l = 0;
            for (int x=0; x<NALS; x++) st.als_map[x] = (als_new & (1u<<x)) ? nout++ : -1;
            for (int x=0; x<NALS; x++)
                for (int y=0; y<=x; y++) { if ( (als_new & (1u<<x)) && (als_new & (1u<<y)) ) { if ( kk<15 ) st.pl_map[kk] = l; kk++; } l++; }
            for (; kk<15; kk++) st.pl_map[kk] = 0;
            if ( unseen && (als_new & (1u<<unseen)) ) flags |= MCB_SITE_UNSEEN_SEL;
            st.pl_dropped = als_new==1;
            st.ref_gt = (als_new==1) || !is_variant;
            if ( st.pl_dropped ) flags |= MCB_SITE_PL_DROPPED;
            if ( st.ref_gt ) flags |= MCB_SITE_REF_GT;
            {
                long long off = site_off;
                if ( a.pl_off_out )
                {
                    off = compact_out_off<true>(a, site, nsmpl, NALS, nals_new, !st.pl_dropped && !st.ret_early, flags);
                    a.pl_off_out[site] = off;
                }
                st.out_off = off;
            }
            st.als_new = als_new; st.nals_new = nals_new; st.is_variant = is_variant; st.flags = flags;
            st.max_qual = max_qual; st.lk_sum = lk_sum; st.ref_lk = ref_lk;
        }
        __syncthreads();
        if ( st.ret_early )
        {
            if ( tid==0 ) { a.ret[site] = 0; if ( a.site_flags ) a.site_flags[site] = st.flags; }
            __syncthreads();
            continue;
        }

        /* =========================== phase C: per-sample genotypes (mcall.c:745-886) ============== */
        {
            const int nals_new = st.nals_new, ngt_new = nals_new*(nals_new+1)/2;
            const bool ref_gt = st.ref_gt;
            const bool want_gq = a.gq && (a.output_tags & (MCB_CALL_FMT_GQ|MCB_CALL_FMT_GP));
            const bool want_gp = a.gp && (a.output_tags & MCB_CALL_FMT_GP) && !ref_gt;
            int32_t *out_pl = (a.out_pl && !st.pl_dropped) ? a.out_pl + st.out_off : nullptr;
            float   *out_gp = want_gp ? a.gp + st.out_off : nullptr;
            int2 *out_gt = a.gt ? reinterpret_cast<int2*>(a.gt) + (size_t)site*nsmpl : nullptr;
            int32_t *out_gq = want_gq ? a.gq + (size_t)site*nsmpl : nullptr;
            uint32_t tflags = 0;
            unsigned long long acc = 0;     /* AC: 12-bit counters per new allele, flushed by warp shuffles (as in the pooled kernel) */
            int acc_n = 0;
            for (int sb=0; sb<nsmpl; sb+=GBLOCK)
            {
                if ( acc_n >= 60 )       /* uniform across the CTA */
                {
                    unsigned long long v = acc;
                    #pragma unroll
                    for (int off=16; off; off>>=1) v += __shfl_xor_sync(0xffffffffu, v, off);
                    if ( lane==0 ) for (int j=0; j<5; j++) { int c = (int)((v >> (12*j)) & 0xfff); if ( c ) atomicAdd(&st.ac[j], c); }
                    acc = 0; acc_n = 0;
                }
                acc_n++;
                const int s = sb + tid;
                if ( s>=nsmpl ) continue;
                const GroupRec &r = grec[a.smpl2grp[s]];
                const int pld = ploidy[s];
                /* ---- the common cases without the full row: phase A left the sample's normaliser, so only the PLs of the
                        group's own genotypes (at most three alleles) and of the kept genotypes are fetched; same expressions
                        in the same order as the general code below */
                {
                    const double sv = ssum[s];
                    const int rn = r.nals;
                    if ( !want_gp && pld<=2 && sv!=GS_GENERIC && (!pld || sv==GS_NODATA || ref_gt || (rn>=1 && rn<=3)) )
                    {
                        const int32_t *row = site_pl + (size_t)s*G;
                        int gt0, gt1, gq = 0;
                        if ( !pld ) { gt0 = MCB_GT_MISSING; gt1 = I32_VEC_END; }
                        else if ( sv==GS_NODATA ) { gt0 = MCB_GT_MISSING; gt1 = pld==2 ? MCB_GT_MISSING : I32_VEC_END; }
                        else if ( ref_gt )
                        {
                            gt0 = MCB_GT_UNPHASED(0); gt1 = pld==2 ? MCB_GT_UNPHASED(0) : I32_VEC_END;
                            acc += (unsigned long long)pld;
                        }
                        else
                        {
                            uint32_t m = r.als;
                            int al[3], nal[3]; double q[3];
                            #pragma unroll
                            for (int i=0; i<3; i++)
                            {
                                al[i] = m ? __ffs(m) - 1 : 0; m &= m - 1;
                                nal[i] = st.als_map[al[i]]; q[i] = r.q[al[i]];
                            }
                            double lkh[3] = {0,0,0}, lkt[3] = {0,0,0};
                            double best = 0; int g0 = 0, g1 = 0;
                            #pragma unroll
                            for (int x=0; x<3; x++)             /* homozygous / haploid (mcall.c:793-808) */
                                if ( x<rn )
                                {
                                    const double pdg = __ddiv_rn(pl_to_p_dev(s_pl2p, a.tab, row[hom_idx(al[x])], &tflags), sv);
                                    lkh[x] = pld==2 ? __dmul_rn(__dmul_rn(pdg, q[x]), q[x]) : __dmul_rn(pdg, q[x]);
                                    if ( best < lkh[x] ) { best = lkh[x]; g0 = nal[x]; }
                                }
                            double gmax = 0, gsum = 0;
                            auto post = [&](double lk) { const double gv = (double)__double2float_rn(lk); if ( gmax < gv ) gmax = gv; gsum = __dadd_rn(gsum, gv); };
                            if ( pld==2 )
                            {
                                g1 = g0;
                                #pragma unroll
                                for (int x=1; x<3; x++)         /* heterozygous (mcall.c:812-834) */
                                    #pragma unroll
                                    for (int y=0; y<x; y++)
                                        if ( x<rn )
                                        {
                                            const double pdg = __ddiv_rn(pl_to_p_dev(s_pl2p, a.tab, row[gt_idx(al[x],al[y])], &tflags), sv);
                                            const double lk = __dmul_rn(__dmul_rn(__dmul_rn(2.0,pdg), q[x]), q[y]);
                                            lkt[x*(x-1)/2 + y] = lk;
                                            if ( best < lk ) { best = lk; g0 = nal[y]; g1 = nal[x]; }
                                        }
                                gt0 = MCB_GT_UNPHASED(g0); gt1 = MCB_GT_UNPHASED(g1);
                                acc += (1ull << (12*min(g0,4))) + (1ull << (12*min(g1,4)));
                                if ( want_gq )                  /* the posteriors in the order of the new genotypes: the kept alleles ascend */
                                {
                                    post(lkh[0]);
                                    if ( rn>1 ) { post(lkt[0]); post(lkh[1]); }
                                    if ( rn>2 ) { post(lkt[1]); post(lkt[2]); post(lkh[2]); }
                                }
                            }
                            else
                            {
                                gt0 = MCB_GT_UNPHASED(g0); gt1 = I32_VEC_END;
                                acc += 1ull << (12*min(g0,4));
                                if ( want_gq )                  /* haploid: the first r.nals entries only (mcall.c:843-850) */
                                {
                                    #pragma unroll
                                    for (int x=0; x<3; x++) if ( x<rn && nal[x]<rn ) post(lkh[x]);
                                }
                            }
                            if ( want_gq ) gq = groups_gq(gmax, gsum, s_thr);
                        }
                        if ( out_gt ) out_gt[s] = make_int2(gt0, gt1);
                        if ( out_gq ) out_gq[s] = gq;
                        if ( out_pl )               /* mcall.c:1158-1194 */
                        {
                            int32_t *dst = out_pl + (size_t)s*ngt_new;
                            for (int k=0; k<ngt_new; k++)
                            {
                                int v;
                                if ( pld==2 ) v = row[st.pl_map[k]];
                                else if ( pld==1 && k<nals_new ) v = row[st.pl_map[hom_idx(k)]];
                                else v = (pld==0 && k==0) ? I32_MISSING : I32_VEC_END;
                                dst[k] = v;
                            }
                        }
                        continue;
                    }
                }
                int pl[G]; double p[G];
                int orv = 0;
                #pragma unroll
                for (int j=0; j<G; j++) { pl[j] = site_pl[(size_t)s*G + j]; orv |= pl[j]; }
                bool has = true;
                if ( orv<0 )
                {
                    int tmp[16];
                    #pragma unroll
                    for (int j=0; j<G; j++) tmp[j] = pl[j];
                    has = fix_missing_local(tmp, NALS, unseen);
                    orv = 0;
                    #pragma unroll
                    for (int j=0; j<G; j++) { if ( has ) pl[j] = tmp[j]; orv |= pl[j]; }
                    if ( orv<0 ) has = false;
                }
                if ( orv==0 ) has = false;
                double sum = 1;
                if ( has )
                {
                    #pragma unroll
                    for (int j=0; j<G; j++) p[j] = pl_to_p_dev(s_pl2p, a.tab, pl[j], &tflags);
                    sum = p[0];
                    #pragma unroll
                    for (int j=1; j<G; j++) sum = __dadd_rn(sum, p[j]);
                }
                int gt0, gt1, gq = 0;
                bool called = false;
                float gps[G];               /* FORMAT/GP scratch in the NEW genotype order, zeroed like mcall.c:1605 */
                #pragma unroll
                for (int j=0; j<G; j++) gps[j] = 0.f;
                double gsum = 0;
                if ( !pld ) { gt0 = MCB_GT_MISSING; gt1 = I32_VEC_END; }
                else if ( !has ) { gt0 = MCB_GT_MISSING; gt1 = pld==2 ? MCB_GT_MISSING : I32_VEC_END; }
                else if ( ref_gt )
                {
                    gt0 = MCB_GT_UNPHASED(0); gt1 = pld==2 ? MCB_GT_UNPHASED(0) : I32_VEC_END;
                    acc += (unsigned long long)pld;
                }
                else
                {
                    called = true;
                    double best = 0; int g0 = 0, g1 = 0;
                    #pragma unroll
                    for (int x=0; x<NALS; x++)          /* homozygous / haploid (mcall.c:793-808) */
                    {
                        if ( !(r.als & (1u<<x)) ) continue;
                        const double pdg = __ddiv_rn(p[hom_idx(x)], sum);
                        const double lk = pld==2 ? __dmul_rn(__dmul_rn(pdg, r.q[x]), r.q[x]) : __dmul_rn(pdg, r.q[x]);
                        const int nx = st.als_map[x];
                        const int igt = pld==2 ? hom_idx(nx) : nx;
                        #pragma unroll
                        for (int j=0; j<G; j++) if ( j==igt ) gps[j] = __double2float_rn(lk);
                        if ( best < lk ) { best = lk; g0 = nx; }
                    }
                    if ( pld==2 )
                    {
                        g1 = g0;
                        #pragma unroll
                        for (int x=1; x<NALS; x++)      /* heterozygous (mcall.c:812-834) */
                            #pragma unroll
                            for (int y=0; y<x; y++)
                            {
                                if ( !(r.als & (1u<<x)) || !(r.als & (1u<<y)) ) continue;
                                const double pdg = __ddiv_rn(p[gt_idx(x,y)], sum);
                                const double lk = __dmul_rn(__dmul_rn(__dmul_rn(2.0,pdg), r.q[x]), r.q[y]);
                                const int igt = gt_idx(st.als_map[x], st.als_map[y]);
                                #pragma unroll
                                for (int j=0; j<G; j++) if ( j==igt ) gps[j] = __double2float_rn(lk);
                                if ( best < lk ) { best = lk; g0 = st.als_map[y]; g1 = st.als_map[x]; }
                            }
                        gt0 = MCB_GT_UNPHASED(g0); gt1 = MCB_GT_UNPHASED(g1);
                        acc += (1ull << (12*min(g0,4))) + (1ull << (12*min(g1,4)));
                    }
                    else
                    {
                        gt0 = MCB_GT_UNPHASED(g0); gt1 = I32_VEC_END;
                        acc += 1ull << (12*min(g0,4));
                    }
                    if ( want_gq || want_gp )           /* mcall.c:843-878 */
                    {
                        const int nmax = pld==2 ? ngt_new : r.nals;
                        double gmax = 0;
                        #pragma unroll
                        for (int j=0; j<G; j++)
                            if ( j<nmax )
                            {
                                const double gv = (double)gps[j];
                                if ( gmax < gv ) gmax = gv;
                                gsum = __dadd_rn(gsum, gv);
                            }
                        gq = groups_gq(gmax, gsum, s_thr);
                    }
                }
                if ( out_gt ) out_gt[s] = make_int2(gt0, gt1);
                if ( out_gq ) out_gq[s] = gq;
                if ( out_pl )               /* mcall.c:1158-1194 on the filled PLs */
                {
                    int32_t *dst = out_pl + (size_t)s*ngt_new;
                    #pragma unroll
                    for (int k=0; k<G; k++)
                    {
                        if ( k>=ngt_new ) continue;
                        int v;
                        if ( pld==2 || (pld==1 && k<nals_new) )
                        {
                            const int src = pld==2 ? st.pl_map[k] : st.pl_map[hom_idx(k)];
                            v = 0;
                            #pragma unroll
                            for (int j=0; j<G; j++) if ( j==src ) v = pl[j];
                        }
                        else v = (pld==0 && k==0) ? I32_MISSING : I32_VEC_END;
                        dst[k] = v;
                    }
                }
                if ( out_gp )               /* mcall.c:859-884 */
                {
                    float *dst = out_gp + (size_t)s*ngt_new;
                    const int nmax = pld==2 ? ngt_new : (pld==1 ? r.nals : 0);
                    if ( !called )
                    {
                        for (int k=0; k<ngt_new; k++) dst[k] = 0.f;
                        if ( nmax==0 ) { dst[0] = __uint_as_float(MCB_FLOAT_MISSING_BITS); if ( 1<ngt_new ) dst[1] = __uint_as_float(MCB_FLOAT_VECTOR_END_BITS); }
                        else if ( nmax<ngt_new ) dst[nmax] = __uint_as_float(MCB_FLOAT_VECTOR_END_BITS);
                    }
                    else
                    {
                        #pragma unroll
                        for (int k=0; k<G; k++)
                            if ( k<ngt_new ) dst[k] = k<nmax ? (float)__ddiv_rn((double)gps[k], gsum) : __uint_as_float(MCB_FLOAT_VECTOR_END_BITS);
                    }
                }
            }
            {
                unsigned long long v = acc;
                #pragma unroll
                for (int off=16; off; off>>=1) v += __shfl_xor_sync(0xffffffffu, v, off);
                if ( lane==0 ) for (int j=0; j<5; j++) { int c = (int)((v >> (12*j)) & 0xfff); if ( c ) atomicAdd(&st.ac[j], c); }
            }
            if ( tflags ) atomicOr(&st.flags, tflags);
        }
        __syncthreads();

        /* ---- site record (mcall.c:1631-1650) */
        if ( tid==0 )
        {
            int nAC = 0;
            if ( !st.ref_gt ) for (int j=1; j<st.nals_new && j<8; j++) nAC += st.ac[j];
            int ret = st.nals_new;
            if ( !st.ref_gt && !nAC && (a.flag & MCB_CALL_VARONLY) ) ret = 0;
            float qual;
            if ( nAC ) qual = (float)st.max_qual;
            else if ( st.lk_sum != -CUDART_INF ) qual = (float)(-4.343*(st.lk_sum - logsumexp2_dev(st.lk_sum, st.ref_lk)));
            else if ( st.ac[0] ) qual = a.theta ? (float)(-4.343*a.theta) : 0.f;
            else qual = __uint_as_float(MCB_FLOAT_MISSING_BITS);
            a.ret[site] = ret;
            if ( a.als_new ) a.als_new[site] = st.als_new;
            if ( a.als_map ) for (int j=0; j<a.max_nals; j++) a.als_map[(size_t)site*a.max_nals + j] = j<NALS ? (int8_t)st.als_map[j] : (int8_t)-1;
            if ( a.qual ) a.qual[site] = qual;
            if ( a.ac ) for (int j=0; j<a.max_nals; j++) a.ac[(size_t)site*a.max_nals + j] = (j<st.nals_new && j<8) ? st.ac[j] : 0;
            if ( a.an ) a.an[site] = nAC + st.ac[0];
            if ( a.site_flags ) a.site_flags[site] = st.flags;
            if ( a.diag ) { double *d = a.diag + (size_t)site*4; d[0] = st.max_qual; d[1] = st.lk_sum; d[2] = st.ref_lk; d[3] = 0; }
        }
        __syncthreads();
    }
}

size_t groups_scratch_bytes(int grid, int ngroups, int nsmpl) { return (size_t)grid*groups_cta_bytes(ngroups, nsmpl); }

cudaError_t launch_groups_kernel(int nals, const KArgs &a, void *scratch, int grid, cudaStream_t st)
{
    GroupRec *sc = (GroupRec*) scratch;
    switch ( nals )
    {
        case 1: mcall_groups_kernel<1><<<grid, GBLOCK, 0, st>>>(a, sc); break;
        case 2: mcall_groups_kernel<2><<<grid, GBLOCK, 0, st>>>(a, sc); break;
        case 3: mcall_groups_kernel<3><<<grid, GBLOCK, 0, st>>>(a, sc); break;
        case 4: mcall_groups_kernel<4><<<grid, GBLOCK, 0, st>>>(a, sc); break;
        case 5: mcall_groups_kernel<5><<<grid, GBLOCK, 0, st>>>(a, sc); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

}   // namespace mcb
