/*  mcall_generic.cu -- correctness-first site kernel for 6..32 alleles (pooled or -G grouped calling).
 *
 *  mpileup never emits more than 5 alleles (B2B_MAX_ALLELES, bam2bcf.h:64), so this path only has to be right, not
 *  fast: the reference accepts up to 32 alleles (call->als_new is a 32-bit mask, mcall.c:1539-1543) and evaluates
 *  every 1-, 2- and 3-allele set, up to 32 + 496 + 4960 = 5488 of them (mcall.c:591-710).
 *
 *    step 0   one thread per sample: copy the PL row to a per-CTA scratch block in global memory, apply the
 *             missing-value fill in place (mcall.c:495-527), store the row's sum (sequential, index order) and a
 *             "has data" flag.
 *    phase A  one warp per group; the allele sets are taken 32 at a time (lane <-> set) and the group's samples are
 *             walked once per chunk of sets, every lane accumulating its set as an exponent-tracked product.  With
 *             KArgs.exact_phase1 every lane sums log(val) sample by sample instead (the literal mcall_find_best_alleles).
 *    phase B  thread 0 combines the groups (mcall.c:1546-1577).
 *    phase C  one thread per sample: literal mcall_call_genotypes (mcall.c:745-886) on the <= 6 genotypes of the
 *             group's <= 3 selected alleles, GQ/GP, PL trimming, AC.
 */
#include "mcall_device.cuh"

namespace mcb {

#define XBLOCK 128
#define XNW    (XBLOCK/32)
#define XMAXA  32
#define XMAXG  (XMAXA*(XMAXA+1)/2)

struct XGroupRec
{
    double q[XMAXA];
    double qual, ref_lk, lk_sum;
    uint32_t als; int nals, has_max, pad;
};
struct XSite
{
    double max_qual, lk_sum, ref_lk;
    uint32_t als_new, flags;
    int nals_new, is_variant, ret_early, pl_dropped, ref_gt;
    long long out_off;
    int als_map[XMAXA], ac[XMAXA+1];
    short pl_map[XMAXG];
};

__device__ int xfix_missing(int *pl, int nals, int unseen)      /* mcall.c:460-527 on a row in global memory */
{
    const int G = nals*(nals+1)/2;
    int j;
    for (j=0; j<G; j++)
    {
        if ( pl[j]==I32_VEC_END ) return 0;
        if ( pl[j]==I32_MISSING ) break;
    }
    if ( j==0 ) return 0;
    if ( j==G ) return 0;
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

__device__ __forceinline__ double xpl_to_p(const double *s_pl2p, const DevTables *tab, int v, uint32_t *flags)
{
    if ( (unsigned)v < 256u ) return s_pl2p[v];
    if ( v > 2500 ) *flags |= MCB_SITE_PL_RANGE;
    return (unsigned)v < (unsigned)MCB_PL2P_BIG ? tab->pl2p_big[v] : 0.0;
}

/*  k-th allele set in the reference's enumeration order: singles, pairs (a>b), triples (a>b>c)  */
__device__ void xdecode_set(int k, int nals, int &sa, int &sb, int &sc)
{
    sb = sc = -1;
    if ( k < nals ) { sa = k; return; }
    k -= nals;
    const int npair = nals*(nals-1)/2;
    if ( k < npair )
    {
        sa = 1; while ( sa*(sa+1)/2 <= k ) sa++;
        sb = k - sa*(sa-1)/2;
        return;
    }
    k -= npair;
    sa = 2; while ( (sa+1)*sa*(sa-1)/6 <= k ) sa++;
    int r = k - sa*(sa-1)*(sa-2)/6;
    sb = 1; while ( sb*(sb+1)/2 <= r ) sb++;
    sc = r - sb*(sb-1)/2;
}

__global__ void __launch_bounds__(XBLOCK) mcall_generic_kernel(const KArgs a, XGroupRec *grp_scratch, int32_t *pl_scratch, double *sum_scratch)
{
    constexpr double LN2 = 0.693147180559945309417232121458;
    __shared__ double s_pl2p[256];
    __shared__ double s_thr[130];
    __shared__ float  s_adc[XNW][8][XMAXA];
    __shared__ XSite  st;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nsmpl = a.nsmpl;
    const bool grouped = a.ngroups > 1;
    const int ngrp = grouped ? a.ngroups : 1;
    XGroupRec *grec = grp_scratch + (size_t)blockIdx.x*ngrp;
    int32_t *fpl = pl_scratch + (size_t)blockIdx.x*nsmpl*XMAXG;         /* filled PL rows of the current site */
    double *fsum = sum_scratch + (size_t)blockIdx.x*nsmpl;              /* per-sample sum, 0 = no data */

    for (int i=tid; i<256; i+=XBLOCK) s_pl2p[i] = a.tab->pl2p[i];
    for (int i=tid; i<130; i+=XBLOCK) s_thr[i] = i<128 ? a.tab->gq_thr[i] : -1.0;
    __syncthreads();

    const int nsites = *a.site_count;
    for (int isite = blockIdx.x; isite < nsites; isite += gridDim.x)
    {
        const int site = a.site_list[isite];
        const int nals = a.nals[site];
        if ( nals<6 || nals>XMAXA )        /* 0 alleles or > 32: skipped like mcall.c:1539-1543 */
        {
            if ( tid==0 ) { a.ret[site] = 0; if ( a.site_flags ) a.site_flags[site] = nals>XMAXA ? MCB_SITE_TOO_MANY_ALS : MCB_SITE_UNSUPPORTED; if ( a.pl_off_out ) a.pl_off_out[site] = -1; }
            continue;
        }
        const int G = nals*(nals+1)/2, npair = nals*(nals-1)/2, nsub = nals + npair + nals*(nals-1)*(nals-2)/6;
        const int64_t site_off = a.pl_off[site];
        const int32_t *site_pl = reinterpret_cast<const int32_t*>(a.pl) + site_off;
        const int unseen = a.unseen ? a.unseen[site] : 0;
        int pid = a.ploidy_id ? a.ploidy_id[site] : 0;
        if ( pid >= a.nploidy ) pid = 0;
        const uint8_t *ploidy = a.ploidy_tab + (size_t)pid*nsmpl;
        const int nad = (grouped && a.nad) ? a.nad[site] : 0;
        const int32_t *site_ad = (grouped && a.ad) ? a.ad + a.ad_off[site] : nullptr;
        const int nqs = a.qs ? (a.nqs ? a.nqs[site] : nals) : 0;
        uint32_t tflags = 0;
        if ( tid==0 )
        {
            st.flags = grouped ? ((site_ad && nad>0) ? 0 : MCB_SITE_NO_QS) : (nqs>0 ? 0 : MCB_SITE_NO_QS);
            for (int j=0; j<=XMAXA; j++) st.ac[j] = 0;
        }
        /* ---- step 0: filled copy of the PL block + per-sample sums */
        for (int s=tid; s<nsmpl; s+=XBLOCK)
        {
            int *row = fpl + (size_t)s*G;
            int orv = 0;
            for (int j=0; j<G; j++) { int v = site_pl[(size_t)s*G + j]; row[j] = v; orv |= v; }
            bool has = true;
            if ( orv<0 )
            {
                has = xfix_missing(row, nals, unseen);
                orv = 0;
                for (int j=0; j<G; j++) orv |= row[j];
                if ( orv<0 ) has = false;
            }
            if ( orv==0 ) has = false;
            double sum = 0;
            if ( has )
            {
                sum = xpl_to_p(s_pl2p, a.tab, row[0], &tflags);
                for (int j=1; j<G; j++) sum = __dadd_rn(sum, xpl_to_p(s_pl2p, a.tab, row[j], &tflags));
            }
            fsum[s] = sum;
        }
        __syncthreads();

        /* =========================== phase A ==================================================== */
        for (int g=warp; g<ngrp; g+=XNW)
        {
            const int beg = grouped ? a.grp_off[g] : 0, end = grouped ? a.grp_off[g+1] : nsmpl;
            /* ---- quality sums: lane a <-> allele a */
            float qa = 0;
            if ( !grouped )
            {
                if ( lane<nals && lane<nqs ) qa = a.qs[(size_t)site*a.max_nals + lane];      /* zero-extended, mcall.c:1458-1464 */
            }
            else if ( site_ad )
                for (int base=beg; base<end; base+=8)
                {
                    if ( lane<8 )
                    {
                        const int i = base + lane;
                        for (int j=0; j<XMAXA; j++) s_adc[warp][lane][j] = 0.f;
                        if ( i<end )
                        {
                            const int32_t *ptr = site_ad + (size_t)a.grp_smpl[i]*nad;
                            float sum = 0; int e = nad<XMAXA ? nad : XMAXA;
                            for (int j=0; j<e; j++)
                            {
                                if ( ptr[j]==I32_VEC_END ) { e = j; break; }
                                if ( ptr[j]!=I32_MISSING ) sum = __fadd_rn(sum, (float)ptr[j]);
                            }
                            if ( sum!=0 )
                                for (int j=0; j<e; j++) if ( ptr[j]!=I32_MISSING ) s_adc[warp][lane][j] = __fdiv_rn((float)ptr[j], sum);
                        }
                    }
                    __syncwarp();
                    const int n = min(8, end-base);
                    for (int k=0; k<n; k++) qa = __fadd_rn(qa, s_adc[warp][k][lane]);
                    __syncwarp();
                }
            /* ---- -F prior + normalisation; lane j holds q[j] */
            if ( a.use_prior && a.prior_an && a.prior_ac )
            {
                const int an = a.prior_an[site];
                if ( an!=I32_MISSING && an>0 )
                {
                    const int32_t *pac = a.prior_ac + (size_t)site*a.max_nals;
                    const double den = __dadd_rn((double)(uint32_t)(end-beg), __dmul_rn(0.5,(double)an));
                    int ac0 = an, stop = nals-1;
                    for (int j=0; j<nals-1; j++)
                    {
                        if ( pac[j]==I32_VEC_END ) { stop = j; break; }
                        if ( pac[j]!=I32_MISSING ) ac0 -= pac[j];
                    }
                    if ( lane>=1 && lane<=stop && pac[lane-1]!=I32_MISSING )
                        qa = (float)__ddiv_rn(__dadd_rn((double)qa, __dmul_rn(0.5,(double)pac[lane-1])), den);
                    if ( ac0<0 && lane==0 ) atomicOr(&st.flags, MCB_SITE_BAD_PRIOR);
                    if ( lane==0 ) qa = (float)__ddiv_rn(__dadd_rn((double)qa, __dmul_rn(0.5,(double)ac0)), den);
                }
            }
            {
                float qs = 0;
                for (int j=0; j<nals; j++) qs = __fadd_rn(qs, __shfl_sync(0xffffffffu, qa, j));
                if ( qs!=0 ) qa = __fdiv_rn(qa, qs);
            }
            if ( lane<nals ) grec[g].q[lane] = (double)qa;
            /* ---- allele sets, 32 at a time */
            double run_best = -CUDART_INF, run_second = -CUDART_INF, run_mx = -CUDART_INF, run_term = 0, ref_lk = 0, run_lse = -CUDART_INF;
            uint32_t run_als = 0; bool any = false;
            uint32_t wflags = 0;
            for (int c0=0; c0<nsub; c0+=32)
            {
                const int k = c0 + lane;
                int sa = 0, sb = -1, sc = -1;
                bool inrange = k < nsub, live = false;
                if ( inrange ) xdecode_set(k, nals, sa, sb, sc);
                const float fqa = __shfl_sync(0xffffffffu, qa, sa), fqb = __shfl_sync(0xffffffffu, qa, sb<0 ? 0 : sb), fqc = __shfl_sync(0xffffffffu, qa, sc<0 ? 0 : sc);
                int tix[6] = {0,0,0,0,0,0}; double cd[6] = {0,0,0,0,0,0}, ch[3] = {0,0,0};
                uint32_t mask = 0; int nonref = 0;
                const bool single = inrange && sb<0;
                if ( single ) { live = true; tix[0] = hom_idx(sa); mask = 1u<<sa; nonref = sa!=0; }
                else if ( inrange && sc<0 )
                {
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
                else if ( inrange )
                {
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
                double M = 1, MN = 1; int E = 0, EN = 0, cnt = 0, since = 0;
                if ( live && !a.exact_phase1 )
                    for (int i=beg; i<end; i++)
                    {
                        const int s = grouped ? a.grp_smpl[i] : i;
                        const double sum = fsum[s];
                        if ( sum==0 ) continue;
                        const int *row = fpl + (size_t)s*G;
                        const int pld = ploidy[s];
                        double val = 0; bool use = false;
                        if ( single ) { val = xpl_to_p(s_pl2p, a.tab, row[tix[0]], &wflags); use = true; }
                        else if ( pld==2 )
                        {
                            val = cd[0]*xpl_to_p(s_pl2p, a.tab, row[tix[0]], &wflags);
                            val = fma(cd[1], xpl_to_p(s_pl2p, a.tab, row[tix[1]], &wflags), val);
                            if ( sc>=0 ) val = fma(cd[2], xpl_to_p(s_pl2p, a.tab, row[tix[2]], &wflags), val);
                            val = fma(cd[3], xpl_to_p(s_pl2p, a.tab, row[tix[3]], &wflags), val);
                            if ( sc>=0 )
                            {
                                val = fma(cd[4], xpl_to_p(s_pl2p, a.tab, row[tix[4]], &wflags), val);
                                val = fma(cd[5], xpl_to_p(s_pl2p, a.tab, row[tix[5]], &wflags), val);
                            }
                            use = true;
                        }
                        else if ( pld==1 )
                        {
                            val = ch[0]*xpl_to_p(s_pl2p, a.tab, row[tix[0]], &wflags);
                            val = fma(ch[1], xpl_to_p(s_pl2p, a.tab, row[tix[1]], &wflags), val);
                            if ( sc>=0 ) val = fma(ch[2], xpl_to_p(s_pl2p, a.tab, row[tix[2]], &wflags), val);
                            use = true;
                        }
                        if ( use && val!=0 ) { acc_mul(M, E, val); acc_mul(MN, EN, sum); cnt++; }
                        if ( ++since >= 256 ) { acc_renorm(M, E); acc_renorm(MN, EN); since = 0; }
                    }
                double lk = 0;
                bool cand = live && cnt>0;
                if ( cand ) lk = (log(M) + (double)(E - 1023*cnt)*LN2) - (log(MN) + (double)(EN - 1023*cnt)*LN2);
                if ( a.exact_phase1 && live )
                {
                    /* literal phase 1 (options exact_phase1 / adjudicate): the group's samples strictly in order, pdg = p/sum by
                       IEEE division (set_pdg, mcall.c:451-544), val in the reference's expression order, lk += log(val)
                       (mcall.c:601-698) -- the numerics of exact_set_lk (mcall_device.cuh) for a set of any 32 alleles */
                    double xt = 0; bool xset = false;
                    for (int i=beg; i<end; i++)
                    {
                        const int s = grouped ? a.grp_smpl[i] : i;
                        const double sum = fsum[s];
                        if ( sum==0 ) continue;
                        const int *row = fpl + (size_t)s*G;
                        auto pdg = [&](int t) -> double { return __ddiv_rn(xpl_to_p(s_pl2p, a.tab, row[tix[t]], &wflags), sum); };
                        const int pld = ploidy[s];
                        double val = 0;
                        if ( single ) val = pdg(0);
                        else if ( pld==2 )
                        {
                            val = __dadd_rn(__dmul_rn(cd[0], pdg(0)), __dmul_rn(cd[1], pdg(1)));
                            if ( sc<0 ) val = __dadd_rn(val, __dmul_rn(cd[3], pdg(3)));
                            else
                            {
                                val = __dadd_rn(val, __dmul_rn(cd[2], pdg(2)));
                                val = __dadd_rn(val, __dmul_rn(cd[3], pdg(3)));
                                val = __dadd_rn(val, __dmul_rn(cd[4], pdg(4)));
                                val = __dadd_rn(val, __dmul_rn(cd[5], pdg(5)));
                            }
                        }
                        else if ( pld==1 )
                        {
                            val = __dadd_rn(__dmul_rn(ch[0], pdg(0)), __dmul_rn(ch[1], pdg(1)));
                            if ( sc>=0 ) val = __dadd_rn(val, __dmul_rn(ch[2], pdg(2)));
                        }
                        if ( val != 0 ) { xt = __dadd_rn(xt, log(val)); xset = true; }
                    }
                    cand = xset; lk = xt;
                }
                if ( inrange ) for (int j=0; j<nonref; j++) lk = __dadd_rn(lk, a.theta);
                const bool in_sum = cand && !(single && sa==0);
                if ( c0==0 ) ref_lk = __shfl_sync(0xffffffffu, lk, 0);
                /* chunk maximum (first in enumeration order), then merge with the running state; earlier chunks win ties */
                double best = cand ? lk : -CUDART_INF; int best_lane = cand ? lane : 64;
                for (int off=16; off; off>>=1)
                {
                    double ob = __shfl_xor_sync(0xffffffffu, best, off);
                    int    ol = __shfl_xor_sync(0xffffffffu, best_lane, off);
                    if ( ob > best || (ob==best && ol < best_lane) ) { best = ob; best_lane = ol; }
                }
                double second = (cand && lane!=best_lane) ? lk : -CUDART_INF;
                for (int off=16; off; off>>=1) second = fmax(second, __shfl_xor_sync(0xffffffffu, second, off));
                const uint32_t cals = __shfl_sync(0xffffffffu, mask, best_lane & 31);
                if ( best_lane < 64 )
                {
                    if ( !any || best > run_best ) { run_second = fmax(run_second, fmax(any ? run_best : -CUDART_INF, second)); run_best = best; run_als = cals; any = true; }
                    else run_second = fmax(run_second, best);
                }
                /* running log-sum-exp over the sets that enter lk_sum (literal path: the reference's logsumexp2 chain) */
                if ( a.exact_phase1 ) run_lse = exact_lk_sum(lk, in_sum, 32, run_lse);
                double mx = in_sum ? lk : -CUDART_INF;
                for (int off=16; off; off>>=1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, off));
                if ( mx > -CUDART_INF )
                {
                    const double nmx = fmax(run_mx, mx);
                    double term = in_sum ? exp(lk - nmx) : 0.0;
                    for (int off=16; off; off>>=1) term += __shfl_xor_sync(0xffffffffu, term, off);
                    run_term = (run_mx > -CUDART_INF ? run_term*exp(run_mx - nmx) : 0.0) + term;
                    run_mx = nmx;
                }
                for (int off=16; off; off>>=1) wflags |= __shfl_xor_sync(0xffffffffu, wflags, off);
            }
            if ( lane==0 )
            {
                XGroupRec &r = grec[g];
                r.als = any ? run_als : 0;
                int n = 0;
                for (int j=0; j<nals; j++) n += (r.als>>j)&1u;
                r.nals = n; r.has_max = any;
                r.ref_lk = ref_lk;
                r.lk_sum = a.exact_phase1 ? run_lse : (run_mx > -CUDART_INF ? run_mx + log(run_term) : -CUDART_INF);
                r.qual = any ? -4.343*(r.ref_lk - logsumexp2_dev(r.lk_sum, r.ref_lk)) : -CUDART_INF;
                uint32_t f = wflags;
                if ( any && run_best - run_second < a.tie_eps ) f |= MCB_SITE_NEAR_TIE;
                if ( f ) atomicOr(&st.flags, f);
            }
        }
        if ( tflags ) atomicOr(&st.flags, tflags);
        __threadfence_block();
        __syncthreads();

        /* =========================== phase B ==================================================== */
        if ( tid==0 )
        {
            uint32_t als_new = 0, flags = st.flags;
            if ( a.adj_pass ) flags |= MCB_SITE_NEAR_TIE | MCB_SITE_ADJUDICATED;
            double ref_lk = -CUDART_INF, lk_sum = -CUDART_INF, max_qual = -CUDART_INF;
            for (int g=0; g<ngrp; g++)
            {
                const XGroupRec &r = grec[g];
                als_new |= r.als;
                if ( !r.has_max ) continue;
                if ( max_qual < r.qual ) { max_qual = r.qual; lk_sum = r.lk_sum; ref_lk = r.ref_lk; }
            }
            als_new |= 1u;
            const int is_variant = als_new!=1;
            st.ret_early = ((a.flag & MCB_CALL_VARONLY) && !is_variant) || (flags & MCB_SITE_NO_QS);
            int nals_new = 0;
            for (int j=0; j<nals; j++)
            {
                if ( j>0 && j==unseen ) continue;
                if ( a.flag & MCB_CALL_KEEPALT ) als_new |= 1u<<j;
                if ( als_new & (1u<<j) ) nals_new++;
            }
            int nout = 0, kk = 0, l = 0;
            for (int x=0; x<nals; x++) st.als_map[x] = (als_new & (1u<<x)) ? nout++ : -1;
            for (int x=0; x<nals; x++)
                for (int y=0; y<=x; y++) { if ( (als_new & (1u<<x)) && (als_new & (1u<<y)) ) { if ( kk<XMAXG ) st.pl_map[kk] = (short)l; kk++; } l++; }
            if ( unseen && (als_new & (1u<<unseen)) ) flags |= MCB_SITE_UNSEEN_SEL;
            st.pl_dropped = als_new==1;
            st.ref_gt = (als_new==1) || !is_variant;
            if ( st.pl_dropped ) flags |= MCB_SITE_PL_DROPPED;
            if ( st.ref_gt ) flags |= MCB_SITE_REF_GT;
            {
                long long off = site_off;
                if ( a.pl_off_out )
                {
                    off = compact_out_off<true>(a, site, nsmpl, nals, nals_new, !st.pl_dropped && !st.ret_early, flags);
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

        /* =========================== phase C ==================================================== */
        {
            const int nals_new = st.nals_new, ngt_new = nals_new*(nals_new+1)/2;
            const bool ref_gt = st.ref_gt;
            const bool want_gq = a.gq && (a.output_tags & (MCB_CALL_FMT_GQ|MCB_CALL_FMT_GP));
            const bool want_gp = a.gp && (a.output_tags & MCB_CALL_FMT_GP) && !ref_gt;
            int32_t *out_pl = (a.out_pl && !st.pl_dropped) ? a.out_pl + st.out_off : nullptr;
            float   *out_gp = want_gp ? a.gp + st.out_off : nullptr;
            int2 *out_gt = a.gt ? reinterpret_cast<int2*>(a.gt) + (size_t)site*nsmpl : nullptr;
            int32_t *out_gq = want_gq ? a.gq + (size_t)site*nsmpl : nullptr;
            uint32_t cflags = 0;
            for (int s=tid; s<nsmpl; s+=XBLOCK)
            {
                const XGroupRec &r = grec[grouped ? a.smpl2grp[s] : 0];
                const int *row = fpl + (size_t)s*G;
                const double sum = fsum[s];
                const bool has = sum!=0;
                const int pld = ploidy[s];
                int gt0, gt1, gq = 0;
                bool called = false;
                double gsum = 0;
                /* the <= 6 genotypes of the <= 3 selected alleles, in the order of the NEW genotype index */
                int sel[3], ns = 0;
                for (int j=0; j<nals && ns<3; j++) if ( (r.als>>j)&1u ) sel[ns++] = j;
                float gpv[6] = {0,0,0,0,0,0}; int gpi[6] = {-1,-1,-1,-1,-1,-1};
                if ( !pld ) { gt0 = MCB_GT_MISSING; gt1 = I32_VEC_END; }
                else if ( !has ) { gt0 = MCB_GT_MISSING; gt1 = pld==2 ? MCB_GT_MISSING : I32_VEC_END; }
                else if ( ref_gt )
                {
                    gt0 = MCB_GT_UNPHASED(0); gt1 = pld==2 ? MCB_GT_UNPHASED(0) : I32_VEC_END;
                    atomicAdd(&st.ac[0], pld);
                }
                else
                {
                    called = true;
                    double best = 0; int g0 = 0, g1 = 0;
                    for (int x=0; x<ns; x++)            /* homozygous / haploid (mcall.c:793-808) */
                    {
                        const int al = sel[x];
                        const double pdg = __ddiv_rn(xpl_to_p(s_pl2p, a.tab, row[hom_idx(al)], &cflags), sum);
                        const double lk = pld==2 ? __dmul_rn(__dmul_rn(pdg, r.q[al]), r.q[al]) : __dmul_rn(pdg, r.q[al]);
                        const int nx = st.als_map[al];
                        const int slot = x*(x+3)/2;
                        gpv[slot] = __double2float_rn(lk); gpi[slot] = pld==2 ? hom_idx(nx) : nx;
                        if ( best < lk ) { best = lk; g0 = nx; }
                    }
                    if ( pld==2 )
                    {
                        g1 = g0;
                        for (int x=1; x<ns; x++)        /* heterozygous (mcall.c:812-834) */
                            for (int y=0; y<x; y++)
                            {
                                const int ax = sel[x], ay = sel[y];
                                const double pdg = __ddiv_rn(xpl_to_p(s_pl2p, a.tab, row[gt_idx(ax,ay)], &cflags), sum);
                                const double lk = __dmul_rn(__dmul_rn(__dmul_rn(2.0,pdg), r.q[ax]), r.q[ay]);
                                const int slot = x*(x+1)/2 + y;
                                gpv[slot] = __double2float_rn(lk); gpi[slot] = gt_idx(st.als_map[ax], st.als_map[ay]);
                                if ( best < lk ) { best = lk; g0 = st.als_map[ay]; g1 = st.als_map[ax]; }
                            }
                        gt0 = MCB_GT_UNPHASED(g0); gt1 = MCB_GT_UNPHASED(g1);
                        atomicAdd(&st.ac[min(g0,XMAXA)], 1); atomicAdd(&st.ac[min(g1,XMAXA)], 1);
                    }
                    else
                    {
                        gt0 = MCB_GT_UNPHASED(g0); gt1 = I32_VEC_END;
                        atomicAdd(&st.ac[min(g0,XMAXA)], 1);
                    }
                    if ( want_gq || want_gp )           /* mcall.c:843-878: slots are already in increasing igt order */
                    {
                        const int nmax = pld==2 ? ngt_new : r.nals;
                        double gmax = 0;
                        for (int k=0; k<6; k++)
                            if ( gpi[k]>=0 && gpi[k]<nmax )
                            {
                                const double gv = (double)gpv[k];
                                if ( gmax < gv ) gmax = gv;
                                gsum = __dadd_rn(gsum, gv);
                            }
                        const double xx = __dadd_rn(1.0, -__ddiv_rn(gmax, gsum));
                        if ( !(xx==xx) ) gq = 127;
                        else
                        {
                            int k = __float2int_rz(-3.0102999f*lg2_approx((float)xx));
                            k = max(0, min(127, k));
                            if ( xx <= s_thr[k+1] ) { k++; while ( xx <= s_thr[k+1] ) k++; }
                            else while ( xx > s_thr[k] ) k--;
                            gq = k;
                        }
                    }
                }
                if ( out_gt ) out_gt[s] = make_int2(gt0, gt1);
                if ( out_gq ) out_gq[s] = gq;
                if ( out_pl )               /* mcall.c:1158-1194 on the filled PLs */
                {
                    int32_t *dst = out_pl + (size_t)s*ngt_new;
                    for (int k=0; k<ngt_new; k++)
                    {
                        int v;
                        if ( pld==2 ) v = row[st.pl_map[k]];
                        else if ( pld==1 ) v = k<nals_new ? row[st.pl_map[hom_idx(k)]] : I32_VEC_END;
                        else v = k==0 ? I32_MISSING : I32_VEC_END;
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
                        const float zero = (float)__ddiv_rn(0.0, gsum);
                        for (int k=0; k<ngt_new; k++) dst[k] = k<nmax ? zero : __uint_as_float(MCB_FLOAT_VECTOR_END_BITS);
                        for (int k=0; k<6; k++)
                            if ( gpi[k]>=0 && gpi[k]<nmax ) dst[gpi[k]] = (float)__ddiv_rn((double)gpv[k], gsum);
                    }
                }
            }
            if ( cflags ) atomicOr(&st.flags, cflags);
        }
        __syncthreads();

        if ( tid==0 )           /* site record (mcall.c:1631-1650) */
        {
            int nAC = 0;
            if ( !st.ref_gt ) for (int j=1; j<st.nals_new && j<=XMAXA; j++) nAC += st.ac[j];
            int ret = st.nals_new;
            if ( !st.ref_gt && !nAC && (a.flag & MCB_CALL_VARONLY) ) ret = 0;
            float qual;
            if ( nAC ) qual = (float)st.max_qual;
            else if ( st.lk_sum != -CUDART_INF ) qual = (float)(-4.343*(st.lk_sum - logsumexp2_dev(st.lk_sum, st.ref_lk)));
            else if ( st.ac[0] ) qual = a.theta ? (float)(-4.343*a.theta) : 0.f;
            else qual = __uint_as_float(MCB_FLOAT_MISSING_BITS);
            a.ret[site] = ret;
            if ( a.als_new ) a.als_new[site] = st.als_new;
            if ( a.als_map ) for (int j=0; j<a.max_nals; j++) a.als_map[(size_t)site*a.max_nals + j] = j<nals ? (int8_t)st.als_map[j] : (int8_t)-1;
            if ( a.qual ) a.qual[site] = qual;
            if ( a.ac ) for (int j=0; j<a.max_nals; j++) a.ac[(size_t)site*a.max_nals + j] = j<st.nals_new ? st.ac[j] : 0;
            if ( a.an ) a.an[site] = nAC + st.ac[0];
            if ( a.site_flags ) a.site_flags[site] = st.flags;
            if ( a.diag ) { double *d = a.diag + (size_t)site*4; d[0] = st.max_qual; d[1] = st.lk_sum; d[2] = st.ref_lk; d[3] = 0; }
        }
        __syncthreads();
    }
}

void generic_scratch_bytes(int grid, int ngroups, int nsmpl, size_t *grp, size_t *pl, size_t *sum)
{
    *grp = (size_t)grid*(ngroups>1 ? ngroups : 1)*sizeof(XGroupRec);
    *pl  = (size_t)grid*nsmpl*XMAXG*sizeof(int32_t);
    *sum = (size_t)grid*nsmpl*sizeof(double);
}

cudaError_t launch_generic_kernel(const KArgs &a, void *grp_scratch, void *pl_scratch, void *sum_scratch, int grid, cudaStream_t st)
{
    mcall_generic_kernel<<<grid, XBLOCK, 0, st>>>(a, (XGroupRec*)grp_scratch, (int32_t*)pl_scratch, (double*)sum_scratch);
    return cudaGetLastError();
}

}   // namespace mcb
