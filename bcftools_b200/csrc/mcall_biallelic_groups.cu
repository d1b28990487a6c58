/*  mcall_biallelic_groups.cu -- grouped calling (`call -m -G`, mcall.c:250-349, 1466-1504, 1546-1561, 1608-1614) for the
 *  dominant site shape: two alleles, int32 PLs, up to 32 sample groups whose member lists are in ascending sample order.
 *
 *  Same mapping as the pooled two-allele kernel (mcall_biallelic.cu): ONE WARP owns one site, no block barrier, a
 *  byte-packed copy of the site (3 bytes per sample) in the warp's shared memory so that HBM sees every PL byte once.
 *  What groups add:
 *
 *    phase 0   the groups' quality sums from FORMAT/AD.  The reference adds the per-sample fractions AD[a]/sum(AD) in
 *              float32 strictly in group order (mcall.c:1484-1501), so the sums stay sequential: lane (g, a) walks the
 *              member list of group g and adds allele a's fractions, which all lanes computed for a chunk of samples
 *              beforehand (coalesced AD reads; the packed-copy buffer is the scratch).  Then the -F prior, the
 *              normalisation and the pair coefficients per group.
 *    phase 1   one pass per group over its member list, gathering from the packed copy: the group's own coefficients are
 *              warp-uniform, the running products are scalars, the totals go to the group's record.
 *    set comparison: lane (g, set) -- 8 groups x {REF}, {ALT}, {ALT,REF} per pass -- then lane 0 combines the groups
 *              (als_new = OR of the groups' sets | REF, QUAL of the best group).
 *    phase 2   one sample per lane with ITS group's record: float32 screen (mcall_device.cuh) where the sample is diploid
 *              and its group selected both alleles, the literal FP64 sequence of mcall_groups.cu otherwise.
 *
 *  Sites this kernel has no code for -- a sample with a partially missing PL vector (set_pdg's fill) or a PL >= 256, a
 *  genuine (255,255,255), the unseen allele selected -- go on the fallback list and are called by mcall_groups.cu.
 */
#include "mcall_device.cuh"

namespace mcb {

#define BG_WARPS     8
#ifndef BG_AD_ASYNC
#define BG_AD_ASYNC  1                  /* phase 0: FORMAT/AD chunks through cp.async when a site has two values per sample */
#endif
#define BG_MINCTA    3
#define BG_MAXGRP    32
#define BG_SITE_BYTES 128

struct __align__(16) BGGroup
{
    float    scr_w[4];              /* float32 screen, diploid samples: weights of 0/0, 0/1, 1/1; [3] != 0: literal path only */
    float    scr_h[4];              /* ... haploid samples: weights of allele 0, (none), allele 1; [3] != 0: literal path only */
    double   q[2];                  /* (double)(float) normalised qsum of REF, ALT (mcall.c:1530-1535) */
    double   cf[5];                 /* pair {ALT,REF}: fa2 (ALT/ALT), fb2 (REF/REF), 2 fa fb, fa, fb (mcall.c:629-633, 642-643) */
    double   accN, accC, accP;      /* products over the group's samples: sum (data), sum (called), val (called); mantissas */
    double   qual, ref_lk, lk_sum;
    int      eN, eC, eP, cnt, cnt_called, ps0, ps1, live;
    uint32_t als; int nals, has_max, pad;
};
struct __align__(16) BGSite
{
    double   max_qual, lk_sum, ref_lk;
    long long out_off;
    uint32_t als_new, flags;
    int      nals_new, ret_early, pl_dropped, ref_gt, fallback;
    int      als_map[2];
};
static_assert(sizeof(BGSite) <= BG_SITE_BYTES, "BGSite grew past its slot");

struct BGTables { double pl2p[256]; double gq_thr[130]; ScreenTabs scr; };

static __device__ __noinline__ double bg_log(double x) { return log(x); }
static __device__ __noinline__ double bg_exp(double x) { return exp(x); }
__device__ __forceinline__ double bg_logsumexp2(double a, double b)
{
    const double hi = a>b ? a : b, lo = a>b ? b : a;
    return bg_log(1 + bg_exp(lo - hi)) + hi;
}
__device__ __forceinline__ uint32_t bg_ldsu8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void bg_sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void bg_cp_async16(uint32_t dst, const void *src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dst), "l"(__cvta_generic_to_global(src)) : "memory");
}
__device__ __forceinline__ void bg_cp_async_wait_all()
{
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void bg_sts_f32x2(uint32_t a, float x, float y) { asm volatile("st.shared.v2.f32 [%0], {%1,%2};" :: "r"(a), "f"(x), "f"(y) : "memory"); }
__device__ __forceinline__ float bg_lds_f32(uint32_t a) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v; }
__device__ __forceinline__ void bg_stg64(void *p, int x, int y) { asm volatile("st.global.cs.v2.s32 [%0], {%1,%2};" :: "l"(p), "r"(x), "r"(y) : "memory"); }
__device__ __forceinline__ void bg_stg32(void *p, int x) { asm volatile("st.global.cs.s32 [%0], %1;" :: "l"(p), "r"(x) : "memory"); }

/*  mcall_call_genotypes (mcall.c:787-878) for one sample of a two-allele site under its group's record: the literal FP64
 *  sequence of mcall_groups.cu phase C.  als: the group's selected alleles, ralsn = grp->nals, map[]: site-level als_map.
 *  Returns g0 | g1 << 8 | gq << 16 (new allele indices; haploid: g1 unused).  */
static __device__ __noinline__ int bg_call_literal(uint32_t a, uint32_t b, uint32_t c, int pld, uint32_t als, int ralsn, double q0, double q1,
                                                   int map0, int map1, int ngt_new, int want_gq, uint32_t pl2p_s, uint32_t thr_s)
{
    const double p0 = lds64c(pl2p_s + 8u*a), p1 = lds64c(pl2p_s + 8u*b), p2 = lds64c(pl2p_s + 8u*c);
    const double sum = __dadd_rn(__dadd_rn(p0, p1), p2);
    float gps[3] = {0.f, 0.f, 0.f};
    double best = 0; int g0 = 0, g1 = 0, gq = 0;
    if ( als & 1u )
    {
        const double pdg = __ddiv_rn(p0, sum);
        const double lk = pld==2 ? __dmul_rn(__dmul_rn(pdg, q0), q0) : __dmul_rn(pdg, q0);
        const int igt = pld==2 ? hom_idx(map0) : map0;
        for (int j=0; j<3; j++) if ( j==igt ) gps[j] = __double2float_rn(lk);
        if ( best < lk ) { best = lk; g0 = map0; }
    }
    if ( als & 2u )
    {
        const double pdg = __ddiv_rn(p2, sum);
        const double lk = pld==2 ? __dmul_rn(__dmul_rn(pdg, q1), q1) : __dmul_rn(pdg, q1);
        const int igt = pld==2 ? hom_idx(map1) : map1;
        for (int j=0; j<3; j++) if ( j==igt ) gps[j] = __double2float_rn(lk);
        if ( best < lk ) { best = lk; g0 = map1; }
    }
    if ( pld==2 )
    {
        g1 = g0;
        if ( als==3u )
        {
            const double pdg = __ddiv_rn(p1, sum);
            const double lk = __dmul_rn(__dmul_rn(__dmul_rn(2.0, pdg), q1), q0);
            const int igt = gt_idx(map1, map0);
            for (int j=0; j<3; j++) if ( j==igt ) gps[j] = __double2float_rn(lk);
            if ( best < lk ) { best = lk; g0 = map0; g1 = map1; }
        }
    }
    if ( want_gq )
    {
        const int nmax = pld==2 ? ngt_new : ralsn;
        double gmax = 0, gsum = 0;
        for (int j=0; j<3; j++)
            if ( j<nmax )
            {
                const double gv = (double)gps[j];
                if ( gmax < gv ) gmax = gv;
                gsum = __dadd_rn(gsum, gv);
            }
        const double xx = __dadd_rn(1.0, -__ddiv_rn(gmax, gsum));
        if ( !(xx==xx) ) gq = 127;
        else
        {
            int k = __float2int_rz(-3.0102999f*lg2_approx((float)xx));
            k = max(0, min(127, k));
            if ( xx <= lds64c(thr_s + 8u*(uint32_t)(k+1)) ) { k++; while ( xx <= lds64c(thr_s + 8u*(uint32_t)(k+1)) ) k++; }
            else while ( xx > lds64c(thr_s + 8u*(uint32_t)k) ) k--;
            gq = k;
        }
    }
    return g0 | g1<<8 | gq<<16;
}

__global__ void __launch_bounds__(BG_WARPS*32, BG_MINCTA) mcall_biallelic_groups_kernel(const KArgs a, int warp_bytes, int buf_bytes)
{
    constexpr double LN2 = 0.693147180559945309417232121458, LN10_10 = 0.2302585092994045684017991454684;
    BGTables &tb = *reinterpret_cast<BGTables*>(mcb_smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t sbase = smem_base();
    const uint32_t pl2p_s = sbase + (uint32_t)offsetof(BGTables, pl2p), thr_s = sbase + (uint32_t)offsetof(BGTables, gq_thr);
    const uint32_t plf_s = sbase + (uint32_t)offsetof(BGTables, scr) + (uint32_t)offsetof(ScreenTabs, plf);
    const uint32_t gqw_s = sbase + (uint32_t)offsetof(BGTables, scr) + (uint32_t)offsetof(ScreenTabs, gqw);
    unsigned char *wmem = mcb_smem + align128(sizeof(BGTables)) + (size_t)warp*warp_bytes;
    const uint32_t wbase_s = sbase + (uint32_t)align128(sizeof(BGTables)) + (uint32_t)warp*(uint32_t)warp_bytes;
    BGSite &rec = *reinterpret_cast<BGSite*>(wmem);
    const int NG = a.ngroups;
    BGGroup *grp = reinterpret_cast<BGGroup*>(wmem + BG_SITE_BYTES);
    const uint32_t grp_s = wbase_s + BG_SITE_BYTES;
    const uint32_t buf_s = grp_s + (uint32_t)(NG*sizeof(BGGroup));

    for (int i=tid; i<256; i+=blockDim.x) tb.pl2p[i] = a.tab->pl2p[i];
    for (int i=tid; i<130; i+=blockDim.x) tb.gq_thr[i] = i<128 ? a.tab->gq_thr[i] : -1.0;
    screen_tabs_fill(&tb.scr, a.tab, tid, blockDim.x);
    __syncthreads();

    const int S = a.nsmpl, nsites = *a.site_count;
    const int CH = (buf_bytes >> 4) << 1;           /* samples per chunk of phase 0: two float32 fractions each; even, so that chunks start on 16 bytes */
    const int want_gq = (a.gq && (a.output_tags & (MCB_CALL_FMT_GQ|MCB_CALL_FMT_GP))) ? 1 : 0;

    for (;;)
    {
        int isite = 0;
        if ( lane==0 ) isite = atomicAdd(a.work_counter, 1);
        isite = __shfl_sync(0xffffffffu, isite, 0);
        if ( isite >= nsites ) break;
        const int site = a.site_list[isite];
        const int64_t site_off = a.pl_off[site];
        const int32_t *site_pl = reinterpret_cast<const int32_t*>(a.pl) + site_off;
        const int unseen = a.unseen ? a.unseen[site] : 0;
        int pid = a.ploidy_id ? a.ploidy_id[site] : 0;
        if ( pid >= a.nploidy ) pid = 0;
        const uint8_t *ploidy = a.ploidy_tab + (size_t)pid*S;
        const int nad = a.nad ? a.nad[site] : 0;
        const int32_t *site_ad = a.ad ? a.ad + a.ad_off[site] : nullptr;
        uint32_t sflags = (site_ad && nad>0) ? 0 : MCB_SITE_NO_QS;
        const bool ad_async = BG_AD_ASYNC && nad==2 && (reinterpret_cast<uintptr_t>(site_ad) & 15)==0;

        /* =========================== phase 0: the groups' quality sums ============================== */
        /*  lane (g, allele) for 16 groups at a time: with more than 16 groups every lane carries two running sums, so that a chunk
            of fractions is staged once and walked by both halves  */
        const int al = lane & 1, NP = NG > 16 ? 2 : 1;
        int mi2[2], end2[2]; float q2[2] = {0.f, 0.f};
        #pragma unroll
        for (int p=0; p<2; p++)
        {
            const int g = p*16 + (lane>>1);
            mi2[p] = g<NG ? (int)a.grp_off[g] : 0; end2[p] = g<NG ? (int)a.grp_off[g+1] : 0;
        }
        {
            if ( site_ad && nad>0 )
                for (int c0=0; c0<S; c0+=CH)
                {
                    const int cend = min(S, c0 + CH);
                    if ( ad_async )
                    {
                        /* two AD values per sample on a 16-byte boundary: the chunk's rows come in with asynchronous copies (one
                           round trip per chunk, not per 32 samples) and are turned into fractions in place */
                        const int n = cend - c0, n16 = n >> 1;
                        const char *src = reinterpret_cast<const char*>(site_ad) + (size_t)c0*8;
                        for (int i=lane; i<n16; i+=32) bg_cp_async16(buf_s + 16u*(uint32_t)i, src + 16*(size_t)i);
                        if ( (n & 1) && lane==0 )
                        {
                            const int2 v = __ldg(reinterpret_cast<const int2*>(src) + (n-1));
                            bg_sts_f32x2(buf_s + 8u*(uint32_t)(n-1), __int_as_float(v.x), __int_as_float(v.y));
                        }
                        bg_cp_async_wait_all();
                        __syncwarp();
                        for (int i=lane; i<n; i+=32)
                        {
                            const uint32_t ad_s = buf_s + 8u*(uint32_t)i;
                            const int a0 = __float_as_int(bg_lds_f32(ad_s)), a1 = __float_as_int(bg_lds_f32(ad_s + 4u));
                            float sum = 0; int e = 2;
                            if ( a0==I32_VEC_END ) e = 0;
                            else
                            {
                                if ( a0!=I32_MISSING ) sum = __fadd_rn(sum, (float)a0);
                                if ( a1==I32_VEC_END ) e = 1;
                                else if ( a1!=I32_MISSING ) sum = __fadd_rn(sum, (float)a1);
                            }
                            float f0 = 0, f1 = 0;
                            if ( sum!=0 )
                            {
                                if ( 0<e && a0!=I32_MISSING ) f0 = __fdiv_rn((float)a0, sum);
                                if ( 1<e && a1!=I32_MISSING ) f1 = __fdiv_rn((float)a1, sum);
                            }
                            bg_sts_f32x2(ad_s, f0, f1);
                        }
                    }
                    else
                    {
                    /* every lane: the fractions AD[a]/sum of its samples of the chunk (independent per sample) */
                    int nxt[5];
                    #pragma unroll
                    for (int j=0; j<5; j++) nxt[j] = (j<nad && c0+lane<cend) ? __ldg(site_ad + (size_t)(c0+lane)*nad + j) : I32_VEC_END;
                    for (int s=c0+lane; s<cend; s+=32)
                    {
                        int adv[5]; float sum = 0; int e = nad<5 ? nad : 5;
                        #pragma unroll
                        for (int j=0; j<5; j++) adv[j] = nxt[j];
                        #pragma unroll
                        for (int j=0; j<5; j++) nxt[j] = (j<nad && s+32<cend) ? __ldg(site_ad + (size_t)(s+32)*nad + j) : I32_VEC_END;     /* the next sample's AD is on its way */
                        #pragma unroll
                        for (int j=0; j<5; j++)
                        {
                            if ( j>=e ) break;
                            if ( adv[j]==I32_VEC_END ) { e = j; break; }
                            if ( adv[j]!=I32_MISSING ) sum = __fadd_rn(sum, (float)adv[j]);
                        }
                        float f0 = 0, f1 = 0;
                        if ( sum!=0 )
                        {
                            if ( 0<e && adv[0]!=I32_MISSING ) f0 = __fdiv_rn((float)adv[0], sum);
                            if ( 1<e && adv[1]!=I32_MISSING ) f1 = __fdiv_rn((float)adv[1], sum);
                        }
                        bg_sts_f32x2(buf_s + 8u*(uint32_t)(s-c0), f0, f1);
                    }
                    }
                    __syncwarp();
                    /* lane (g, a): the float32 running sum over the members of g inside the chunk, in group order (adding +0 is exact) */
                    #pragma unroll
                    for (int p=0; p<2; p++)
                    {
                    if ( p>=NP ) continue;
                    int mi = mi2[p]; const int end = end2[p]; float q = q2[p];
                    for (;;)
                    {
                        /* four member indices per round: their loads are independent, the float32 additions stay in order */
                        const int i0 = mi  <end ? (int)__ldg(a.grp_smpl + mi)   : 0x7fffffff, i1 = mi+1<end ? (int)__ldg(a.grp_smpl + mi+1) : 0x7fffffff;
                        const int i2 = mi+2<end ? (int)__ldg(a.grp_smpl + mi+2) : 0x7fffffff, i3 = mi+3<end ? (int)__ldg(a.grp_smpl + mi+3) : 0x7fffffff;
                        const uint32_t fo = buf_s + 4u*(uint32_t)al - 8u*(uint32_t)c0;
                        if ( i0 >= cend ) break;
                        q = __fadd_rn(q, bg_lds_f32(fo + 8u*(uint32_t)i0)); mi++;
                        if ( i1 >= cend ) break;
                        q = __fadd_rn(q, bg_lds_f32(fo + 8u*(uint32_t)i1)); mi++;
                        if ( i2 >= cend ) break;
                        q = __fadd_rn(q, bg_lds_f32(fo + 8u*(uint32_t)i2)); mi++;
                        if ( i3 >= cend ) break;
                        q = __fadd_rn(q, bg_lds_f32(fo + 8u*(uint32_t)i3)); mi++;
                    }
                    mi2[p] = mi; q2[p] = q;
                    }
                    __syncwarp();
                }
        }
        #pragma unroll
        for (int p=0; p<2; p++)
        {
            if ( p>=NP ) continue;
            const int g = p*16 + (lane>>1);
            const bool gvalid = g < NG;
            const int beg = gvalid ? (int)a.grp_off[g] : 0, end = end2[p];
            const float q = q2[p];
            const float qo = __shfl_xor_sync(0xffffffffu, q, 1);
            float qf0 = al ? qo : q, qf1 = al ? q : qo;
            /* -F prior (mcall.c:1507-1527) with this group's sample count, then normalisation (1530-1535) */
            if ( a.use_prior && a.prior_an && a.prior_ac )
            {
                const int an = a.prior_an[site];
                if ( an!=I32_MISSING && an>0 )
                {
                    const int32_t *pac = a.prior_ac + (size_t)site*a.max_nals;
                    const double den = __dadd_rn((double)(uint32_t)(end-beg), __dmul_rn(0.5,(double)an));
                    int ac0 = an;
                    if ( pac[0]!=I32_VEC_END && pac[0]!=I32_MISSING )
                    {
                        ac0 -= pac[0];
                        qf1 = (float)__ddiv_rn(__dadd_rn((double)qf1, __dmul_rn(0.5,(double)pac[0])), den);
                    }
                    if ( ac0<0 ) sflags |= MCB_SITE_BAD_PRIOR;
                    qf0 = (float)__ddiv_rn(__dadd_rn((double)qf0, __dmul_rn(0.5,(double)ac0)), den);
                }
            }
            {
                const float qs = __fadd_rn(__fadd_rn(0.f, qf0), qf1);
                if ( qs!=0 ) { qf0 = __fdiv_rn(qf0, qs); qf1 = __fdiv_rn(qf1, qs); }
            }
            if ( gvalid && al==0 )
            {
                BGGroup &r = grp[g];
                r.q[0] = (double)qf0; r.q[1] = (double)qf1;
                const bool live = qf1!=0 && qf0!=0;
                double fa = 0, fb = 0;
                if ( live )
                {
                    const float den = __fadd_rn(qf1, qf0);
                    fa = (double)__fdiv_rn(qf1, den); fb = (double)__fdiv_rn(qf0, den);
                }
                r.cf[0] = __dmul_rn(fa,fa); r.cf[1] = __dmul_rn(fb,fb); r.cf[2] = __dmul_rn(__dmul_rn(2.0,fa),fb); r.cf[3] = fa; r.cf[4] = fb;
                r.live = live;
            }
        }
        #pragma unroll
        for (int off=16; off; off>>=1) sflags |= __shfl_xor_sync(0xffffffffu, sflags, off);
        __syncwarp();

        /* =========================== packed copy of the site (as phase 1 of mcall_biallelic.cu) ===== */
        bool need_fb = false;
        {
            const int ngrp4 = (S + 3) >> 2, niter = (ngrp4 + 31) >> 5;
            const int4 *site_pl4 = reinterpret_cast<const int4*>(site_pl);
            const char *site_end = reinterpret_cast<const char*>(site_pl) + (size_t)S*12;
            const char *pf = reinterpret_cast<const char*>(site_pl) + (size_t)4*1536 + 128*lane;
            #pragma unroll 1
            for (int it=0; it<niter; it++)
            {
                const int g4 = it*32 + lane;
                if ( lane < 12 && pf < site_end ) asm volatile("prefetch.global.L2 [%0];" :: "l"(pf));
                pf += 1536;
                int x[12];
                if ( 4*g4 + 3 < S )
                {
                    const int4 v0 = __ldg(site_pl4 + 3*g4), v1 = __ldg(site_pl4 + 3*g4 + 1), v2 = __ldg(site_pl4 + 3*g4 + 2);
                    x[0] = v0.x; x[1] = v0.y; x[2] = v0.z; x[3] = v0.w; x[4] = v1.x; x[5] = v1.y; x[6] = v1.z; x[7] = v1.w;
                    x[8] = v2.x; x[9] = v2.y; x[10] = v2.z; x[11] = v2.w;
                }
                else
                {
                    #pragma unroll
                    for (int k=0; k<12; k++) x[k] = (4*g4 + k/3 < S) ? __ldg(site_pl + 12*g4 + k) : 0;
                }
                uint32_t pk[3] = {0,0,0};
                #pragma unroll
                for (int j=0; j<4; j++)
                {
                    const int pa = x[3*j], pb = x[3*j+1], pc = x[3*j+2];
                    const int orv = pa | pb | pc;
                    uint32_t tri;
                    if ( (unsigned)orv <= 255u ) { tri = (uint32_t)pa | (uint32_t)pb<<8 | (uint32_t)pc<<16; if ( tri==0xffffffu ) need_fb = true; }
                    else
                    {
                        /* sentinels: a vector whose FIRST value is missing / vector_end carries no data (mcall.c:465-481) and keeps its
                           raw values; anything else (partial fill, PL >= 256) is the general kernel's */
                        tri = 0xffffffu;
                        if ( pa!=I32_MISSING && pa!=I32_VEC_END ) need_fb = true;
                    }
                    if ( j==0 ) pk[0] |= tri;
                    if ( j==1 ) { pk[0] |= tri<<24; pk[1] |= tri>>8; }
                    if ( j==2 ) { pk[1] |= tri<<16; pk[2] |= tri>>16; }
                    if ( j==3 ) pk[2] |= tri<<8;
                }
                if ( g4 < ngrp4 ) { bg_sts32(buf_s + 12u*(uint32_t)g4, pk[0]); bg_sts32(buf_s + 12u*(uint32_t)g4 + 4u, pk[1]); bg_sts32(buf_s + 12u*(uint32_t)g4 + 8u, pk[2]); }
            }
        }
        if ( __any_sync(0xffffffffu, need_fb) )
        {
            if ( lane==0 ) a.fb_list[atomicAdd(a.fb_count, 1)] = site;
            __syncwarp();
            continue;
        }
        __syncwarp();

        /* =========================== phase 1: one pass per group over its member list ================ */
        #pragma unroll 1
        for (int g=0; g<NG; g++)
        {
            BGGroup &r = grp[g];
            const int beg = (int)a.grp_off[g], end = (int)a.grp_off[g+1];
            const double cf0 = r.cf[0], cf1 = r.cf[1], cf2 = r.cf[2], fa = r.cf[3], fb = r.cf[4];
            const bool live = r.live != 0;
            double accN = 1.0, accC = 1.0, accP = 1.0; int eN = 0, eC = 0, eP = 0;
            int cnt = 0, cnt_called = 0, ps0 = 0, ps1 = 0;
            int s_n = beg+lane<end ? (int)__ldg(a.grp_smpl + beg + lane) : 0;
            #pragma unroll 1
            for (int mi=beg+lane; mi<end; mi+=32)
            {
                const int s = s_n;
                if ( mi+32 < end ) s_n = (int)__ldg(a.grp_smpl + mi + 32);
                const uint32_t ad = buf_s + 3u*(uint32_t)s;
                const uint32_t pa = bg_ldsu8(ad), pb = bg_ldsu8(ad + 1u), pc = bg_ldsu8(ad + 2u);
                const uint32_t tri = pa | pb<<8 | pc<<16;
                if ( tri==0u || tri==0xffffffu ) continue;             /* PL=0,0,0 / all missing: no data (mcall.c:529-537) */
                const int pld = (int)__ldg(ploidy + s);
                const double p0 = lds64c(pl2p_s + 8u*pa), p1 = lds64c(pl2p_s + 8u*pb), p2 = lds64c(pl2p_s + 8u*pc);
                const double sum = __dadd_rn(__dadd_rn(p0, p1), p2);
                cnt++; ps0 += (int)pa; ps1 += (int)pc;                  /* single-allele sets: every sample with data, also ploidy 0 (mcall.c:607-611) */
                acc_mul(accN, eN, sum);
                if ( pld==0 ) continue;
                cnt_called++;
                acc_mul(accC, eC, sum);
                if ( live )
                {
                    const double val = pld==2 ? fma(cf2, p1, fma(cf1, p0, cf0*p2)) : fma(fb, p0, fa*p2);
                    acc_mul(accP, eP, val);
                }
            }
            acc_renorm(accN, eN); acc_renorm(accC, eC); acc_renorm(accP, eP);
            #pragma unroll
            for (int off=16; off; off>>=1)
            {
                accN = __dmul_rn(accN, __shfl_xor_sync(0xffffffffu, accN, off)); eN += __shfl_xor_sync(0xffffffffu, eN, off);
                accC = __dmul_rn(accC, __shfl_xor_sync(0xffffffffu, accC, off)); eC += __shfl_xor_sync(0xffffffffu, eC, off);
                accP = __dmul_rn(accP, __shfl_xor_sync(0xffffffffu, accP, off)); eP += __shfl_xor_sync(0xffffffffu, eP, off);
                cnt += __shfl_xor_sync(0xffffffffu, cnt, off); cnt_called += __shfl_xor_sync(0xffffffffu, cnt_called, off);
                ps0 += __shfl_xor_sync(0xffffffffu, ps0, off); ps1 += __shfl_xor_sync(0xffffffffu, ps1, off);
            }
            acc_renorm(accN, eN); acc_renorm(accC, eC); acc_renorm(accP, eP);
            if ( lane==0 )
            {
                /* acc_mul adds the BIASED exponent of every factor; acc_renorm removes its own bias */
                r.accN = accN; r.eN = eN - 1023*cnt;
                r.accC = accC; r.eC = eC - 1023*cnt_called;
                r.accP = accP; r.eP = eP - 1023*(live ? cnt_called : 0);
                r.cnt = cnt; r.cnt_called = cnt_called; r.ps0 = ps0; r.ps1 = ps1;
            }
        }
        __syncwarp();

        /* =========================== the groups' best sets: lane (g, set), 8 groups per pass ========= */
        uint32_t tie = 0;
        #pragma unroll 1
        for (int gbase=0; gbase<NG; gbase+=8)
        {
            const int g = gbase + (lane>>2), set = lane & 3, seg = lane & ~3;
            const bool gvalid = g < NG && set < 3;
            double lg = 0;          /* set 0: log prod sum (data), set 1: log prod sum (called), set 2: log prod val */
            int cnt = 0, cnt_called = 0, live = 0, ps = 0;
            if ( gvalid )
            {
                const BGGroup &r = grp[g];
                cnt = r.cnt; cnt_called = r.cnt_called; live = r.live;
                if ( set==0 ) { if ( cnt ) lg = bg_log(r.accN) + (double)r.eN*LN2; ps = r.ps0; }
                else if ( set==1 ) { if ( cnt_called ) lg = bg_log(r.accC) + (double)r.eC*LN2; ps = r.ps1; }
                else if ( live && cnt_called ) lg = bg_log(r.accP) + (double)r.eP*LN2;
            }
            const double lnN = __shfl_sync(0xffffffffu, lg, seg), lnNc = __shfl_sync(0xffffffffu, lg, seg+1);
            double lk = 0; bool cand = false, in_sum = false; uint32_t mask = 0;
            if ( gvalid )
            {
                if ( set < 2 )
                {
                    const bool isset = cnt > 0;
                    lk = isset ? -LN10_10*(double)ps - lnN : 0.0;
                    if ( set>0 ) lk += a.theta;
                    cand = isset; in_sum = isset && set>0; mask = 1u<<set;
                }
                else
                {
                    const bool isset = live && cnt_called > 0;
                    lk = isset ? lg - lnNc : 0.0;
                    lk += a.theta;
                    cand = isset; in_sum = isset; mask = 3u;
                }
            }
            /* first strict maximum in enumeration order inside the group's four lanes (UPDATE_MAX_LKs, mcall.c:582-585) */
            double best = cand ? lk : -CUDART_INF; int best_lane = cand ? lane : 64;
            #pragma unroll
            for (int off=2; off; off>>=1)
            {
                const double ob = __shfl_xor_sync(0xffffffffu, best, off);
                const int    ol = __shfl_xor_sync(0xffffffffu, best_lane, off);
                if ( ob > best || (ob==best && ol < best_lane) ) { best = ob; best_lane = ol; }
            }
            double second = (cand && lane!=best_lane) ? lk : -CUDART_INF;
            #pragma unroll
            for (int off=2; off; off>>=1) second = fmax(second, __shfl_xor_sync(0xffffffffu, second, off));
            double mx = in_sum ? lk : -CUDART_INF;
            #pragma unroll
            for (int off=2; off; off>>=1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, off));
            double term = in_sum ? bg_exp(lk - mx) : 0.0;
            #pragma unroll
            for (int off=2; off; off>>=1) term += __shfl_xor_sync(0xffffffffu, term, off);
            const double ref_lk = __shfl_sync(0xffffffffu, lk, seg);
            const uint32_t g_als = __shfl_sync(0xffffffffu, mask, best_lane & 31);
            if ( g < NG && set==0 )
            {
                BGGroup &r = grp[g];
                const bool any = best_lane < 64;
                const double g_lk_sum = mx > -CUDART_INF ? mx + bg_log(term) : -CUDART_INF;
                r.als = any ? g_als : 0;
                r.nals = (int)((r.als & 1u) + ((r.als >> 1) & 1u));
                r.has_max = any;
                r.ref_lk = ref_lk; r.lk_sum = g_lk_sum;
                r.qual = any ? -4.343*(ref_lk - bg_logsumexp2(g_lk_sum, ref_lk)) : -CUDART_INF;
                if ( any && best - second < a.tie_eps ) tie = MCB_SITE_NEAR_TIE;
                bool scr = r.als==3u;
                r.scr_w[0] = screen_weight(r.q[0], r.q[0], 1.0, scr); r.scr_w[1] = screen_weight(r.q[1], r.q[0], 2.0, scr);
                r.scr_w[2] = screen_weight(r.q[1], r.q[1], 1.0, scr); r.scr_w[3] = scr ? 0.f : 1.f;
                bool scrh = r.als==3u;      /* haploid: lk = pdg*q over the two alleles (mcall.c:793-808): the same screen with no het term */
                r.scr_h[0] = screen_weight(r.q[0], 1.0, 1.0, scrh); r.scr_h[1] = 0.f;
                r.scr_h[2] = screen_weight(r.q[1], 1.0, 1.0, scrh); r.scr_h[3] = scrh ? 0.f : 1.f;
            }
        }
        #pragma unroll
        for (int off=16; off; off>>=1) tie |= __shfl_xor_sync(0xffffffffu, tie, off);
        __syncwarp();

        /* =========================== combine the groups (mcall.c:1546-1577), lane 0 ================== */
        if ( lane==0 )
        {
            uint32_t als_new = 0, flags = sflags | tie;
            double ref_lk = -CUDART_INF, lk_sum = -CUDART_INF, max_qual = -CUDART_INF;
            for (int g=0; g<NG; g++)
            {
                const BGGroup &r = grp[g];
                als_new |= r.als;
                if ( !r.has_max ) continue;
                if ( max_qual < r.qual ) { max_qual = r.qual; lk_sum = r.lk_sum; ref_lk = r.ref_lk; }
            }
            als_new |= 1u;
            const int is_variant = als_new!=1;
            rec.ret_early = ((a.flag & MCB_CALL_VARONLY) && !is_variant) || (flags & MCB_SITE_NO_QS);
            int nals_new = 1;
            if ( unseen!=1 )
            {
                if ( a.flag & MCB_CALL_KEEPALT ) als_new |= 2u;
                if ( als_new & 2u ) nals_new++;
            }
            rec.als_map[0] = 0; rec.als_map[1] = (als_new & 2u) ? 1 : -1;
            rec.fallback = (unseen && (als_new & (1u<<unseen))) ? 1 : 0;      /* the unseen allele was selected: the general kernel's (flags it) */
            rec.pl_dropped = als_new==1;
            rec.ref_gt = (als_new==1) || !is_variant;
            if ( rec.pl_dropped ) flags |= MCB_SITE_PL_DROPPED;
            if ( rec.ref_gt ) flags |= MCB_SITE_REF_GT;
            long long off = site_off;
            if ( a.pl_off_out && !rec.fallback )
            {
                off = compact_out_off<false>(a, site, S, 2, nals_new, !rec.pl_dropped && !rec.ret_early, flags);
                a.pl_off_out[site] = off;
            }
            rec.out_off = off;
            rec.als_new = als_new; rec.nals_new = nals_new; rec.flags = flags;
            rec.max_qual = max_qual; rec.lk_sum = lk_sum; rec.ref_lk = ref_lk;
            if ( rec.fallback ) a.fb_list[atomicAdd(a.fb_count, 1)] = site;
        }
        __syncwarp();
        if ( rec.fallback ) { __syncwarp(); continue; }
        if ( rec.ret_early )
        {
            if ( lane==0 ) { a.ret[site] = 0; if ( a.site_flags ) a.site_flags[site] = rec.flags; }
            __syncwarp();
            continue;
        }

        /* =========================== phase 2: per-sample genotypes (mcall.c:745-886) ================= */
        int ac0 = 0, ac1 = 0;
        {
            const int nals_new = rec.nals_new, ngt_new = nals_new*(nals_new+1)/2;
            const bool ref_gt = rec.ref_gt != 0;
            const int map0 = rec.als_map[0], map1 = rec.als_map[1];
            int32_t *out_pl = (a.out_pl && !rec.pl_dropped) ? a.out_pl + rec.out_off : nullptr;
            int2 *out_gt = a.gt ? reinterpret_cast<int2*>(a.gt) + (size_t)site*S : nullptr;
            int32_t *out_gq = want_gq ? a.gq + (size_t)site*S : nullptr;
            const bool scr_site = nals_new==2 && map0==0 && map1==1 && want_gq;
            int pld_n = lane<S ? (int)__ldg(ploidy + lane) : 0;
            uint32_t gi_n = lane<S ? __ldg(a.smpl2grp + lane) : 0;
            #pragma unroll 1
            for (int s=lane; s<S; s+=32)
            {
                const uint32_t ad = buf_s + 3u*(uint32_t)s;
                const uint32_t pa = bg_ldsu8(ad), pb = bg_ldsu8(ad + 1u), pc = bg_ldsu8(ad + 2u);
                const uint32_t tri = pa | pb<<8 | pc<<16;
                const int pld = pld_n;
                const uint32_t gi = gi_n;
                if ( s+32 < S ) { pld_n = (int)__ldg(ploidy + s + 32); gi_n = __ldg(a.smpl2grp + s + 32); }
                const bool esc = tri==0xffffffu, has = !esc && tri!=0u;
                int gt0, gt1, gq = 0;
                if ( !pld ) { gt0 = MCB_GT_MISSING; gt1 = I32_VEC_END; }
                else if ( !has ) { gt0 = MCB_GT_MISSING; gt1 = pld==2 ? MCB_GT_MISSING : I32_VEC_END; }
                else if ( ref_gt ) { gt0 = MCB_GT_UNPHASED(0); gt1 = pld==2 ? MCB_GT_UNPHASED(0) : I32_VEC_END; ac0 += pld; }
                else
                {
                    const uint32_t r_s = grp_s + gi*(uint32_t)sizeof(BGGroup) + (pld==2 ? 0u : 16u);       /* scr_w / scr_h */
                    float w0, w1, w2, wn;
                    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(w0), "=f"(w1), "=f"(w2), "=f"(wn) : "r"(r_s));
                    int g0, g1;
                    bool done = false;
                    if ( scr_site && wn==0.f )
                    {
                        int k, q;
                        if ( screen2_call(pa, pb, pc, w0, w1, w2, plf_s, gqw_s, k, q) ) { g0 = k==2 ? 1 : 0; g1 = k ? 1 : 0; gq = q; done = true; }
                    }
                    if ( !done )
                    {
                        const BGGroup &r = grp[gi];
                        const int e = bg_call_literal(pa, pb, pc, pld, r.als, r.nals, r.q[0], r.q[1], map0, map1, ngt_new, want_gq, pl2p_s, thr_s);
                        g0 = e & 255; g1 = (e >> 8) & 255; gq = e >> 16;
                    }
                    gt0 = MCB_GT_UNPHASED(g0);
                    if ( pld==2 ) { gt1 = MCB_GT_UNPHASED(g1); ac0 += (g0==0) + (g1==0); ac1 += (g0==1) + (g1==1); }
                    else { gt1 = I32_VEC_END; ac0 += g0==0; ac1 += g0==1; }
                }
                if ( out_gt ) bg_stg64(out_gt + s, gt0, gt1);
                if ( out_gq ) bg_stg32(out_gq + s, gq);
                if ( out_pl )           /* mcall.c:1158-1194: both alleles kept (the only shape with a PL tag here), rows by ploidy */
                {
                    int v0 = (int)pa, v1 = (int)pb, v2 = (int)pc;
                    if ( esc ) { v0 = __ldg(site_pl + 3*s); v1 = __ldg(site_pl + 3*s + 1); v2 = __ldg(site_pl + 3*s + 2); }     /* the raw sentinels are what gets copied */
                    int32_t *d = out_pl + 3*(size_t)s;
                    if ( pld==2 ) { bg_stg32(d, v0); bg_stg32(d+1, v1); bg_stg32(d+2, v2); }
                    else if ( pld==1 ) { bg_stg32(d, v0); bg_stg32(d+1, v2); bg_stg32(d+2, I32_VEC_END); }
                    else { bg_stg32(d, I32_MISSING); bg_stg32(d+1, I32_VEC_END); bg_stg32(d+2, I32_VEC_END); }
                }
            }
        }
        #pragma unroll
        for (int off=16; off; off>>=1) { ac0 += __shfl_xor_sync(0xffffffffu, ac0, off); ac1 += __shfl_xor_sync(0xffffffffu, ac1, off); }

        /* ---- site record (mcall.c:1631-1650) */
        if ( lane==0 )
        {
            const int nals_new = rec.nals_new;
            int nAC = 0;
            if ( !rec.ref_gt && nals_new>1 ) nAC = ac1;
            int ret = nals_new;
            if ( !rec.ref_gt && !nAC && (a.flag & MCB_CALL_VARONLY) ) ret = 0;
            float qual;
            if ( nAC ) qual = (float)rec.max_qual;
            else if ( rec.lk_sum != -CUDART_INF ) qual = (float)(-4.343*(rec.lk_sum - bg_logsumexp2(rec.lk_sum, rec.ref_lk)));
            else if ( ac0 ) qual = a.theta ? (float)(-4.343*a.theta) : 0.f;
            else qual = __uint_as_float(MCB_FLOAT_MISSING_BITS);
            a.ret[site] = ret;
            if ( a.als_new ) a.als_new[site] = rec.als_new;
            if ( a.als_map ) for (int j=0; j<a.max_nals; j++) a.als_map[(size_t)site*a.max_nals + j] = j<2 ? (int8_t)rec.als_map[j] : (int8_t)-1;
            if ( a.qual ) a.qual[site] = qual;
            if ( a.ac ) for (int j=0; j<a.max_nals; j++) a.ac[(size_t)site*a.max_nals + j] = j==0 ? ac0 : ((j==1 && nals_new>1) ? ac1 : 0);
            if ( a.an ) a.an[site] = nAC + ac0;
            if ( a.site_flags ) a.site_flags[site] = rec.flags;
            if ( a.diag ) { double *d = a.diag + (size_t)site*4; d[0] = rec.max_qual; d[1] = rec.lk_sum; d[2] = rec.ref_lk; d[3] = 0; }
        }
        __syncwarp();
    }
}

/* ------------------------------------------------------------------------------------------------
 *  launcher
 * ---------------------------------------------------------------------------------------------- */
static size_t bg_buf_bytes(int nsmpl)      /* the packed copy; at least one 32-sample chunk of phase-0 fractions */
{
    const size_t packed = ((size_t)3*(((size_t)nsmpl + 3) & ~(size_t)3) + 15) & ~(size_t)15;
    return packed < 256 ? 256 : packed;
}
size_t biallelic_groups_smem_bytes(int nsmpl, int ngroups)
{
    const size_t wb = BG_SITE_BYTES + (size_t)ngroups*sizeof(BGGroup) + bg_buf_bytes(nsmpl);
    return align128(sizeof(BGTables)) + (size_t)BG_WARPS*((wb + 15) & ~(size_t)15);
}
bool biallelic_groups_ok(int nsmpl, int ngroups) { return ngroups >= 2 && ngroups <= BG_MAXGRP && nsmpl >= 1 && biallelic_groups_smem_bytes(nsmpl, ngroups) <= 227u*1024u; }
int biallelic_groups_warps() { return BG_WARPS; }
int biallelic_groups_ctas_per_sm() { return BG_MINCTA; }

cudaError_t launch_biallelic_groups_kernel(const KArgs &a, int grid, cudaStream_t st)
{
    const size_t smem = biallelic_groups_smem_bytes(a.nsmpl, a.ngroups);
    const size_t wb = ((BG_SITE_BYTES + (size_t)a.ngroups*sizeof(BGGroup) + bg_buf_bytes(a.nsmpl)) + 15) & ~(size_t)15;
    cudaError_t e = cudaFuncSetAttribute(mcall_biallelic_groups_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if ( e != cudaSuccess ) return e;
    mcall_biallelic_groups_kernel<<<grid, BG_WARPS*32, smem, st>>>(a, (int)wb, (int)bg_buf_bytes(a.nsmpl));
    return cudaGetLastError();
}

}   // namespace mcb
