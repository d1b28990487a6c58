/*  mcall_triallelic.cu -- warp-per-site kernel of the 3-allele class (int32 PLs, one sample group, every sample diploid,
 *  GT + GQ + trimmed PL all requested, no GP, no -A, an even sample count whose byte-packed copy fits a warp's share of
 *  shared memory).
 *
 *  Same algorithm, numerics and decision code as the CTA-per-site kernel of mcall_multi.cu (the shared parts live in
 *  mcall_multi.cuh); what differs is the mapping, which is the one of the two-allele kernel (mcall_biallelic.cu):
 *
 *    - ONE WARP owns one site: no block barrier, warps of a CTA share only the read-only tables.  The serial part of a
 *      site (allele-set decision, set-up of the next site) stalls its own warp only while the other resident warps keep
 *      issuing; in the CTA kernel a third of every warp's time went to the block barriers around that serial part.
 *    - phase 1 reads the site's PL block straight from global memory, two adjacent samples (12 int32 = 3 x 128 bit) per
 *      lane and iteration with an L2 prefetch TW_PF_DIST iterations ahead.  It keeps one plain double product per allele
 *      set and one of the normalisers (exponents split off every MM_RENORM iterations, partials reduced with shuffles) and
 *      leaves a 6-byte packed row per sample in the warp's buffer (15 KB at 2,504 samples: 2 CTAs x 7 warps per SM).
 *    - no row of normalisers: "has data" is "a packed byte is non-zero" (PL = 0,..,0 carries none), rows that still hold
 *      sentinels are known from the escape list, and the literal FP64 path of phase 2 recomputes a sample's normaliser
 *      from its packed bytes in the order of phase 1, so it is bit-identical to the one phase 1 multiplied in.
 *    - a sample with a value outside 0..255 is packed as no-data and listed (up to MM_ESC_CAP per site); mm_decide
 *      evaluates the list one sample per lane with the general per-sample code.  List overflow, a PL >= 256 after the
 *      fill and every outcome phase 2 has no straight-line code for send the site to the general kernel (fallback list).
 *    - phase 2: REF only / the pair {REF,b} / the triple {REF,b,c}, float32 screen then the literal FP64 call
 *      (mcall_device.cuh); allele counts in 16-bit fields (a warp counts up to 2 x nsmpl alleles).
 */

#include "mcall_multi.cuh"

namespace mcb {

#ifndef TW_MAXWARP
#define TW_MAXWARP   7                  /* warps per CTA the kernel is compiled for */
#endif
#define TW_MINCTA    2                  /* CTAs per SM it is compiled for: 448 threads => at most 144 registers */
#ifndef TW_PF_DIST
#define TW_PF_DIST   4                  /* L2 prefetch distance of phase 1, in iterations of 64 samples (1,536 bytes) */
#endif

struct TWRec                            /* per warp, in front of its packed buffer; the member names are the ones mm_decide / mm_finalize use */
{
    MMSetup<3> su;
    double   max_qual, lk_sum, ref_lk, gap, lse;
    double   q[3];
    float    scr_w[8];                  /* screen weights of the slots 0..5; [6] != 0: this site stays on the literal path */
    int4     slot_out[8];               /* {gt0, gt1, AC increment lo, hi} of slot k */
    uint32_t als_new, flags;
    int      path;                      /* 0 nothing to do, 1 REF only, 2 pair {REF,b}, 3 triple {REF,b,c} */
    int      nals_new, ref_gt, site;
    long long out_off;
    int      als_map[3];
    int      jgt[6];                    /* byte offset of slot k's genotype in a packed row */
    int      ac[8];
    int      nesc;                      /* samples listed for the general path (> MM_ESC_CAP: overflowed) */
    unsigned short esc[MM_ESC_CAP];
};
constexpr int TW_REC_BYTES = (int)((sizeof(TWRec) + 15) & ~(size_t)15);
static_assert(offsetof(TWRec, scr_w) % 16 == 0 && offsetof(TWRec, slot_out) % 16 == 0, "read with 128-bit loads");

__device__ __forceinline__ void tw_prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" :: "l"(p)); }

/*  a sample's normaliser from its packed row: the sum of phase 1 (and of mm_slow_sample), same order, same roundings  */
static __device__ __noinline__ double tw_row_sum(uint32_t row_s, uint32_t pl2p_s)
{
    double s = lds64c(pl2p_s + 8u*mm_ldsu8(row_s));
    #pragma unroll
    for (int j=1; j<6; j++) s = __dadd_rn(s, lds64c(pl2p_s + 8u*mm_ldsu8(row_s + (uint32_t)j)));
    return s;
}

__global__ void __launch_bounds__(TW_MAXWARP*32, TW_MINCTA) mcall_triallelic_warp_kernel(const KArgs a, int warp_bytes)
{
    using S = Shape<3>;
    constexpr int G = S::G, NPAIR = S::NPAIR, NSET = MMGeom<3>::NSET, NACC = MMGeom<3>::NACC;
    constexpr double LN2 = 0.693147180559945309417232121458;
    BWTables &tb = *reinterpret_cast<BWTables*>(mcb_smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t sbase = smem_base();
    const uint32_t pl2p_s = sbase + (uint32_t)offsetof(BWTables, pl2p), thr_s = sbase + (uint32_t)offsetof(BWTables, gq_thr);
    const uint32_t plf_s = sbase + (uint32_t)offsetof(BWTables, scr) + (uint32_t)offsetof(ScreenTabs, plf);
    const uint32_t gqw_s = sbase + (uint32_t)offsetof(BWTables, scr) + (uint32_t)offsetof(ScreenTabs, gqw);
    const size_t wofs = align128(sizeof(BWTables)) + (size_t)warp*(size_t)warp_bytes;
    TWRec &rec = *reinterpret_cast<TWRec*>(mcb_smem + wofs);
    const uint32_t rec_s = sbase + (uint32_t)wofs, pack_s = rec_s + (uint32_t)TW_REC_BYTES;
    const uint32_t q_s = rec_s + (uint32_t)offsetof(TWRec, q), jgt_s = rec_s + (uint32_t)offsetof(TWRec, jgt);
    const uint32_t slot_s = rec_s + (uint32_t)offsetof(TWRec, slot_out), scrw_s = rec_s + (uint32_t)offsetof(TWRec, scr_w);
    const uint32_t cfp_s = rec_s + (uint32_t)offsetof(TWRec, su) + (uint32_t)offsetof(MMSetup<3>, cfp);
    const uint32_t cft_s = rec_s + (uint32_t)offsetof(TWRec, su) + (uint32_t)offsetof(MMSetup<3>, cft);

    for (int i=tid; i<256; i+=blockDim.x) tb.pl2p[i] = a.tab->pl2p[i];
    for (int i=tid; i<130; i+=blockDim.x) tb.gq_thr[i] = i<128 ? a.tab->gq_thr[i] : -1.0;
    screen_tabs_fill(&tb.scr, a.tab, tid, blockDim.x);
    __syncthreads();            /* the only block barrier: from here on every warp runs on its own */

    const int nsmpl = a.nsmpl, npair = nsmpl >> 1, niter = (npair + 31) >> 5;
    const int nsites = *a.site_count;
    if ( lane==0 ) rec.su.isite = atomicAdd(a.work_counter, 1);
    mm_setup<3>(&rec.su, a, lane, nsites);

    for (;;)
    {
        const MMSetup<3> &su = rec.su;
        if ( su.isite >= nsites ) break;
        const int32_t *site_pl = reinterpret_cast<const int32_t*>(a.pl) + su.pl_off;
        const int4 *pl4 = reinterpret_cast<const int4*>(site_pl);
        const char *site_end = reinterpret_cast<const char*>(site_pl) + (size_t)nsmpl*(G*4);
        const uint32_t live = su.live;
        const int unseen = su.unseen;
        double cfr[NPAIR*3 + 6];
        #pragma unroll
        for (int k=0; k<NPAIR; k++)
            #pragma unroll
            for (int c=0; c<3; c++) cfr[k*3+c] = lds64(cfp_s + 8u*(uint32_t)(k*4+c));
        #pragma unroll
        for (int c=0; c<6; c++) cfr[NPAIR*3+c] = lds64(cft_s + 8u*(uint32_t)c);
        if ( lane==0 ) rec.nesc = 0;
        __syncwarp();

        /* =========================== phase 1: site reduction ==================================== */
        const char *pf = reinterpret_cast<const char*>(site_pl) + 128*lane;
        if ( lane < 12 )
        {
            #pragma unroll
            for (int d=1; d<TW_PF_DIST; d++) if ( pf + d*1536 < site_end ) tw_prefetch_l2(pf + d*1536);
        }
        pf += TW_PF_DIST*1536;
        double accM[NACC]; int accE[NACC];
        int plsum[3] = {0,0,0};
        int n0 = 0, since = 0;
        #pragma unroll
        for (int k=0; k<NACC; k++) { accM[k] = 1.0; accE[k] = 0; }
        #pragma unroll 1
        for (int it=0; it<niter; it++)
        {
            if ( lane < 12 && pf < site_end ) tw_prefetch_l2(pf);      /* 12 lines of 128 bytes = the 64 samples of iteration it+TW_PF_DIST */
            pf += 1536;
            const int pr = it*32 + lane;                            /* this lane's samples: 2pr, 2pr+1 */
            if ( pr >= npair ) continue;
            const int4 v0 = __ldg(pl4 + 3*pr), v1 = __ldg(pl4 + 3*pr + 1), v2 = __ldg(pl4 + 3*pr + 2);
            int x[2*G] = { v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w, v2.x, v2.y, v2.z, v2.w };
            int orA = 0, orB = 0;
            #pragma unroll
            for (int i=0; i<G; i++) { orA |= x[i]; orB |= x[G+i]; }
            if ( (unsigned)(orA | orB) > 255u )
            {
                /* a missing / vector_end value or a PL >= 256: listed for the general path, and through the loop below as a
                   no-data sample (its constant factor is divided out with the other no-data samples) */
                if ( (unsigned)orA > 255u )
                {
                    const int pos = atomicAdd(&rec.nesc, 1);
                    if ( pos < MM_ESC_CAP ) rec.esc[pos] = (unsigned short)(2*pr);
                    #pragma unroll
                    for (int i=0; i<G; i++) asm volatile("mov.s32 %0, 0;" : "+r"(x[i]));      /* in place: the common path keeps its registers */
                    orA = 0;
                }
                if ( (unsigned)orB > 255u )
                {
                    const int pos = atomicAdd(&rec.nesc, 1);
                    if ( pos < MM_ESC_CAP ) rec.esc[pos] = (unsigned short)(2*pr + 1);
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
            /* PL = 0,..,0: no data (mcall.c:529-537), multiplied in like any other sample and divided out per site */
            n0 += (orA==0) + (orB==0);
            #pragma unroll
            for (int k=0; k<3; k++) plsum[k] += x[hom_idx(k)] + x[G+hom_idx(k)];       /* mcall.c:607-611 */
            accM[NSET] = __dmul_rn(accM[NSET], __dmul_rn(sumA, sumB));
            #pragma unroll
            for (int xx=1; xx<3; xx++)
                #pragma unroll
                for (int yy=0; yy<xx; yy++)
                {
                    const int k = pair_idx(xx,yy);
                    if ( live & (1u<<k) )
                    {
                        const double c0 = cfr[k*3], c1 = cfr[k*3+1], c2 = cfr[k*3+2];
                        const double vA = fma(c2, pA[gt_idx(xx,yy)], fma(c1, pA[hom_idx(yy)], c0*pA[hom_idx(xx)]));
                        const double vB = fma(c2, pB[gt_idx(xx,yy)], fma(c1, pB[hom_idx(yy)], c0*pB[hom_idx(xx)]));
                        accM[k] = __dmul_rn(accM[k], __dmul_rn(vA, vB));
                    }
                }
            if ( live & (1u<<NPAIR) )          /* the triple {2,1,0} */
            {
                const double *c = cfr + NPAIR*3;
                const double vA = fma(c[5], pA[gt_idx(1,0)], fma(c[4], pA[gt_idx(2,0)], fma(c[3], pA[gt_idx(2,1)],
                                  fma(c[2], pA[hom_idx(0)], fma(c[1], pA[hom_idx(1)], c[0]*pA[hom_idx(2)])))));
                const double vB = fma(c[5], pB[gt_idx(1,0)], fma(c[4], pB[gt_idx(2,0)], fma(c[3], pB[gt_idx(2,1)],
                                  fma(c[2], pB[hom_idx(0)], fma(c[1], pB[hom_idx(1)], c[0]*pB[hom_idx(2)])))));
                accM[NPAIR] = __dmul_rn(accM[NPAIR], __dmul_rn(vA, vB));
            }
            const uint32_t prow_s = pack_s + 12u*(uint32_t)pr;
            mm_sts32(prow_s,      mm_pack4(x[0],x[1],x[2],x[3]));
            mm_sts32(prow_s + 4u, mm_pack4(x[4],x[5],x[6],x[7]));
            mm_sts32(prow_s + 8u, mm_pack4(x[8],x[9],x[10],x[11]));
            if ( ++since == MM_RENORM )         /* ten more samples in every product: split the exponents off before anything can underflow */
            {
                #pragma unroll
                for (int k=0; k<NACC; k++) acc_renorm(accM[k], accE[k]);
                since = 0;
            }
        }

        /* ---- warp reduction: mantissa products (32 values in [1,2) stay below 2^32), exponent and integer sums */
        #pragma unroll
        for (int k=0; k<NACC; k++) acc_renorm(accM[k], accE[k]);
        #pragma unroll
        for (int off=16; off; off>>=1)
        {
            #pragma unroll
            for (int k=0; k<NACC; k++)
            {
                accM[k] = __dmul_rn(accM[k], __shfl_xor_sync(0xffffffffu, accM[k], off));
                accE[k] += __shfl_xor_sync(0xffffffffu, accE[k], off);
            }
            #pragma unroll
            for (int k=0; k<3; k++) plsum[k] += __shfl_xor_sync(0xffffffffu, plsum[k], off);
            n0 += __shfl_xor_sync(0xffffffffu, n0, off);
        }
        /* lane 31: the normalisers, lanes 3..6: the allele sets (mm_decide's layout) */
        double tl = 0;
        {
            double M = accM[NSET]; int E = accE[NSET];
            #pragma unroll
            for (int k=0; k<NSET; k++) if ( lane==3+k ) { M = accM[k]; E = accE[k]; }
            acc_renorm(M, E);
            if ( lane==31 || (lane>=3 && lane<3+NSET && ((live >> (lane-3)) & 1u)) ) tl = mm_log(M) + (double)E*LN2;
        }
        const long long ps = lane==0 ? plsum[0] : (lane==1 ? plsum[1] : (lane==2 ? plsum[2] : 0));
        __syncwarp();               /* the list and the packed rows of every lane are visible */
        const int nesc_raw = rec.nesc;
        const int my_esc = lane < min(nesc_raw, MM_ESC_CAP) ? (int)rec.esc[lane] : 0;
        const bool my_raw = mm_decide<3,16>(&rec, &su, a, lane, pl2p_s, pack_s + (uint32_t)(my_esc*6), nesc_raw, site_pl + (size_t)my_esc*G, nullptr, tl, n0, ps);
        __syncwarp();

        /* the next site is claimed now: the atomic's latency hides behind phase 2.  Its set-up (site_list, then qs / pl_off /
           unseen / prior: two dependent L2 round trips and four logs) stays after phase 2: loading those fields here would stall
           this warp on the claim's result right away.  Either way only the owning warp waits while the other resident warps
           issue; in the two-allele kernel an earlier claim measured no gain (profiles/r02_biallelic_base_claim_ab.log). */
        int next = 0;
        if ( lane==0 ) next = atomicAdd(a.work_counter, 1);

        /* =========================== phase 2: per-sample genotypes ============================== */
        /* a pair of samples is 12 bytes at pack_s + 12 pr: words W0 = A0..A3, W1 = A4 A5 B0 B1, W2 = B2..B5 */
        const int path = rec.path;
        if ( path==1 )              /* REF only: mcall_set_ref_genotypes (mcall.c:713-743); the PL tag is dropped */
        {
            int2 *out_gt = reinterpret_cast<int2*>(a.gt) + (size_t)rec.site*nsmpl;
            int32_t *out_gq = a.gq + (size_t)rec.site*nsmpl;
            int called = 0;
            #pragma unroll 1
            for (int pr=lane; pr<npair; pr+=32)
            {
                const uint32_t r = pack_s + 12u*(uint32_t)pr;
                const uint32_t W0 = (uint32_t)lds32(r), W1 = (uint32_t)lds32(r + 4u), W2 = (uint32_t)lds32(r + 8u);
                const bool has0 = (W0 | (W1 & 0xffffu)) != 0, has1 = ((W1 >> 16) | W2) != 0;
                const int g0 = has0 ? MCB_GT_UNPHASED(0) : MCB_GT_MISSING, g1 = has1 ? MCB_GT_UNPHASED(0) : MCB_GT_MISSING;
                called += (int)has0 + (int)has1;
                mm_stg128(out_gt + 2*(size_t)pr, g0, g0, g1, g1);
                mm_stg64(out_gq + 2*(size_t)pr, 0, 0);
            }
            #pragma unroll
            for (int off=16; off; off>>=1) called += __shfl_xor_sync(0xffffffffu, called, off);
            if ( lane==0 ) rec.ac[0] = 2*called;
        }
        else if ( path==2 )         /* the pair {REF, b}, both kept: new genotypes 0/0, 0/1, 1/1 are slots 0, 1, 2 */
        {
            int2 *out_gt = reinterpret_cast<int2*>(a.gt) + (size_t)rec.site*nsmpl;
            int32_t *out_gq = a.gq + (size_t)rec.site*nsmpl;
            int32_t *out_pl = a.out_pl + rec.out_off;
            float w0, w1, w2, wn;
            asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(w0), "=f"(w1), "=f"(w2), "=f"(wn) : "r"(scrw_s));
            asm volatile("ld.shared.f32 %0, [%1+24];" : "=f"(wn) : "r"(scrw_s));
            const bool noscr = wn != 0.f;
            const uint32_t j0 = (uint32_t)rec.jgt[0], j1 = (uint32_t)rec.jgt[1], j2 = (uint32_t)rec.jgt[2];
            int f_alt = 0, f_called = 0;
            #pragma unroll 1
            for (int pr=lane; pr<npair; pr+=32)
            {
                const uint32_t rA = pack_s + 12u*(uint32_t)pr;
                const uint32_t W0 = (uint32_t)lds32(rA), W1 = (uint32_t)lds32(rA + 4u), W2 = (uint32_t)lds32(rA + 8u);
                const uint32_t a0 = __byte_perm(W0, W1, j0) & 0xffu, b0 = __byte_perm(W0, W1, j1) & 0xffu, c0 = __byte_perm(W0, W1, j2) & 0xffu;
                const uint32_t a1 = __byte_perm(W1, W2, j0 + 2u) & 0xffu, b1 = __byte_perm(W1, W2, j1 + 2u) & 0xffu, c1 = __byte_perm(W1, W2, j2 + 2u) & 0xffu;
                int k0, k1, g0, g1;
                const bool ok0 = screen2_call(a0, b0, c0, w0, w1, w2, plf_s, gqw_s, k0, g0);
                const bool ok1 = screen2_call(a1, b1, c1, w0, w1, w2, plf_s, gqw_s, k1, g1);
                const bool has0 = (W0 | (W1 & 0xffffu)) != 0, has1 = ((W1 >> 16) | W2) != 0;      /* PL=0,..,0 / no data: ./. and GQ 0 */
                if ( (!ok0 || noscr) && has0 ) { const int e = mm_fast2_exact(a0, b0, c0, tw_row_sum(rA, pl2p_s), q_s, pl2p_s, thr_s); k0 = e & 255; g0 = e >> 8; }
                if ( (!ok1 || noscr) && has1 ) { const int e = mm_fast2_exact(a1, b1, c1, tw_row_sum(rA + 6u, pl2p_s), q_s, pl2p_s, thr_s); k1 = e & 255; g1 = e >> 8; }
                /* new alleles 0 and 1: GT codes 2 and 4, slot index = copies of allele 1 */
                const int x0 = has0 ? (k0==2 ? 4 : 2) : 0, y0 = has0 ? (k0 ? 4 : 2) : 0;
                const int x1 = has1 ? (k1==2 ? 4 : 2) : 0, y1 = has1 ? (k1 ? 4 : 2) : 0;
                f_alt += (has0 ? k0 : 0) + (has1 ? k1 : 0); f_called += (int)has0 + (int)has1;
                mm_stg128(out_gt + 2*(size_t)pr, x0, y0, x1, y1);
                mm_stg64(out_gq + 2*(size_t)pr, has0 ? g0 : 0, has1 ? g1 : 0);
                int32_t *dst = out_pl + 6*(size_t)pr;           /* mcall.c:1158-1194: the kept genotypes are the three slots */
                mm_stg64(dst, (int)a0, (int)b0); mm_stg64(dst + 2, (int)c0, (int)a1); mm_stg64(dst + 4, (int)b1, (int)c1);
            }
            #pragma unroll
            for (int off=16; off; off>>=1) { f_alt += __shfl_xor_sync(0xffffffffu, f_alt, off); f_called += __shfl_xor_sync(0xffffffffu, f_called, off); }
            if ( lane==0 ) { rec.ac[0] = 2*f_called - f_alt; rec.ac[1] = f_alt; }
            __syncwarp();           /* a listed row that still holds sentinels: its output row carries them (after the stores above) */
            if ( my_raw )
            {
                const int jg[3] = { (int)j0, (int)j1, (int)j2 };
                mm_raw_pl_row<3>(site_pl + (size_t)my_esc*G, unseen, jg, 3, out_pl + 3*(size_t)my_esc);
            }
        }
        else if ( path==3 )         /* the triple {REF, b, c}, all kept: slot k = new genotype k */
        {
            int2 *out_gt = reinterpret_cast<int2*>(a.gt) + (size_t)rec.site*nsmpl;
            int32_t *out_gq = a.gq + (size_t)rec.site*nsmpl;
            int32_t *out_pl = a.out_pl + rec.out_off;
            float w[6], wn;
            asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(w[0]), "=f"(w[1]), "=f"(w[2]), "=f"(w[3]) : "r"(scrw_s));
            asm volatile("ld.shared.v2.f32 {%0,%1}, [%2+16];" : "=f"(w[4]), "=f"(w[5]) : "r"(scrw_s));
            asm volatile("ld.shared.f32 %0, [%1+24];" : "=f"(wn) : "r"(scrw_s));
            const bool noscr = wn != 0.f;
            uint32_t jg[6];
            #pragma unroll
            for (int k=0; k<6; k++) jg[k] = (uint32_t)rec.jgt[k];
            unsigned long long acc = 0;     /* AC: 16-bit counters, new allele j at bits [16j,16j+16); a warp counts at most 2 x nsmpl */
            #pragma unroll 1
            for (int pr=lane; pr<npair; pr+=32)
            {
                const uint32_t rA = pack_s + 12u*(uint32_t)pr;
                const uint32_t W0 = (uint32_t)lds32(rA), W1 = (uint32_t)lds32(rA + 4u), W2 = (uint32_t)lds32(rA + 8u);
                uint32_t vA[6], vB[6];
                #pragma unroll
                for (int k=0; k<6; k++) { vA[k] = __byte_perm(W0, W1, jg[k]) & 0xffu; vB[k] = __byte_perm(W1, W2, jg[k] + 2u) & 0xffu; }
                int32_t *dst = out_pl + 12*(size_t)pr;
                mm_stg128(dst,     (int)vA[0], (int)vA[1], (int)vA[2], (int)vA[3]);
                mm_stg128(dst + 4, (int)vA[4], (int)vA[5], (int)vB[0], (int)vB[1]);
                mm_stg128(dst + 8, (int)vB[2], (int)vB[3], (int)vB[4], (int)vB[5]);
                int k0, k1, g0, g1;
                const bool ok0 = screen3_call(vA, w, plf_s, gqw_s, k0, g0);
                const bool ok1 = screen3_call(vB, w, plf_s, gqw_s, k1, g1);
                const bool has0 = (W0 | (W1 & 0xffffu)) != 0, has1 = ((W1 >> 16) | W2) != 0;
                if ( (!ok0 || noscr) && has0 ) { const int e = mm_fast3_exact(rA, jgt_s, tw_row_sum(rA, pl2p_s), q_s, pl2p_s, thr_s); k0 = e & 255; g0 = e >> 8; }
                if ( (!ok1 || noscr) && has1 ) { const int e = mm_fast3_exact(rA + 6u, jgt_s, tw_row_sum(rA + 6u, pl2p_s), q_s, pl2p_s, thr_s); k1 = e & 255; g1 = e >> 8; }
                const int4 o0 = lds128(slot_s + 16u*(uint32_t)(has0 ? k0 : 6));
                const int4 o1 = lds128(slot_s + 16u*(uint32_t)(has1 ? k1 : 6));
                acc += ((unsigned long long)(uint32_t)o0.z | ((unsigned long long)(uint32_t)o0.w << 32))
                     + ((unsigned long long)(uint32_t)o1.z | ((unsigned long long)(uint32_t)o1.w << 32));
                mm_stg128(out_gt + 2*(size_t)pr, o0.x, o0.y, o1.x, o1.y);
                mm_stg64(out_gq + 2*(size_t)pr, has0 ? g0 : 0, has1 ? g1 : 0);
            }
            #pragma unroll
            for (int off=16; off; off>>=1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
            if ( lane==0 )
            {
                #pragma unroll
                for (int j=0; j<3; j++) rec.ac[j] = (int)((acc >> (16*j)) & 0xffffu);
            }
            __syncwarp();
            if ( my_raw )
            {
                int jgi[6];
                #pragma unroll
                for (int k=0; k<6; k++) jgi[k] = (int)jg[k];
                mm_raw_pl_row<3>(site_pl + (size_t)my_esc*G, unseen, jgi, 6, out_pl + 6*(size_t)my_esc);
            }
        }
        __syncwarp();
        if ( lane==0 )
        {
            if ( path>0 ) mm_finalize<3>(&rec, a);
            rec.su.isite = next;
        }
        mm_setup<3>(&rec.su, a, lane, nsites);
    }
}

/* ------------------------------------------------------------------------------------------------
 *  launcher
 * ---------------------------------------------------------------------------------------------- */
size_t triallelic_warp_bytes(int nsmpl)
{
    return (size_t)TW_REC_BYTES + (((size_t)6*(size_t)nsmpl + 15) & ~(size_t)15);
}
size_t triallelic_smem_bytes(int nsmpl, int nwarp)
{
    return align128(sizeof(BWTables)) + (size_t)nwarp*triallelic_warp_bytes(nsmpl);
}
int triallelic_max_warps() { return TW_MAXWARP; }
int triallelic_ctas_per_sm() { return TW_MINCTA; }

cudaError_t launch_triallelic_warp_kernel(const KArgs &a, int grid, int nwarp, cudaStream_t st)
{
    const size_t smem = triallelic_smem_bytes(a.nsmpl, nwarp);
    cudaError_t e = cudaFuncSetAttribute(mcall_triallelic_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if ( e != cudaSuccess ) return e;
    mcall_triallelic_warp_kernel<<<grid, nwarp*32, smem, st>>>(a, (int)triallelic_warp_bytes(a.nsmpl));
    return cudaGetLastError();
}

}   // namespace mcb
