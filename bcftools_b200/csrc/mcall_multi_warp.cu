/*  mcall_multi_warp.cu -- warp-per-site kernel of the 4-allele class (int32 PLs, one sample group, every sample diploid,
 *  GT + GQ + trimmed PL all requested, no GP, no -A, an even sample count).
 *
 *  The mapping, phase structure and decision code of the 3-allele warp kernel (mcall_triallelic.cu; the shared parts live in
 *  mcall_multi.cuh): one warp owns one site, claims the next one when phase 2 starts, and the only block barrier follows the
 *  table fill.  What differs is the size of a site's byte-packed copy, 10 bytes per sample for 10 genotypes:
 *
 *    - HEAD AND TAIL: the first `head` samples of the copy live in the warp's shared-memory buffer, the rest in a per-warp row
 *      of global scratch written with the evict_last policy, so that it stays in L2 until phase 2 reads it back (the CTA
 *      kernel keeps its row of normalisers that way).  With the whole copy in shared memory a 2,504-sample site would leave
 *      room for 8 warps per SM; the split gives 16.  The head is a multiple of 64 samples: an iteration of either phase is
 *      in the head or in the tail for the whole warp.
 *    - phase 1: two adjacent samples per lane and iteration (80 bytes, 128-bit loads).  One plain double product per live
 *      allele set and one of the normalisers, exponents split off every ten samples, partials reduced with shuffles.  The
 *      coefficients are read from the warp's MMSetup in shared memory with 128-bit loads, once per pair of samples.
 *    - no row of normalisers: "has data" is "a packed byte is non-zero", and the literal FP64 path of phase 2 recomputes a
 *      sample's normaliser from its packed bytes in the order of phase 1 (bit-identical).
 *    - phase 2: REF only / the pair {REF,b} / the triple {REF,b,c}, two samples per lane, 16-bit allele counters; every other
 *      outcome goes to the fallback list that the general kernel walks.
 *
 *  The 5-allele class stays on the CTA kernel: the same scheme for it (16-byte rows, 168 registers with spills at 12 warps
 *  per SM, or 222 registers at 8) measured slower than the CTA kernel on the bench step (DESIGN.md section 4b'').
 */

#include "mcall_multi.cuh"

namespace mcb {

#define MW_MINCTA    2                  /* CTAs per SM the kernel is compiled for */
#ifndef MW_PF_DIST
#define MW_PF_DIST   4                  /* L2 prefetch distance of phase 1, in iterations */
#endif

#define MW_MAXWARP   8                  /* warps per CTA: 2 x 8 warps per SM at <= 128 registers */

template<int NALS> struct MWRec         /* per warp, in front of its packed buffer; the member names are the ones mm_decide / mm_finalize use */
{
    MMSetup<NALS> su;
    double   max_qual, lk_sum, ref_lk, gap, lse;
    double   q[3];
    float    scr_w[8];                  /* screen weights of the slots 0..5; [6] != 0: this site stays on the literal path */
    int4     slot_out[8];               /* {gt0, gt1, AC increment lo, hi} of slot k */
    uint32_t als_new, flags;
    int      path;                      /* 0 nothing to do, 1 REF only, 2 pair {REF,b}, 3 triple {REF,b,c} */
    int      nals_new, ref_gt, site;
    long long out_off;
    int      als_map[NALS];
    int      jgt[6];                    /* byte offset of slot k's genotype in a packed row */
    int      ac[8];
    int      nesc;                      /* samples listed for the general path (> MM_ESC_CAP: overflowed) */
    unsigned short esc[MM_ESC_CAP];
};
template<int NALS> __host__ __device__ constexpr int mw_rec_bytes() { return (int)((sizeof(MWRec<NALS>) + 15) & ~(size_t)15); }

__device__ __forceinline__ void mw_lds_f64x2(uint32_t a, double &x, double &y)
{
    asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(x), "=d"(y) : "r"(a));
}
__device__ __forceinline__ void mw_prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" :: "l"(p)); }
__device__ __forceinline__ void mw_stg32_last(void *p, uint32_t v, uint64_t pol)
{
    asm volatile("st.global.L2::cache_hint.b32 [%0], %1, %2;" :: "l"(p), "r"(v), "l"(pol) : "memory");
}

/*  a sample's normaliser from its packed row: the sum of phase 1 (and of mm_slow_sample), same order, same roundings  */
template<int G>
static __device__ __noinline__ double mw_row_sum(const uint8_t *row, uint32_t pl2p_s)
{
    double s = lds64c(pl2p_s + 8u*(uint32_t)row[0]);
    #pragma unroll
    for (int j=1; j<G; j++) s = __dadd_rn(s, lds64c(pl2p_s + 8u*(uint32_t)row[j]));
    return s;
}

/*  "has data" of the two samples of a packed pair row, 20 bytes, 4-byte aligned: A = bytes 0..9, B = 10..19
 *  (PL = 0,..,0 and rows without data are all zero bytes)  */
__device__ __forceinline__ void mw_has(const uint8_t *rA, bool &has0, bool &has1)
{
    const uint32_t *w = reinterpret_cast<const uint32_t*>(rA);
    const uint32_t W0 = w[0], W1 = w[1], W2 = w[2], W3 = w[3], W4 = w[4];
    has0 = (W0 | W1 | (W2 & 0xffffu)) != 0; has1 = ((W2 >> 16) | W3 | W4) != 0;
}

template<int NALS>
__global__ void __launch_bounds__(MW_MAXWARP*32, MW_MINCTA)
mcall_multi_warp_kernel(const KArgs a, int warp_bytes, int head, uint8_t *tail_g, long long tail_bytes)
{
    using S = Shape<NALS>;
    using GE = MMGeom<NALS>;
    constexpr int G = S::G, NPAIR = S::NPAIR, NSET = GE::NSET, NACC = GE::NACC, RS = GE::RS;
    constexpr int SPL = 2, REC = mw_rec_bytes<NALS>();
    constexpr int IT_SMPL = 32*SPL, IT_BYTES = IT_SMPL*G*4, IT_LINES = IT_BYTES/128;
    constexpr int RENORM = 10/SPL;      /* iterations between exponent splits: ten more samples in every product */
    static_assert(NALS==4 && RS==10, "the 20-byte pair rows of mw_has and the stores below");
    static_assert(IT_BYTES % 128 == 0 && IT_LINES <= 32, "one prefetch per lane and 128-byte line");
    static_assert(offsetof(MWRec<NALS>, scr_w) % 16 == 0 && offsetof(MWRec<NALS>, slot_out) % 16 == 0, "read with 128-bit loads");
    constexpr double LN2 = 0.693147180559945309417232121458;
    BWTables &tb = *reinterpret_cast<BWTables*>(mcb_smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t sbase = smem_base();
    const uint32_t pl2p_s = sbase + (uint32_t)offsetof(BWTables, pl2p), thr_s = sbase + (uint32_t)offsetof(BWTables, gq_thr);
    const uint32_t plf_s = sbase + (uint32_t)offsetof(BWTables, scr) + (uint32_t)offsetof(ScreenTabs, plf);
    const uint32_t gqw_s = sbase + (uint32_t)offsetof(BWTables, scr) + (uint32_t)offsetof(ScreenTabs, gqw);
    const size_t wofs = align128(sizeof(BWTables)) + (size_t)warp*(size_t)warp_bytes;
    MWRec<NALS> &rec = *reinterpret_cast<MWRec<NALS>*>(mcb_smem + wofs);
    const uint32_t rec_s = sbase + (uint32_t)wofs, pack_s = rec_s + (uint32_t)REC;
    uint8_t *const head_g = mcb_smem + wofs + REC;                 /* the same buffer as a generic pointer */
    uint8_t *const tail_w = tail_g + (size_t)(blockIdx.x*(blockDim.x >> 5) + warp)*(size_t)tail_bytes - (size_t)head*RS;   /* indexed by sample */
    const uint32_t q_s = rec_s + (uint32_t)offsetof(MWRec<NALS>, q), jgt_s = rec_s + (uint32_t)offsetof(MWRec<NALS>, jgt);
    const uint32_t slot_s = rec_s + (uint32_t)offsetof(MWRec<NALS>, slot_out), scrw_s = rec_s + (uint32_t)offsetof(MWRec<NALS>, scr_w);
    const uint32_t cfp_s = rec_s + (uint32_t)offsetof(MWRec<NALS>, su) + (uint32_t)offsetof(MMSetup<NALS>, cfp);
    const uint32_t cft_s = rec_s + (uint32_t)offsetof(MWRec<NALS>, su) + (uint32_t)offsetof(MMSetup<NALS>, cft);
    auto row_of = [&](int s) -> uint8_t* { return (s < head ? head_g : tail_w) + (size_t)s*RS; };   /* the packed row of sample s */

    for (int i=tid; i<256; i+=blockDim.x) tb.pl2p[i] = a.tab->pl2p[i];
    for (int i=tid; i<130; i+=blockDim.x) tb.gq_thr[i] = i<128 ? a.tab->gq_thr[i] : -1.0;
    screen_tabs_fill(&tb.scr, a.tab, tid, blockDim.x);
    __syncthreads();            /* the only block barrier: from here on every warp runs on its own */

    const int nsmpl = a.nsmpl, npair = nsmpl >> 1, niter = (nsmpl + IT_SMPL - 1)/IT_SMPL;
    const int nsites = *a.site_count;
    const uint64_t pol_last = mm_policy_evict_last();
    if ( lane==0 ) rec.su.isite = atomicAdd(a.work_counter, 1);
    mm_setup<NALS>(&rec.su, a, lane, nsites);

    for (;;)
    {
        const MMSetup<NALS> &su = rec.su;
        if ( su.isite >= nsites ) break;
        const int32_t *site_pl = reinterpret_cast<const int32_t*>(a.pl) + su.pl_off;
        const char *site_end = reinterpret_cast<const char*>(site_pl) + (size_t)nsmpl*(G*4);
        const uint32_t live = su.live;
        const int unseen = su.unseen;
        if ( lane==0 ) rec.nesc = 0;
        __syncwarp();

        /* =========================== phase 1: site reduction ==================================== */
        const char *pf = reinterpret_cast<const char*>(site_pl) + 128*lane;
        if ( lane < IT_LINES )
        {
            #pragma unroll
            for (int d=1; d<MW_PF_DIST; d++) if ( pf + d*IT_BYTES < site_end ) mw_prefetch_l2(pf + d*IT_BYTES);
        }
        pf += MW_PF_DIST*IT_BYTES;
        double accM[NACC]; int accE[NACC];
        int plsum[NALS];
        int n0 = 0, since = 0;
        #pragma unroll
        for (int k=0; k<NACC; k++) { accM[k] = 1.0; accE[k] = 0; }
        #pragma unroll
        for (int k=0; k<NALS; k++) plsum[k] = 0;
        #pragma unroll 1
        for (int it=0; it<niter; it++)
        {
            if ( lane < IT_LINES && pf < site_end ) mw_prefetch_l2(pf);       /* the lines of iteration it+MW_PF_DIST */
            pf += IT_BYTES;
            const int s0 = (it*32 + lane)*SPL;                      /* this lane's samples: s0 .. s0+SPL-1 */
            if ( s0 >= nsmpl ) continue;
            int x[SPL*G];
            {
                const int4 *src = reinterpret_cast<const int4*>(site_pl + (size_t)s0*G);
                #pragma unroll
                for (int i=0; i<SPL*G/4; i++) { const int4 v = __ldg(src + i); x[4*i] = v.x; x[4*i+1] = v.y; x[4*i+2] = v.z; x[4*i+3] = v.w; }
            }
            int orv[SPL];
            #pragma unroll
            for (int h=0; h<SPL; h++)
            {
                orv[h] = 0;
                #pragma unroll
                for (int i=0; i<G; i++) orv[h] |= x[h*G+i];
                if ( (unsigned)orv[h] > 255u )
                {
                    /* a missing / vector_end value or a PL >= 256: listed for the general path, and through the loop below as a
                       no-data sample (its constant factor is divided out with the other no-data samples) */
                    const int pos = atomicAdd(&rec.nesc, 1);
                    if ( pos < MM_ESC_CAP ) rec.esc[pos] = (unsigned short)(s0 + h);
                    #pragma unroll
                    for (int i=0; i<G; i++) asm volatile("mov.s32 %0, 0;" : "+r"(x[h*G+i]));     /* in place: the common path keeps its registers */
                    orv[h] = 0;
                }
            }
            double p[SPL][G];
            #pragma unroll
            for (int h=0; h<SPL; h++)
                #pragma unroll
                for (int i=0; i<G; i++) p[h][i] = lds64c(pl2p_s + 8u*(uint32_t)x[h*G+i]);
            double nrm = 1.0;
            #pragma unroll
            for (int h=0; h<SPL; h++)
            {
                double sum = p[h][0];
                #pragma unroll
                for (int i=1; i<G; i++) sum = __dadd_rn(sum, p[h][i]);
                nrm = h ? __dmul_rn(nrm, sum) : sum;
                /* PL = 0,..,0: no data (mcall.c:529-537), multiplied in like any other sample and divided out per site */
                n0 += orv[h]==0;
                #pragma unroll
                for (int k=0; k<NALS; k++) plsum[k] += x[h*G + hom_idx(k)];       /* mcall.c:607-611 */
            }
            accM[NSET] = __dmul_rn(accM[NSET], nrm);
            #pragma unroll
            for (int xx=1; xx<NALS; xx++)
                #pragma unroll
                for (int yy=0; yy<xx; yy++)
                {
                    const int k = pair_idx(xx,yy);
                    if ( live & (1u<<k) )
                    {
                        double c0, c1, c2, c3;
                        mw_lds_f64x2(cfp_s + 32u*(uint32_t)k, c0, c1); mw_lds_f64x2(cfp_s + 32u*(uint32_t)k + 16u, c2, c3);
                        double v = 1.0;
                        #pragma unroll
                        for (int h=0; h<SPL; h++)
                        {
                            const double vh = fma(c2, p[h][gt_idx(xx,yy)], fma(c1, p[h][hom_idx(yy)], c0*p[h][hom_idx(xx)]));
                            v = h ? __dmul_rn(v, vh) : vh;
                        }
                        accM[k] = __dmul_rn(accM[k], v);
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
                            const uint32_t c_s = cft_s + 48u*(uint32_t)k;
                            double c0, c1, c2, c3, c4, c5;
                            mw_lds_f64x2(c_s, c0, c1); mw_lds_f64x2(c_s + 16u, c2, c3); mw_lds_f64x2(c_s + 32u, c4, c5);
                            double v = 1.0;
                            #pragma unroll
                            for (int h=0; h<SPL; h++)
                            {
                                const double vh = fma(c5, p[h][gt_idx(yy,zz)], fma(c4, p[h][gt_idx(xx,zz)], fma(c3, p[h][gt_idx(xx,yy)],
                                                  fma(c2, p[h][hom_idx(zz)], fma(c1, p[h][hom_idx(yy)], c0*p[h][hom_idx(xx)])))));
                                v = h ? __dmul_rn(v, vh) : vh;
                            }
                            accM[NPAIR+k] = __dmul_rn(accM[NPAIR+k], v);
                        }
                    }
            /* the packed copy: shared-memory head or L2-resident tail (warp-uniform: head is a multiple of 64 samples) */
            {
                const uint32_t w0 = mm_pack4(x[0],x[1],x[2],x[3]), w1 = mm_pack4(x[4],x[5],x[6],x[7]), w2 = mm_pack4(x[8],x[9],x[10],x[11]);
                const uint32_t w3 = mm_pack4(x[12],x[13],x[14],x[15]), w4 = mm_pack4(x[16],x[17],x[18],x[19]);
                if ( s0 < head )
                {
                    const uint32_t r = pack_s + (uint32_t)(s0*RS);
                    mm_sts32(r, w0); mm_sts32(r + 4u, w1); mm_sts32(r + 8u, w2); mm_sts32(r + 12u, w3); mm_sts32(r + 16u, w4);
                }
                else
                {
                    uint8_t *r = tail_w + (size_t)s0*RS;
                    mw_stg32_last(r, w0, pol_last); mw_stg32_last(r + 4, w1, pol_last); mw_stg32_last(r + 8, w2, pol_last);
                    mw_stg32_last(r + 12, w3, pol_last); mw_stg32_last(r + 16, w4, pol_last);
                }
            }
            if ( ++since == RENORM )            /* split the exponents off before anything can underflow */
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
            for (int k=0; k<NALS; k++) plsum[k] += __shfl_xor_sync(0xffffffffu, plsum[k], off);
            n0 += __shfl_xor_sync(0xffffffffu, n0, off);
        }
        /* lane 31: the normalisers, lanes NALS..NALS+NSET-1: the allele sets (mm_decide's layout) */
        double tl = 0;
        {
            double M = accM[NSET]; int E = accE[NSET];
            #pragma unroll
            for (int k=0; k<NSET; k++) if ( lane==NALS+k ) { M = accM[k]; E = accE[k]; }
            acc_renorm(M, E);
            if ( lane==31 || (lane>=NALS && lane<NALS+NSET && ((live >> (lane-NALS)) & 1u)) ) tl = mm_log(M) + (double)E*LN2;
        }
        long long ps = 0;
        #pragma unroll
        for (int k=0; k<NALS; k++) if ( lane==k ) ps = plsum[k];
        __syncwarp();               /* the list and the packed rows of every lane are visible */
        const int nesc_raw = rec.nesc;
        const int my_esc = lane < min(nesc_raw, MM_ESC_CAP) ? (int)rec.esc[lane] : 0;
        const bool my_raw = mm_decide<NALS,16>(&rec, &su, a, lane, pl2p_s, row_of(my_esc), nesc_raw, site_pl + (size_t)my_esc*G, nullptr, tl, n0, ps);
        __syncwarp();               /* the rows mm_decide filled for listed samples (written by other lanes) */

        /* the next site is claimed now: the atomic's latency hides behind phase 2 (its set-up follows phase 2, as in mcall_triallelic.cu) */
        int next = 0;
        if ( lane==0 ) next = atomicAdd(a.work_counter, 1);

        /* =========================== phase 2: per-sample genotypes ============================== */
        /* lane takes samples 2pr, 2pr+1 with pr = lane + 32k: the rows phase 1 wrote in iterations 2k/SPL.. of the same block of 64 */
        const int path = rec.path;
        if ( path==1 )              /* REF only: mcall_set_ref_genotypes (mcall.c:713-743); the PL tag is dropped */
        {
            int2 *out_gt = reinterpret_cast<int2*>(a.gt) + (size_t)rec.site*nsmpl;
            int32_t *out_gq = a.gq + (size_t)rec.site*nsmpl;
            int called = 0;
            #pragma unroll 1
            for (int pr=lane; pr<npair; pr+=32)
            {
                bool has0, has1;
                mw_has(row_of(2*pr), has0, has1);
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
                const uint8_t *rA = row_of(2*pr), *rB = rA + RS;
                bool has0, has1;
                mw_has(rA, has0, has1);       /* PL=0,..,0 / no data: ./. and GQ 0 */
                const uint32_t a0 = rA[j0], b0 = rA[j1], c0 = rA[j2], a1 = rB[j0], b1 = rB[j1], c1 = rB[j2];
                int k0, k1, g0, g1;
                const bool ok0 = screen2_call(a0, b0, c0, w0, w1, w2, plf_s, gqw_s, k0, g0);
                const bool ok1 = screen2_call(a1, b1, c1, w0, w1, w2, plf_s, gqw_s, k1, g1);
                if ( (!ok0 || noscr) && has0 ) { const int e = mm_fast2_exact(a0, b0, c0, mw_row_sum<G>(rA, pl2p_s), q_s, pl2p_s, thr_s); k0 = e & 255; g0 = e >> 8; }
                if ( (!ok1 || noscr) && has1 ) { const int e = mm_fast2_exact(a1, b1, c1, mw_row_sum<G>(rB, pl2p_s), q_s, pl2p_s, thr_s); k1 = e & 255; g1 = e >> 8; }
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
                mm_raw_pl_row<NALS>(site_pl + (size_t)my_esc*G, unseen, jg, 3, out_pl + 3*(size_t)my_esc);
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
                const uint8_t *rA = row_of(2*pr), *rB = rA + RS;
                bool has0, has1;
                mw_has(rA, has0, has1);
                uint32_t vA[6], vB[6];
                #pragma unroll
                for (int k=0; k<6; k++) { vA[k] = rA[jg[k]]; vB[k] = rB[jg[k]]; }
                int32_t *dst = out_pl + 12*(size_t)pr;
                mm_stg128(dst,     (int)vA[0], (int)vA[1], (int)vA[2], (int)vA[3]);
                mm_stg128(dst + 4, (int)vA[4], (int)vA[5], (int)vB[0], (int)vB[1]);
                mm_stg128(dst + 8, (int)vB[2], (int)vB[3], (int)vB[4], (int)vB[5]);
                int k0, k1, g0, g1;
                const bool ok0 = screen3_call(vA, w, plf_s, gqw_s, k0, g0);
                const bool ok1 = screen3_call(vB, w, plf_s, gqw_s, k1, g1);
                if ( (!ok0 || noscr) && has0 ) { const int e = mm_fast3_exact(rA, jgt_s, mw_row_sum<G>(rA, pl2p_s), q_s, pl2p_s, thr_s); k0 = e & 255; g0 = e >> 8; }
                if ( (!ok1 || noscr) && has1 ) { const int e = mm_fast3_exact(rB, jgt_s, mw_row_sum<G>(rB, pl2p_s), q_s, pl2p_s, thr_s); k1 = e & 255; g1 = e >> 8; }
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
                mm_raw_pl_row<NALS>(site_pl + (size_t)my_esc*G, unseen, jgi, 6, out_pl + 6*(size_t)my_esc);
            }
        }
        __syncwarp();
        if ( lane==0 )
        {
            if ( path>0 ) mm_finalize<NALS>(&rec, a);
            rec.su.isite = next;
        }
        mm_setup<NALS>(&rec.su, a, lane, nsites);
    }
}

/* ------------------------------------------------------------------------------------------------
 *  launcher
 * ---------------------------------------------------------------------------------------------- */
static size_t mw_warp_bytes(int head) { return (size_t)mw_rec_bytes<4>() + (((size_t)head*(size_t)MMGeom<4>::RS + 15) & ~(size_t)15); }
size_t multi_warp_smem_bytes(int head, int nwarp) { return align128(sizeof(BWTables)) + (size_t)nwarp*mw_warp_bytes(head); }
int multi_warp_max_warps() { return MW_MAXWARP; }
int multi_warp_ctas_per_sm() { return MW_MINCTA; }
int multi_warp_head(int nsmpl, int nwarp, size_t smem_per_cta)
{
    int head = ((nsmpl + 63) & ~63);
    while ( head > 0 && multi_warp_smem_bytes(head, nwarp) > smem_per_cta ) head -= 64;
    return head;
}
size_t multi_warp_tail_bytes(int nsmpl, int head)
{
    return head >= nsmpl ? 0 : (((size_t)(nsmpl - head)*(size_t)MMGeom<4>::RS + 127) & ~(size_t)127);
}

cudaError_t launch_multi_warp_kernel(const KArgs &a, int grid, int nwarp, int head, uint8_t *tail, cudaStream_t st)
{
    const size_t smem = multi_warp_smem_bytes(head, nwarp);
    cudaError_t e = cudaFuncSetAttribute(mcall_multi_warp_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if ( e != cudaSuccess ) return e;
    mcall_multi_warp_kernel<4><<<grid, nwarp*32, smem, st>>>(a, (int)mw_warp_bytes(head), head, tail, (long long)multi_warp_tail_bytes(a.nsmpl, head));
    return cudaGetLastError();
}

}   // namespace mcb
