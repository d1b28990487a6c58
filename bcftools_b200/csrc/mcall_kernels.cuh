/*  mcall_kernels.cuh -- sm_100a kernels of the B200-native `call -m` hot path.
 *
 *  One CTA owns one site (record).  A site's FORMAT/PL block ([nsmpl][G] int32, contiguous) is moved
 *  into shared memory by the bulk-copy engine (cp.async.bulk + mbarrier, "TMA 1-D") in tiles of
 *  TILE samples through an NSTAGE ring, and is consumed twice by the same CTA:
 *
 *    phase 1  "site reduction"   = set_pdg (mcall.c:451-544) + mcall_find_best_alleles (mcall.c:591-710)
 *                                   + QUAL candidates (mcall.c:1546-1561) + trimming maps (mcall.c:547-570)
 *    phase 2  "per-sample genotype" = mcall_call_genotypes incl. GQ (mcall.c:745-886),
 *                                   mcall_set_ref_genotypes (mcall.c:713-743), mcall_trim_and_update_PLs
 *                                   (mcall.c:1158-1194), AC/AN and the final QUAL (mcall.c:1631-1650)
 *
 *  When the whole site fits in the ring the second pass re-reads shared memory; otherwise the tiles are
 *  fetched again and hit L2 (the CTA read them microseconds earlier), so HBM sees each PL byte once.
 *
 *  Numerics (DESIGN.md "numerics"):
 *    phase 2 is a literal FP64 transcription (IEEE divide, no FMA contraction, float32 round trip of
 *    every GP, float32 qsum) => GT / AC / AN / trimmed PL / GQ are bit-exact versus the reference.
 *    GQ's -4.34294*log(1-max/sum) is evaluated with a 127-entry threshold table built on the HOST
 *    with the host libm, so it reproduces glibc's log() rounding instead of CUDA's.
 *    phase 1 replaces "one log() per sample per allele set" by exponent-tracked running products
 *    (one log per allele set per site) and folds the per-sample normaliser 1/sum out of the loop;
 *    the single-allele sets are exact integer PL sums.  Likelihood totals agree with the reference
 *    to ~1e-11 absolute (the reference's own rounding noise is ~1e-10); QUAL within 1e-6 relative;
 *    allele-set near-ties (gap < tie_eps) are flagged per site (MCB_SITE_NEAR_TIE).
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "mcall_b200.h"

namespace mcb {

#define MCB_PL2P_BIG 3300           /* host-built pow(10,-i/10) for i<3300; beyond that glibc's pow() underflows to 0 */

struct DevTables
{
    double pl2p[256];               /* call->pl2p, built on the host with glibc pow (mcall.c:56-61) */
    double gq_thr[128];             /* gq_thr[k] = largest x with (int)(-4.34294*log(x)) >= k, host libm (mcall.c:877) */
    double pl2p_big[MCB_PL2P_BIG];  /* same function for PL >= 256 (mcall.c:472), rare path, read from global */
};

struct KArgs
{
    /* batch (device pointers) */
    const void     *pl;  const int64_t *pl_off;  const uint8_t *nals;  const uint8_t *unseen;
    const uint16_t *ploidy_id;  const float *qs;  const uint8_t *nqs;
    const int32_t  *ad;  const int64_t *ad_off;  const uint8_t *nad;
    const int32_t  *prior_an;  const int32_t *prior_ac;
    /* result (device pointers, may be NULL) */
    int32_t *ret;  uint32_t *als_new;  int8_t *als_map;  float *qual;  int32_t *ac;  int32_t *an;
    uint32_t *site_flags;  double *diag;  int32_t *gt;  int32_t *gq;  float *gp;  int32_t *out_pl;
    int64_t *pl_off_out;  unsigned long long *pl_cursor;     /* compacted PL/GP output (optional) */
    /* context */
    const DevTables *tab;
    const uint8_t *ploidy_tab;  int nploidy;
    const uint32_t *grp_off;  const uint32_t *grp_smpl;  const uint32_t *smpl2grp;  int ngroups;
    const int32_t *site_list;  const int32_t *site_count;      /* the sites of this allele-count class */
    int32_t *work_counter;                                      /* next unclaimed entry of site_list (warp-per-site kernel) */
    /* sites the multi-allelic kernel (mcall_multi.cu) hands back to the general tiled kernel */
    int32_t *fb_list;  int32_t *fb_count;
    double  *mm_sums;                                            /* its per-CTA rows of per-sample normalisers (L2-resident scratch) */
    int nsmpl, max_nals;
    uint32_t flag, output_tags;
    double theta, tie_eps;
    int use_prior;
    int tile_smpl, nstage;
    int exact_phase1;                                           /* literal sample-sequential sums of logs (general, grouped and 6..32 allele kernels) */
    int adj_reserve;                                            /* compacted output: a site flagged MCB_SITE_NEAR_TIE reserves its full-G block */
    int adj_pass;                                               /* second evaluation of the flagged sites: writes into that block in place */
};

}   // namespace mcb

namespace mcb {
/*  launchers implemented in mcall_kernels.cu  */
cudaError_t launch_site_kernel(int nals, bool ploidy, bool gp, int block, int pl_es, const KArgs &a, int grid, size_t ring_bytes, cudaStream_t st);
cudaError_t launch_classify(const uint8_t *nals, int nsites, int32_t *lists, int32_t *counts, int list_stride, int max_nals, int32_t *ret, uint32_t *site_flags, int64_t *pl_off_out, cudaStream_t st);
cudaError_t launch_collect_near_ties(const uint8_t *nals, int nsites, const uint32_t *site_flags, int32_t *lists, int32_t *counts, int list_stride, cudaStream_t st);
cudaError_t launch_unsupported(const int32_t *list, const int32_t *count, int32_t *ret, uint32_t *site_flags, const uint8_t *nals, int64_t *pl_off_out, cudaStream_t st);
cudaError_t site_kernel_occupancy(int nals, bool ploidy, bool gp, int block, int pl_es, size_t ring_bytes, int *blocks_per_sm);
size_t groups_scratch_bytes(int grid, int ngroups, int nsmpl);
cudaError_t launch_groups_kernel(int nals, const KArgs &a, void *scratch, int grid, cudaStream_t st);
void generic_scratch_bytes(int grid, int ngroups, int nsmpl, size_t *grp, size_t *pl, size_t *sum);
cudaError_t launch_generic_kernel(const KArgs &a, void *grp_scratch, void *pl_scratch, void *sum_scratch, int grid, cudaStream_t st);
/*  warp-per-site kernel for biallelic, int32, single-group, GP-less calls (mcall_biallelic.cu)  */
size_t biallelic_smem_bytes(int nsmpl, int nwarp);
int biallelic_max_warps();
int biallelic_ctas_per_sm();
cudaError_t launch_biallelic_warp_kernel(const KArgs &a, bool ploidy, int grid, int nwarp, cudaStream_t st);
/*  CTA-per-site kernel of the 3-5 allele classes over a byte-packed shared-memory copy (mcall_multi.cu)  */
int multi_block_for(int nsmpl);
size_t multi_smem_bytes(int nals, int block, int nsmpl, int nst);
size_t multi_scratch_bytes(int nsmpl, int grid);
cudaError_t multi_kernel_occupancy(int nals, int block, int nsmpl, int nst, int *blocks_per_sm);
cudaError_t launch_multi_kernel(int nals, int block, const KArgs &a, int grid, cudaStream_t st);
/*  warp-per-site kernel of the 3-allele class over the same packed copy (mcall_triallelic.cu)  */
size_t triallelic_smem_bytes(int nsmpl, int nwarp);
int triallelic_max_warps();
int triallelic_ctas_per_sm();
cudaError_t launch_triallelic_warp_kernel(const KArgs &a, int grid, int nwarp, cudaStream_t st);
/*  warp-per-site kernel of the 4-allele class: the first `head` samples of the packed copy in shared memory, the rest in a
 *  per-warp row of L2-resident global scratch (mcall_multi_warp.cu)  */
size_t multi_warp_smem_bytes(int head, int nwarp);
int multi_warp_max_warps();
int multi_warp_ctas_per_sm();
int multi_warp_head(int nsmpl, int nwarp, size_t smem_per_cta);
size_t multi_warp_tail_bytes(int nsmpl, int head);
cudaError_t launch_multi_warp_kernel(const KArgs &a, int grid, int nwarp, int head, uint8_t *tail, cudaStream_t st);
/*  warp-per-site kernel for grouped calling (-G) of two-allele sites (mcall_biallelic_groups.cu)  */
bool biallelic_groups_ok(int nsmpl, int ngroups);
int biallelic_groups_warps();
int biallelic_groups_ctas_per_sm();
cudaError_t launch_biallelic_groups_kernel(const KArgs &a, int grid, cudaStream_t st);
cudaError_t launch_selftest_div(const DevTables *tab, int mode, unsigned long long n, unsigned long long seed, unsigned long long *mismatch, cudaStream_t st);
}
