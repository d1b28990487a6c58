/*  mcall_b200.h -- C-ABI of the B200-native multiallelic caller (`bcftools call -m` hot path).
 *
 *  This is the drop-in boundary.  It replaces, for a BATCH of records, what the
 *  reference does one record at a time behind call.h:131-147
 *      void mcall_init(call_t*);  int mcall(call_t*, bcf1_t*);  void mcall_destroy(call_t*);
 *  (callers: vcfcall.c:697-698, vcfcall.c:1136-1137, vcfcall.c:722-723).
 *
 *  Everything that touches bcf1_t/bcf_hdr_t stays on the host (htslib); what crosses this
 *  boundary is exactly what mcall() obtains from / hands to htslib:
 *      in : FORMAT/PL  (bcf_get_format_int32, mcall.c:1444), INFO/QS (mcall.c:1456) or
 *           FORMAT/AD|QS for -G (mcall.c:1475), -F prior AN/AC (mcall.c:1507-1510),
 *           rec->n_allele (mcall.c:1438), call->unseen (vcfcall.c:1101-1111),
 *           call->ploidy (vcfcall.c:807-825)
 *      out: the return value of mcall(), call->als_new/nals_new/als_map (mcall.c:1546-1577),
 *           rec->qual (mcall.c:1631-1645), AC/AN (mcall.c:1648-1650), GT (mcall.c:1657),
 *           GQ/GP (mcall.c:1620-1623), trimmed PL (mcall.c:1158-1194).
 *
 *  Plain C: pointers and sizes only.  No function here ever calls exit(); all return
 *  0 on success or a negative MCB_E* code (the host wrapper maps that to error(),
 *  version.c:40-47, see INTEGRATION.md).
 */
#ifndef MCALL_B200_H
#define MCALL_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- flags: identical values to call.h:32-39 ------------------------------------------- */
#define MCB_CALL_KEEPALT   (1u<<0)      /* CALL_KEEPALT  (-A) */
#define MCB_CALL_VARONLY   (1u<<1)      /* CALL_VARONLY  (-v) */
#define MCB_CALL_FMT_GQ    (1u<<6)      /* CALL_FMT_GQ   (-a GQ) */
#define MCB_CALL_FMT_GP    (1u<<7)      /* CALL_FMT_GP   (-a GP) */

/* ---- htslib sentinels [htslib vcf.h] ---------------------------------------------------- */
#define MCB_INT32_MISSING     INT32_MIN         /* bcf_int32_missing     */
#define MCB_INT32_VECTOR_END  (INT32_MIN+1)     /* bcf_int32_vector_end  */
#define MCB_FLOAT_MISSING_BITS     0x7F800001u  /* bcf_float_missing     */
#define MCB_FLOAT_VECTOR_END_BITS  0x7F800002u  /* bcf_float_vector_end  */
#define MCB_GT_MISSING        0                 /* bcf_gt_missing        */
#define MCB_GT_UNPHASED(a)    (((a)+1)<<1)      /* bcf_gt_unphased(a)    */

#define MCB_MAX_NALS 32     /* call->als_new is a 32-bit mask; larger sites are skipped, mcall.c:1539-1543 */

/* ---- error codes --------------------------------------------------------------------------- */
#define MCB_OK          0
#define MCB_EINVAL     -1   /* bad argument */
#define MCB_ENOMEM     -2   /* host or device allocation failed */
#define MCB_ECUDA      -3   /* CUDA runtime error (mcb_last_cuda_error() has the text) */
#define MCB_ENODEV     -4   /* no CUDA device: there is NO CPU fallback */
#define MCB_EPL        -5   /* "Wrong number of PL fields" (mcall.c:1445-1446) */
#define MCB_EQS        -6   /* "The QS annotation not present" (mcall.c:1457) / AD missing with -G (mcall.c:1476) */
#define MCB_EPRIOR     -7   /* "Incorrect AN,AC values" (mcall.c:1523) */

/* ---- per-site flag bits reported in mcb_result.site_flags --------------------------------- */
#define MCB_SITE_PL_DROPPED   (1u<<0)   /* REF-only output: FORMAT/PL removed (mcall.c:1583) */
#define MCB_SITE_NEAR_TIE     (1u<<1)   /* two best allele sets closer than params.tie_eps: listed, see DESIGN.md */
#define MCB_SITE_UNSEEN_SEL   (1u<<2)   /* the unseen allele <*> was selected: reference behaviour undefined (SURVEY §8 quirks) */
#define MCB_SITE_TOO_MANY_ALS (1u<<3)   /* n_allele > 32: skipped (mcall.c:1539-1543) */
#define MCB_SITE_NO_QS        (1u<<4)   /* nqs<=0: reference would error() out (mcall.c:1457) */
#define MCB_SITE_PL_RANGE      (1u<<6)   /* a PL > 2500 was seen: likelihoods underflow, parity with the reference not guaranteed */
#define MCB_SITE_BAD_PRIOR     (1u<<7)   /* -F: AN < sum(AC); the reference error()s out (mcall.c:1523) */
#define MCB_SITE_UNSUPPORTED   (1u<<8)   /* site shape not covered by the device kernels (n_allele==0, n_allele > max_nals, > 5 alleles with int16 PLs) */
#define MCB_SITE_REF_GT       (1u<<5)   /* genotypes come from mcall_set_ref_genotypes (mcall.c:1582,1587): no GQ/GP written */
#define MCB_SITE_ADJUDICATED  (1u<<9)   /* near tie evaluated a second time with the literal phase 1 (option "adjudicate"); always
                                           set together with MCB_SITE_NEAR_TIE */

typedef struct mcb_ctx mcb_ctx;     /* opaque; one per GPU, used from one host thread (like call_t).  Calls on one context
                                       must be stream-ordered: mcb_call_device shares work lists and scratch between calls,
                                       so two calls on different streams need an event (or a sync) between them */

/*  What mcall_init() reads from call_t (mcall.c:361-417).  */
typedef struct mcb_params
{
    int32_t  nsmpl;             /* bcf_hdr_nsamples(call->hdr) */
    int32_t  max_nals;          /* stride of the per-site allele arrays (qs, prior_ac, ac, als_map); 1..32 */
    double   theta;             /* call->theta as the driver sets it BEFORE mcall_init (vcfcall.c:933, -P); the
                                   Watterson factor and log() of mcall.c:397-416 are applied inside mcb_init  */
    const uint8_t *init_ploidy; /* call->ploidy[nsmpl] as it is at mcall_init time (vcfcall.c:652-655), NULL = all 2 */
    uint32_t flag;              /* MCB_CALL_KEEPALT | MCB_CALL_VARONLY */
    uint32_t output_tags;       /* MCB_CALL_FMT_GQ | MCB_CALL_FMT_GP */
    int32_t  ngroups;           /* call->nsmpl_grp (mcall.c:250-349); <=1: one pooled group, QS comes from INFO/QS */
    const uint32_t *grp_off;    /* [ngroups+1] offsets into grp_smpl (ignored when ngroups<=1) */
    const uint32_t *grp_smpl;   /* [nsmpl] sample indices, group after group = smpl_grp_t.smpl (call.h:58) */
    int32_t  use_prior;         /* -F prior_AN,prior_AC given (mcall.c:1507) */
    int32_t  device;            /* CUDA device ordinal */
    double   tie_eps;           /* near-tie listing threshold on the allele-set log-likelihood gap; <=0: default 1e-6 */
}
mcb_params;

/*  One batch of R records, structure-of-arrays.  Site i has A_i = nals[i] alleles and
 *  G_i = A_i(A_i+1)/2 diploid genotypes; its PL block is pl + pl_off[i], laid out
 *  [nsmpl][G_i] row-major exactly as bcf_get_format_int32 returns it (mcall.c:1444),
 *  short vectors padded with MCB_INT32_VECTOR_END.  pl_off[i] must be a multiple of 4
 *  (16-byte alignment for bulk copies), and the bytes between the end of a site's block and
 *  the next 16-byte boundary must be READABLE (bulk copies round a tile up to 16 bytes;
 *  their content is ignored) -- also behind the last site of the slab.
 *  nals[i] must not exceed params.max_nals: mcb_call_host returns MCB_EINVAL, mcb_call_device
 *  reports the site as skipped with MCB_SITE_UNSUPPORTED.                               */
typedef struct mcb_batch
{
    int32_t  nsites;
    const int32_t  *pl;         /* PL slab */
    const int64_t  *pl_off;     /* [nsites] int32-unit offset of site i in pl (and in mcb_result.pl) */
    const uint8_t  *nals;       /* [nsites] rec->n_allele */
    const uint8_t  *unseen;     /* [nsites] call->unseen, 0 = none (vcfcall.c:1102) */
    const uint16_t *ploidy_id;  /* [nsites] id given to mcb_set_ploidy, NULL = id 0 for all */
    const float    *qs;         /* [nsites][max_nals] INFO/QS, zero-extended (mcall.c:1458-1464); pooled calling */
    const uint8_t  *nqs;        /* [nsites] number of QS values present, NULL = nals[i] */
    const int32_t  *ad;         /* -G: FORMAT/AD (or QS) slab, site i at ad + ad_off[i], [nsmpl][nad[i]] */
    const int64_t  *ad_off;     /* [nsites] */
    const uint8_t  *nad;        /* [nsites] values per sample in ad (mcall.c:1477) */
    const int32_t  *prior_an;   /* [nsites] -F: AN, <=0 or MCB_INT32_MISSING = absent (mcall.c:1507-1510) */
    const int32_t  *prior_ac;   /* [nsites][max_nals] -F: AC for ALT 1..A-1 in [0..A-2], MCB_INT32_VECTOR_END-terminated */
    int32_t  pl_type;           /* element type of `pl`: 0 or 4 = int32 (bcf_get_format_int32), 2 = int16 = the BCF on-disk
                                   typed vector (BCF_BT_INT16, sentinels INT16_MIN / INT16_MIN+1) shipped as is and widened
                                   on the device.  pl_off stays in ELEMENTS; pl + pl_off[i] must be 16-byte aligned
                                   (pl_off[i] % 8 == 0 for int16).  Outputs are int32 in either case. */
}
mcb_batch;

/*  Results.  Any pointer may be NULL = not wanted (except ret).  */
typedef struct mcb_result
{
    /* per site */
    int32_t  *ret;          /* [nsites] return value of mcall(): 0 = skipped/not a variant under -v, else nals_new */
    uint32_t *als_new;      /* [nsites] call->als_new bitmask over the ORIGINAL alleles */
    int8_t   *als_map;      /* [nsites][max_nals] call->als_map: old allele -> new index, -1 dropped (mcall.c:547-556) */
    float    *qual;         /* [nsites] rec->qual; missing = MCB_FLOAT_MISSING_BITS */
    int32_t  *ac;           /* [nsites][max_nals] call->ac[0..nals_new): ac[0]=REF count, INFO/AC = ac[1..) */
    int32_t  *an;           /* [nsites] INFO/AN */
    uint32_t *site_flags;   /* [nsites] MCB_SITE_* */
    double   *diag;         /* [nsites][4] {max_qual, lk_sum, ref_lk, gap between best and runner-up allele set} */
    /* per sample */
    int32_t  *gt;           /* [nsites][nsmpl][2] call->gts, htslib encoding; haploid: second = MCB_INT32_VECTOR_END */
    int32_t  *gq;           /* [nsites][nsmpl] FORMAT/GQ (only with MCB_CALL_FMT_GQ|GP) */
    float    *gp;           /* FORMAT/GP, site i at gp + pl_off[i], [nsmpl][G'_i] (only with MCB_CALL_FMT_GP) */
    int32_t  *pl;           /* trimmed FORMAT/PL, site i at pl + pl_off[i], [nsmpl][G'_i], G'_i from ret[i] */
    int64_t  *pl_off_out;   /* [nsites] optional.  If non-NULL the trimmed PLs (and GP) are written COMPACTED: site i lies
                               at pl + pl_off_out[i] (16-byte aligned blocks in no particular order, -1 when the site has
                               no PL); the used prefix of pl is all that travels device->host in mcb_call_host.  It never
                               exceeds sum_i (nsmpl*G_i + 3) & ~3 int32 units, which is at most the extent of the input
                               layout, so a buffer sized for pl_off[] indexing always suffices (also with "adjudicate") */
    /* BCF typed-vector outputs (mcb_call_host only; SURVEY.md §8f N1).  When non-NULL they are filled INSTEAD of gt / gq / pl:
       the per-sample results are narrowed on the device to the types a BCF record stores them in (what bcf_update_genotypes /
       bcf_update_format_int32 + vcf_write would re-encode the int32 arrays to), so 9 instead of 24 bytes per biallelic call
       cross PCIe.  Sentinels are the BCF ones: missing = INT8_MIN / INT16_MIN, vector_end = INT8_MIN+1 / INT16_MIN+1;
       a PL above INT16_MAX saturates (such sites carry MCB_SITE_PL_RANGE).  */
    int8_t   *gt8;          /* [nsites][nsmpl][2] BCF_BT_INT8 */
    int8_t   *gq8;          /* [nsites][nsmpl]    BCF_BT_INT8 */
    int16_t  *pl16;         /* BCF_BT_INT16, same ELEMENT offsets as pl (pl_off, or pl_off_out when compacted) */
}
mcb_result;

/* ---- lifecycle (mcall_init / mcall_destroy) ------------------------------------------------ */
int  mcb_init(mcb_ctx **ctx, const mcb_params *params);
void mcb_destroy(mcb_ctx *ctx);

/*  Register a ploidy vector (values 0/1/2): what set_ploidy() writes into call->ploidy
 *  (vcfcall.c:807-825).  Few distinct vectors exist (one per ploidy region), sites refer
 *  to them by id.  id 0 defaults to all-diploid.  Registering a NEW id uploads that one row and
 *  does not wait for work in flight; re-defining an id that earlier batches used synchronises
 *  the device first.                                                                    */
int  mcb_set_ploidy(mcb_ctx *ctx, int id, const uint8_t *ploidy);

/* ---- the hot path (mcall) -------------------------------------------------------------------
 *  mcb_call_device: every pointer inside batch/result is a DEVICE pointer; the two kernels are
 *  enqueued on `cuda_stream` (a cudaStream_t, NULL = default stream) and the call returns
 *  without synchronising.
 *  mcb_call_host: every pointer is a HOST pointer (pinned memory from mcb_host_alloc overlaps
 *  best); the batch is cut into slabs that are double-buffered H2D -> kernels -> D2H over two
 *  CUDA streams; returns when all results are in host memory.                               */
int  mcb_call_device(mcb_ctx *ctx, const mcb_batch *batch, const mcb_result *result, void *cuda_stream);
int  mcb_call_host(mcb_ctx *ctx, const mcb_batch *batch, const mcb_result *result);

/* ---- helpers -------------------------------------------------------------------------------- */
void *mcb_host_alloc(size_t bytes);         /* pinned host memory (cudaHostAlloc) */
void  mcb_host_free(void *ptr);
const char *mcb_strerror(int code);
const char *mcb_last_cuda_error(const mcb_ctx *ctx);
double mcb_get_theta(const mcb_ctx *ctx);   /* call->theta after mcall_init (log space), for tests */
int   mcb_get_pl2p(const mcb_ctx *ctx, double *pl2p256);   /* call->pl2p (mcall.c:56-61) */
/*  kernel launch statistics of the last mcb_call_* (bench.py's gpu_launches / roofline):
 *  stats[0]=kernel launches, [1]=sites, [2]=algorithmic bytes read, [3]=algorithmic bytes written */
int   mcb_get_stats(const mcb_ctx *ctx, int64_t stats[4]);
/*  tuning knob for experiments (threads per block, tile samples, ...): see DESIGN.md.
 *  "adjudicate" (0|1, default 0): every site of an mcb_call_device / mcb_call_host call that comes back with MCB_SITE_NEAR_TIE
 *  is evaluated a second time inside the same call, on the same stream and without a host synchronisation, with the literal
 *  sample-sequential sums of logs of mcall_find_best_alleles (mcall.c:591-710).  All of the site's outputs are overwritten
 *  by that evaluation and it carries MCB_SITE_NEAR_TIE | MCB_SITE_ADJUDICATED.  Needs result.site_flags: a call without it
 *  returns MCB_EINVAL.  Compacted PL output (pl_off_out) stays within the documented capacity: a flagged site reserves the
 *  block of its full genotype count.  "exact_phase1" (0|1): every site through the literal phase 1.  */
int   mcb_set_option(mcb_ctx *ctx, const char *key, int64_t value);
int   mcb_version(void);
/*  device milliseconds of the site kernel per allele-count class (ms[1..5], ms[0]=sum) of the last
 *  mcb_call_device; requires mcb_set_option(ctx,"time_kernels",1) */
int   mcb_get_kernel_times(mcb_ctx *ctx, float ms[6]);
/*  sites of each allele-count class (n[3..5]) that the multi-allelic kernels of the last mcb_call_device handed back to the
 *  general kernel (DESIGN.md 4b); synchronises the device  */
int   mcb_get_fallback_counts(mcb_ctx *ctx, int32_t n[6]);
/*  device self-test of the shared-reciprocal IEEE division (mode 0: exhaustive 256^3 biallelic domain;
 *  mode 6/10/15: n random vectors of that many genotypes); *mismatch must come back 0 */
int   mcb_selftest_div(mcb_ctx *ctx, int mode, uint64_t n, uint64_t seed, uint64_t *mismatch);

#ifdef __cplusplus
}
#endif
#endif
