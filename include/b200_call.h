/*  b200_call.h -- host side of the B200 `call -m` path, in C, mirroring the reference's calling interface.
 *
 *  The reference exposes  void mcall_init(call_t*); int mcall(call_t*, bcf1_t*); void mcall_destroy(call_t*)
 *  (call.h:131-147) and drives them one record at a time from main_vcfcall() (vcfcall.c:1089-1148).  A GPU cannot be
 *  fed one record at a time, so this layer keeps the same three hooks but batches: b200_mcall() queues the record
 *  (after unpacking what mcall() would fetch with bcf_get_format_int32 / bcf_get_info_float, mcall.c:1444-1510, into
 *  pinned structure-of-arrays slabs) and flushes through the C-ABI (mcall_b200.h) when the batch is full.
 *  b200_call_t carries the call_t fields this path reads (call.h:72-123), with the same names and meaning.
 *  htslib-free: the caller hands the already-unpacked arrays (see INTEGRATION.md for the htslib glue).
 */
#ifndef B200_CALL_H
#define B200_CALL_H
#include <stdint.h>
#include "mcall_b200.h"
#ifdef __cplusplus
extern "C" {
#endif

/* same values as call.h:32-39 */
#define CALL_KEEPALT   1
#define CALL_VARONLY   (1<<1)
#define CALL_FMT_GQ    (1<<6)
#define CALL_FMT_GP    (1<<7)
#define B200_SITE_ADJUDICATED MCB_SITE_ADJUDICATED   /* b200_out_t.site_flags: the record's near tie was re-evaluated in the reference's summation order */

typedef struct b200_batcher b200_batcher_t;

typedef struct
{
    /* ---- set by the driver before b200_mcall_init, like vcfcall.c does for call_t ---- */
    int      nsmpl;             /* bcf_hdr_nsamples(call->hdr) */
    uint32_t flag;              /* CALL_KEEPALT | CALL_VARONLY            (call.h:112) */
    uint32_t output_tags;       /* CALL_FMT_GQ | CALL_FMT_GP              (call.h:93)  */
    double   theta;             /* prior, vcfcall.c:933; turned into log(theta*aM) by init (mcall.c:397-416) */
    uint8_t *ploidy;            /* [nsmpl] 0/1/2, rewritten per region by the driver (vcfcall.c:807-825); call.h:113 */
    uint8_t  unseen;            /* index of <*>, 0 = none (vcfcall.c:1101-1111); call.h:113 */
    int      nsmpl_grp;         /* number of -G groups, <=1 = pooled      (call.h:98-99) */
    const uint32_t *grp_off;    /* [nsmpl_grp+1] */
    const uint32_t *grp_smpl;   /* [nsmpl] smpl_grp_t.smpl lists, group after group (call.h:58) */
    int      use_prior;         /* -F prior_AN,prior_AC given (call.h:94) */
    int      max_records;       /* records per batch, 0 = 4096 */
    int      max_nals;          /* 0 = 5 (B2B_MAX_ALLELES, bam2bcf.h:64) */
    int      device;            /* CUDA device ordinal */
    int      bcf_typed;         /* 1: BCF typed vectors both ways (SURVEY.md 8f N1): FORMAT/PL is handed over as the record's own
                                   int8/int16 vector (b200_rec_t.PL_typed, e.g. bcf_fmt_t.p or b200_bcf_fmt_t.p) and GT / GQ / PL
                                   come back as int8 / int8 / int16 vectors (b200_out_t.gts8 / GQs8 / PLs16); pooled calling only.
                                   Near ties are adjudicated on the device from the int16 PLs as in the int32 mode */
    int      async_flush;       /* 1: a full batch is handed to the GPU in the background and b200_mcall keeps queuing into the second
                                   slab set; the results it then reports are those of the PREVIOUS batch (see b200_mcall_flush_async) */
    double   tie_eps;           /* allele sets closer than this in log-likelihood are near ties (0 = 1e-6): such records are called a second
                                   time with the literal sample-sequential sums of logs (mcall.c:607-611, 635-645, 680-690), inside the same device
                                   call (mcb_set_option "adjudicate"), and come back with MCB_SITE_NEAR_TIE | B200_SITE_ADJUDICATED in
                                   site_flags.  Every mode: pooled or grouped (-G), int32 or typed PLs, 1..32 alleles */
    /* ---- owned by this layer ---- */
    b200_batcher_t *batcher;
}
b200_call_t;

/*  What mcall() pulls out of one bcf1_t (mcall.c:1438-1510).  Pointers are only read during b200_mcall().  */
typedef struct
{
    int n_allele;               /* rec->n_allele */
    const int32_t *PLs; int nPLs;   /* bcf_get_format_int32(..."PL"...): nsmpl*G values (mcall.c:1444) */
    const float   *QS;  int nQS;    /* bcf_get_info_float(..."QS"...) (mcall.c:1456); pooled calling */
    const int32_t *ADs; int nADs;   /* FORMAT/AD for -G (mcall.c:1475): nsmpl*nad values */
    int32_t prior_an;               /* -F: INFO AN or INT32_MIN if absent (mcall.c:1507) */
    const int32_t *prior_ac; int n_prior_ac;
    void *user;                 /* e.g. the retained bcf1_t*, handed back with the result */
    const void *PL_typed; int PL_bt;    /* bcf_typed: the PL vector as stored in the record, nPLs values of BCF_BT_INT8 (1) or BCF_BT_INT16 (2) */
}
b200_rec_t;

/*  What mcall() writes back into the record (mcall.c:1546-1657), valid until the next b200_mcall on the same call.  */
typedef struct
{
    int ret;                    /* mcall()'s return value: 0 = not a variant / skipped, else number of output alleles */
    uint32_t als_new;           /* call->als_new */
    const int8_t *als_map;      /* [max_nals] call->als_map */
    float qual;                 /* rec->qual */
    const int32_t *ac; int an;  /* call->ac[0..ret), INFO/AN */
    uint32_t site_flags;        /* MCB_SITE_* (PL dropped, near tie, ...) */
    const int32_t *gts;         /* [nsmpl*2] call->gts */
    const int32_t *GQs;         /* [nsmpl] or NULL */
    const int32_t *PLs; int nPLs;   /* trimmed PLs: nsmpl*G' values, NULL when the tag is dropped (mcall.c:1583) */
    const float   *GPs;             /* FORMAT/GP (-a GP, mcall.c:859-884, 1621): nPLs float32 values laid out like PLs, or NULL */
    void *user;
    /* bcf_typed: the same three vectors in the types a BCF record stores them in (gts / GQs / PLs are NULL then) */
    const int8_t  *gts8;        /* [nsmpl*2] */
    const int8_t  *GQs8;        /* [nsmpl] or NULL */
    const int16_t *PLs16;       /* nPLs values or NULL */
}
b200_out_t;

/*  error handler: default prints and exit(-1) like error() in version.c:40-47  */
void b200_set_error_handler(void (*handler)(const char *msg));

void b200_mcall_init(b200_call_t *call);                            /* = mcall_init, vcfcall.c:697-698 */
/*  = mcall(), vcfcall.c:1136-1137, batched: queues the record.  Returns the number of results that became
 *  available: 0 while the batch is filling; after an automatic flush the size of the batch just run (async_flush = 0)
 *  or of the batch that was in flight before it (async_flush = 1, 0 the first time).  Results stay valid until the
 *  next call that returns results.                                                                               */
int  b200_mcall(b200_call_t *call, const b200_rec_t *rec);
/*  Two slab sets: one batch runs on the GPU (a worker thread inside this layer drives mcb_call_host) while the driver
 *  fills the other, the way vcfcall.c:1089-1148 keeps reading while earlier records are written.
 *    b200_mcall_flush_async  waits for the batch in flight (if any; its results become current and their number is
 *                            returned, else 0), then starts the queued records in the background and returns at once.
 *    b200_mcall_wait         waits for the batch in flight; returns the number of its results (0: nothing was in flight).
 *    b200_mcall_flush        = flush_async, then wait if that returned nothing.  `while ((n = b200_mcall_flush(c)) > 0) consume(n);`
 *                            drains everything in either mode; with async_flush = 0 it is the old synchronous flush.        */
int  b200_mcall_flush_async(b200_call_t *call);
int  b200_mcall_wait(b200_call_t *call);
int  b200_mcall_flush(b200_call_t *call);
int  b200_mcall_result(b200_call_t *call, int i, b200_out_t *out);  /* i-th current result, in input order */
int  b200_mcall_n_ploidy(const b200_call_t *call);                  /* distinct ploidy vectors registered so far (id 0 = all diploid included) */
void b200_mcall_destroy(b200_call_t *call);                         /* = mcall_destroy, vcfcall.c:722-723 */

#ifdef __cplusplus
}
#endif
#endif
