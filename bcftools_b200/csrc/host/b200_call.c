/*  b200_call.c -- the host batcher (plain C): mirrors mcall_init / mcall / mcall_destroy (call.h:131-147) over
 *  pinned structure-of-arrays slabs and the C-ABI of mcall_b200.h.  See include/b200_call.h.
 *
 *  Two slab sets: while the GPU works on one batch (mcb_call_host on a worker thread), the driver keeps unpacking
 *  records into the other, the way vcfcall.c:1089-1148 keeps reading while the previous record is written.
 *  Every mcb_* call on the context is made by the worker thread (or while it is idle), so the context is still used by
 *  one thread at a time (call_t is not re-entrant either).
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <stdarg.h>
#include <pthread.h>
#include "b200_call.h"

typedef struct
{
    /* pinned input slabs (structure of arrays, site x sample x genotype) */
    int n;
    int32_t *pl;   int64_t pl_used;   int64_t *pl_off;
    int32_t *ad;   int64_t ad_used;   int64_t *ad_off;   uint8_t *nad;
    uint8_t *nals, *unseen, *nqs;   uint16_t *ploidy_id;
    float *qs;   int32_t *prior_an, *prior_ac;
    void **user_in;
    /* pinned result slabs of the batch last run from this set */
    mcb_result res;
    void **user_out;
    int nres;
    int ploidy_upto;        /* ploidy ids below this must be registered with the context before the batch runs */
}
b200_slabs_t;

struct b200_batcher
{
    mcb_ctx *ctx;
    int nsmpl, max_nals, cap;
    int64_t pl_cap, ad_cap;     /* elements of the PL / AD slabs */
    int64_t pl_rec, ad_rec;     /* ... of one worst-case record (max_nals alleles) */
    b200_slabs_t set[2];
    int fill;               /* set the driver is queuing records into */
    int inflight;           /* set the worker is running, -1 = none */
    int current;            /* set whose results b200_mcall_result serves, -1 = none */
    int nready;
    /* distinct ploidy vectors seen so far (id 0 = all diploid, registered by mcb_init); new ones are handed to the context
       by the worker right before the first batch that refers to them */
    uint8_t *ploidy_tab;   int n_ploidy, cap_ploidy, n_registered;
    int last_ploidy_id;
    int grouped, use_prior, typed, async;
    /* worker */
    pthread_t thr;   int thr_started;
    pthread_mutex_t mu;   pthread_cond_t cv_work, cv_done;
    int job;                /* set to run, -1 = idle */
    int job_done, job_rc, quit;
    char job_err[512];
};

static void default_handler(const char *msg) { fputs(msg, stderr); exit(-1); }      /* version.c:40-47 */
static void (*g_handler)(const char *msg) = default_handler;
void b200_set_error_handler(void (*handler)(const char *msg)) { g_handler = handler ? handler : default_handler; }

static void b200_error(const char *fmt, ...)
{
    char buf[1024];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    g_handler(buf);
}

static void *pinned(size_t bytes)
{
    void *p = mcb_host_alloc(bytes ? bytes : 1);
    if ( !p ) b200_error("b200: could not allocate %zu bytes of pinned memory\n", bytes);
    return p;
}
static void *xcalloc(size_t n, size_t size)
{
    void *p = calloc(n ? n : 1, size);
    if ( !p ) b200_error("b200: could not allocate %zu bytes\n", n*size);
    return p;
}

static int run_batch(b200_batcher_t *b, b200_slabs_t *s, char *err, size_t nerr)
{
    /* ploidy vectors this batch is the first to use */
    for (; b->n_registered < s->ploidy_upto; b->n_registered++)
    {
        int rc = mcb_set_ploidy(b->ctx, b->n_registered, b->ploidy_tab + (size_t)b->n_registered*b->nsmpl);
        if ( rc ) { snprintf(err, nerr, "b200_mcall: mcb_set_ploidy: %s (%s)\n", mcb_strerror(rc), mcb_last_cuda_error(b->ctx)); return rc; }
    }
    mcb_batch in; memset(&in, 0, sizeof in);
    in.pl_type = b->typed ? 2 : 4;
    in.nsites = s->n;  in.pl = s->pl;  in.pl_off = s->pl_off;  in.nals = s->nals;  in.unseen = s->unseen;
    in.ploidy_id = s->ploidy_id;
    if ( b->grouped ) { in.ad = s->ad; in.ad_off = s->ad_off; in.nad = s->nad; }
    else { in.qs = s->qs; in.nqs = s->nqs; }
    if ( b->use_prior ) { in.prior_an = s->prior_an; in.prior_ac = s->prior_ac; }
    int rc = mcb_call_host(b->ctx, &in, &s->res);
    if ( rc ) snprintf(err, nerr, "b200_mcall: %s (%s)\n", mcb_strerror(rc), mcb_last_cuda_error(b->ctx));
    return rc;
}

static void *worker_main(void *arg)
{
    b200_batcher_t *b = (b200_batcher_t*) arg;
    pthread_mutex_lock(&b->mu);
    for (;;)
    {
        while ( b->job < 0 && !b->quit ) pthread_cond_wait(&b->cv_work, &b->mu);
        if ( b->quit ) break;
        const int k = b->job;
        pthread_mutex_unlock(&b->mu);
        char err[512]; err[0] = 0;
        const int rc = run_batch(b, &b->set[k], err, sizeof err);
        pthread_mutex_lock(&b->mu);
        b->job_rc = rc;  memcpy(b->job_err, err, sizeof err);
        b->job = -1;  b->job_done = 1;
        pthread_cond_signal(&b->cv_done);
    }
    pthread_mutex_unlock(&b->mu);
    return NULL;
}

static void alloc_set(b200_batcher_t *b, b200_slabs_t *s, uint32_t output_tags)
{
    const int S = b->nsmpl, M = b->max_nals, R = b->cap;
    s->pl = (int32_t*) pinned((size_t)b->pl_cap*(b->typed ? 2 : 4));      /* typed: an int16 slab (mcb_batch.pl_type = 2) */
    s->pl_off = (int64_t*) pinned(sizeof(int64_t)*R);
    if ( b->grouped )
    {
        s->ad = (int32_t*) pinned((size_t)b->ad_cap*4);
        s->ad_off = (int64_t*) pinned(sizeof(int64_t)*R);
        s->nad = (uint8_t*) pinned(R);
    }
    s->nals = (uint8_t*) pinned(R);  s->unseen = (uint8_t*) pinned(R);  s->nqs = (uint8_t*) pinned(R);
    s->ploidy_id = (uint16_t*) pinned(2*(size_t)R);
    s->qs = (float*) pinned(sizeof(float)*(size_t)R*M);
    s->prior_an = (int32_t*) pinned(4*(size_t)R);  s->prior_ac = (int32_t*) pinned(4*(size_t)R*M);
    s->user_in = (void**) xcalloc(R, sizeof(void*));  s->user_out = (void**) xcalloc(R, sizeof(void*));
    s->res.ret = (int32_t*) pinned(4*(size_t)R);          s->res.als_new = (uint32_t*) pinned(4*(size_t)R);
    s->res.als_map = (int8_t*) pinned((size_t)R*M);       s->res.qual = (float*) pinned(4*(size_t)R);
    s->res.ac = (int32_t*) pinned(4*(size_t)R*M);         s->res.an = (int32_t*) pinned(4*(size_t)R);
    s->res.site_flags = (uint32_t*) pinned(4*(size_t)R);  s->res.diag = NULL;
    const int want_gq = (output_tags & (CALL_FMT_GQ|CALL_FMT_GP)) != 0;
    if ( b->typed )
    {
        s->res.gt8 = (int8_t*) pinned(2*(size_t)R*S);
        s->res.gq8 = want_gq ? (int8_t*) pinned((size_t)R*S) : NULL;
        s->res.pl16 = (int16_t*) pinned((size_t)b->pl_cap*2);
    }
    else
    {
        s->res.gt = (int32_t*) pinned(8*(size_t)R*S);
        s->res.gq = want_gq ? (int32_t*) pinned(4*(size_t)R*S) : NULL;
        s->res.pl = (int32_t*) pinned((size_t)b->pl_cap*4);
    }
    s->res.gp = (output_tags & CALL_FMT_GP) ? (float*) pinned((size_t)b->pl_cap*4) : NULL;
    s->res.pl_off_out = (int64_t*) pinned(sizeof(int64_t)*R);
}
static void free_set(b200_slabs_t *s)
{
    mcb_host_free(s->pl); mcb_host_free(s->pl_off); mcb_host_free(s->ad); mcb_host_free(s->ad_off); mcb_host_free(s->nad);
    mcb_host_free(s->nals); mcb_host_free(s->unseen); mcb_host_free(s->nqs); mcb_host_free(s->ploidy_id);
    mcb_host_free(s->qs); mcb_host_free(s->prior_an); mcb_host_free(s->prior_ac);
    mcb_host_free(s->res.ret); mcb_host_free(s->res.als_new); mcb_host_free(s->res.als_map); mcb_host_free(s->res.qual);
    mcb_host_free(s->res.ac); mcb_host_free(s->res.an); mcb_host_free(s->res.site_flags); mcb_host_free(s->res.gt);
    mcb_host_free(s->res.gq); mcb_host_free(s->res.gp); mcb_host_free(s->res.pl); mcb_host_free(s->res.pl_off_out);
    mcb_host_free(s->res.gt8); mcb_host_free(s->res.gq8); mcb_host_free(s->res.pl16);
    free(s->user_in); free(s->user_out);
}

void b200_mcall_init(b200_call_t *call)
{
    b200_batcher_t *b = (b200_batcher_t*) xcalloc(1, sizeof *b);
    b->nsmpl = call->nsmpl;
    b->max_nals = call->max_nals>0 ? call->max_nals : 5;
    b->cap = call->max_records>0 ? call->max_records : 4096;
    b->grouped = call->nsmpl_grp > 1;
    b->use_prior = call->use_prior;
    b->typed = call->bcf_typed && !b->grouped;
    b->async = call->async_flush;
    b->fill = 0;  b->inflight = -1;  b->current = -1;  b->job = -1;

    mcb_params p; memset(&p, 0, sizeof p);
    p.nsmpl = call->nsmpl;  p.max_nals = b->max_nals;
    p.theta = call->theta;                      /* raw: mcb_init applies the Watterson factor and log (mcall.c:397-416) */
    p.init_ploidy = call->ploidy;               /* as it is at init time: all ploidy_max, vcfcall.c:652-655 */
    p.flag = call->flag & (CALL_KEEPALT|CALL_VARONLY);
    p.output_tags = call->output_tags & (CALL_FMT_GQ|CALL_FMT_GP);
    p.ngroups = b->grouped ? call->nsmpl_grp : 1;
    p.grp_off = call->grp_off;  p.grp_smpl = call->grp_smpl;
    p.use_prior = call->use_prior;  p.device = call->device;  p.tie_eps = call->tie_eps;
    int rc = mcb_init(&b->ctx, &p);
    if ( rc ) b200_error("b200_mcall_init: %s (%s)\n", mcb_strerror(rc), b->ctx ? mcb_last_cuda_error(b->ctx) : "");
    /* the sites whose two best allele sets are closer than tie_eps are evaluated a second time inside each mcb_call_host, with
       the literal sample-sequential sums of logs of the reference (DESIGN.md §5): in every mode, grouped and typed included */
    rc = mcb_set_option(b->ctx, "adjudicate", 1);
    if ( rc ) b200_error("b200_mcall_init: %s\n", mcb_strerror(rc));

    const int S = b->nsmpl, M = b->max_nals, R = b->cap;
    const int64_t gmax = (int64_t)M*(M+1)/2;
    /*  The PL / AD slabs hold a VOLUME, not max_records worst-case records (1,024 records x 2,504 samples x 528 genotypes of a
     *  32-allele site would be 5.4 GB per slab, four slabs, all pinned): a batch is also full when less than one worst-case record
     *  is left (b200_mcall).  Sites start on 16-byte boundaries (8 int16 / 4 int32 elements).  */
    b->pl_rec = ((int64_t)S*gmax + 7) & ~7ll;
    b->ad_rec = ((int64_t)S*M + 3) & ~3ll;
    b->pl_cap = (int64_t)R*b->pl_rec;
    b->ad_cap = (int64_t)R*b->ad_rec;
    {
        int64_t budget = 64ll<<20;                          /* elements */
        const char *e = getenv("B200_PL_SLAB_ELEMS");       /* tests shrink the slab to reach the volume limit with small batches */
        if ( e && atoll(e) > 0 ) budget = atoll(e);
        if ( b->pl_cap > budget ) b->pl_cap = budget > 2*b->pl_rec ? budget : 2*b->pl_rec;
    }
    { const int64_t budget = 16ll<<20; if ( b->ad_cap > budget ) b->ad_cap = budget > 2*b->ad_rec ? budget : 2*b->ad_rec; }
    for (int k=0; k<2; k++) alloc_set(b, &b->set[k], p.output_tags);
    b->cap_ploidy = 8;
    b->ploidy_tab = (uint8_t*) xcalloc((size_t)b->cap_ploidy*S, 1);
    memset(b->ploidy_tab, 2, S);                /* id 0 of the context = all diploid */
    b->n_ploidy = 1;  b->n_registered = 1;  b->last_ploidy_id = 0;
    pthread_mutex_init(&b->mu, NULL);  pthread_cond_init(&b->cv_work, NULL);  pthread_cond_init(&b->cv_done, NULL);
    if ( pthread_create(&b->thr, NULL, worker_main, b) ) b200_error("b200_mcall_init: could not start the worker thread\n");
    b->thr_started = 1;
    call->batcher = b;
}

/*  the batch in flight, if any, has finished: its results become the current ones.  The reference error()s out of
 *  mcall() where the device can only flag the site (mcall.c:1523), so the flags are checked here, on the caller's thread.  */
static int wait_inflight(b200_batcher_t *b)
{
    if ( b->inflight < 0 ) return 0;
    pthread_mutex_lock(&b->mu);
    while ( !b->job_done ) pthread_cond_wait(&b->cv_done, &b->mu);
    const int rc = b->job_rc;
    char err[512]; memcpy(err, b->job_err, sizeof err);
    pthread_mutex_unlock(&b->mu);
    b200_slabs_t *s = &b->set[b->inflight];
    b->inflight = -1;
    if ( rc ) { b->current = -1; b->nready = 0; b200_error("%s", err); return 0; }
    for (int i=0; i<s->nres; i++)
    {
        const uint32_t f = s->res.site_flags[i];
        if ( f & MCB_SITE_BAD_PRIOR ) b200_error("Incorrect prior AN,AC values at record %d of the batch\n", i);                          /* mcall.c:1523 */
        if ( f & MCB_SITE_UNSUPPORTED ) b200_error("b200_mcall: record %d of the batch (%d alleles) is not covered by the device kernels%s\n",
                                                   i, (int)s->nals[i], b->typed ? " in bcf_typed mode (more than 5 alleles need int32 PLs)" : "");
    }
    b->current = (int)(s - b->set);
    b->nready = s->nres;
    return b->nready;
}

int b200_mcall_wait(b200_call_t *call)
{
    b200_batcher_t *b = call->batcher;
    if ( b->inflight < 0 ) { b->nready = 0; b->current = -1; return 0; }
    return wait_inflight(b);
}

int b200_mcall_flush_async(b200_call_t *call)
{
    b200_batcher_t *b = call->batcher;
    int n = 0;
    if ( b->inflight >= 0 ) n = wait_inflight(b);       /* one batch in flight at most: the older one completes first */
    else { b->nready = 0; b->current = -1; }
    b200_slabs_t *s = &b->set[b->fill];
    if ( !s->n ) return n;
    /* hand the filled set to the worker; the other set (whose results, if any, are the current ones: inputs and results
       are separate arrays) becomes the one records are queued into */
    s->nres = s->n;
    s->ploidy_upto = b->n_ploidy;
    { void **t = s->user_in; s->user_in = s->user_out; s->user_out = t; }
    pthread_mutex_lock(&b->mu);
    b->job = b->fill;  b->job_done = 0;
    pthread_cond_signal(&b->cv_work);
    pthread_mutex_unlock(&b->mu);
    b->inflight = b->fill;
    b->fill ^= 1;
    s = &b->set[b->fill];
    s->n = 0;  s->pl_used = 0;  s->ad_used = 0;
    return n;
}

int b200_mcall_flush(b200_call_t *call)
{
    const int n = b200_mcall_flush_async(call);
    if ( n ) return n;
    return b200_mcall_wait(call);
}

static int ploidy_id_of(b200_batcher_t *b, const uint8_t *ploidy)
{
    const int S = b->nsmpl;
    if ( !memcmp(b->ploidy_tab + (size_t)b->last_ploidy_id*S, ploidy, S) ) return b->last_ploidy_id;
    for (int id=0; id<b->n_ploidy; id++)        /* few distinct vectors exist: one per ploidy region and sex combination */
        if ( !memcmp(b->ploidy_tab + (size_t)id*S, ploidy, S) ) return b->last_ploidy_id = id;
    if ( b->n_ploidy >= 65535 ) b200_error("b200_mcall: more than 65535 distinct ploidy vectors\n");
    if ( b->n_ploidy == b->cap_ploidy )
    {
        /* the worker may be reading the table: grow it only while no batch is in flight */
        pthread_mutex_lock(&b->mu);
        while ( b->job >= 0 ) pthread_cond_wait(&b->cv_done, &b->mu);
        b->cap_ploidy *= 2;
        uint8_t *t = (uint8_t*) realloc(b->ploidy_tab, (size_t)b->cap_ploidy*S);
        if ( !t ) { pthread_mutex_unlock(&b->mu); b200_error("b200: could not allocate %zu bytes\n", (size_t)b->cap_ploidy*S); return 0; }
        b->ploidy_tab = t;
        pthread_mutex_unlock(&b->mu);
    }
    memcpy(b->ploidy_tab + (size_t)b->n_ploidy*S, ploidy, S);
    return b->last_ploidy_id = b->n_ploidy++;
}

int b200_mcall(b200_call_t *call, const b200_rec_t *rec)
{
    b200_batcher_t *b = call->batcher;
    b200_slabs_t *s = &b->set[b->fill];
    const int S = b->nsmpl, M = b->max_nals, nals = rec->n_allele;
    if ( nals<1 || nals>M ) b200_error("b200_mcall: %d alleles, the batcher was initialised for at most %d\n", nals, M);
    const int ngt = nals*(nals+1)/2;
    /* mcall.c:1445-1446.  The reference also lets nPLs == nsmpl*nals (haploid-shaped vectors) through this check, but its
       set_pdg strides by the diploid genotype count anyway (SURVEY.md 8 quirks): only diploid-shaped PLs are accepted here. */
    if ( rec->nPLs != S*ngt )
        b200_error("Wrong number of PL fields? nals=%d npl=%d\n", nals, rec->nPLs);
    int i = s->n;
    s->pl_off[i] = s->pl_used;
    if ( b->typed )             /* the record's own typed vector goes into the int16 slab; int8 is widened here */
    {
        int16_t *dst = (int16_t*) s->pl + s->pl_used;
        if ( !rec->PL_typed || (rec->PL_bt!=1 && rec->PL_bt!=2) ) b200_error("b200_mcall: bcf_typed needs FORMAT/PL as an int8 or int16 typed vector\n");
        if ( rec->PL_bt==2 ) memcpy(dst, rec->PL_typed, sizeof(int16_t)*(size_t)rec->nPLs);
        else
        {
            const int8_t *src = (const int8_t*) rec->PL_typed;
            for (int k=0; k<rec->nPLs; k++) dst[k] = src[k]==INT8_MIN ? INT16_MIN : (src[k]==INT8_MIN+1 ? INT16_MIN+1 : src[k]);
        }
        s->pl_used += ((int64_t)rec->nPLs + 7) & ~7ll;         /* 16-byte aligned sites */
    }
    else
    {
        memcpy(s->pl + s->pl_used, rec->PLs, sizeof(int32_t)*(size_t)rec->nPLs);
        s->pl_used += ((int64_t)rec->nPLs + 3) & ~3ll;
    }
    s->nals[i] = (uint8_t)nals;  s->unseen[i] = call->unseen;
    if ( b->grouped )
    {
        if ( rec->nADs < 1 || rec->nADs % S )   /* mcall.c:1476 */
            b200_error("Error: FORMAT/AD is required with the -G option, mpileup must be run with \"-a AD\" or \"-a QS\"\n");
        s->ad_off[i] = s->ad_used;  s->nad[i] = (uint8_t)(rec->nADs/S);
        memcpy(s->ad + s->ad_used, rec->ADs, sizeof(int32_t)*(size_t)rec->nADs);
        s->ad_used += ((int64_t)rec->nADs + 3) & ~3ll;
    }
    else
    {
        if ( rec->nQS<=0 ) b200_error("The QS annotation not present at record %d of the batch\n", i);   /* mcall.c:1457 */
        int nq = rec->nQS < M ? rec->nQS : M;
        memset(s->qs + (size_t)i*M, 0, sizeof(float)*M);
        memcpy(s->qs + (size_t)i*M, rec->QS, sizeof(float)*nq);
        s->nqs[i] = (uint8_t)nq;
    }
    if ( b->use_prior )
    {
        s->prior_an[i] = rec->prior_an;
        for (int j=0; j<M; j++) s->prior_ac[(size_t)i*M+j] = j<rec->n_prior_ac ? rec->prior_ac[j] : MCB_INT32_VECTOR_END;
    }
    /* set_ploidy() rewrites call->ploidy between records (vcfcall.c:807-825): each DISTINCT vector is registered once */
    s->ploidy_id[i] = (uint16_t)(call->ploidy ? ploidy_id_of(b, call->ploidy) : 0);
    s->user_in[i] = rec->user;
    /* full: max_records records, or no room left for a worst-case record */
    if ( ++s->n == b->cap || b->pl_cap - s->pl_used < b->pl_rec || (b->grouped && b->ad_cap - s->ad_used < b->ad_rec) )
        return b->async ? b200_mcall_flush_async(call) : b200_mcall_flush(call);
    return 0;
}

int b200_mcall_result(b200_call_t *call, int i, b200_out_t *out)
{
    b200_batcher_t *b = call->batcher;
    if ( b->current<0 || i<0 || i>=b->nready ) return -1;
    const b200_slabs_t *s = &b->set[b->current];
    const int S = b->nsmpl, M = b->max_nals;
    memset(out, 0, sizeof *out);
    out->ret = s->res.ret[i];
    out->user = s->user_out[i];
    out->site_flags = s->res.site_flags[i];
    if ( out->ret<=0 ) return 0;
    out->als_new = s->res.als_new[i];
    out->als_map = s->res.als_map + (size_t)i*M;
    out->qual = s->res.qual[i];
    out->ac = s->res.ac + (size_t)i*M;  out->an = s->res.an[i];
    const int ref_gt = (out->site_flags & MCB_SITE_REF_GT) != 0;
    if ( b->typed )
    {
        out->gts8 = s->res.gt8 + (size_t)i*S*2;
        out->GQs8 = (s->res.gq8 && !ref_gt) ? s->res.gq8 + (size_t)i*S : NULL;
    }
    else
    {
        out->gts = s->res.gt + (size_t)i*S*2;
        out->GQs = (s->res.gq && !ref_gt) ? s->res.gq + (size_t)i*S : NULL;
    }
    if ( !(out->site_flags & MCB_SITE_PL_DROPPED) && s->res.pl_off_out[i]>=0 )
    {
        if ( b->typed ) out->PLs16 = s->res.pl16 + s->res.pl_off_out[i];
        else out->PLs = s->res.pl + s->res.pl_off_out[i];
        out->nPLs = S*out->ret*(out->ret+1)/2;
        if ( s->res.gp && !(out->site_flags & MCB_SITE_REF_GT) ) out->GPs = s->res.gp + s->res.pl_off_out[i];
    }
    return 0;
}

int b200_mcall_n_ploidy(const b200_call_t *call) { return call->batcher ? call->batcher->n_ploidy : 0; }

void b200_mcall_destroy(b200_call_t *call)
{
    b200_batcher_t *b = call->batcher;
    if ( !b ) return;
    if ( b->thr_started )
    {
        pthread_mutex_lock(&b->mu);
        while ( b->job >= 0 ) pthread_cond_wait(&b->cv_done, &b->mu);      /* a batch in flight finishes first */
        b->quit = 1;
        pthread_cond_signal(&b->cv_work);
        pthread_mutex_unlock(&b->mu);
        pthread_join(b->thr, NULL);
    }
    pthread_mutex_destroy(&b->mu);  pthread_cond_destroy(&b->cv_work);  pthread_cond_destroy(&b->cv_done);
    mcb_destroy(b->ctx);
    for (int k=0; k<2; k++) free_set(&b->set[k]);
    free(b->ploidy_tab); free(b);
    call->batcher = NULL;
}
