/*  mcall_abi.cu -- the C-ABI of include/mcall_b200.h: context, host-built tables, the device entry
 *  point (kernels enqueued on the caller's stream) and the host entry point (slabs double-buffered
 *  H2D -> kernels -> D2H over two CUDA streams).
 *
 *  There is NO CPU fallback: without a CUDA device mcb_init fails with MCB_ENODEV.
 */
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include <algorithm>
#include <utility>
#include "mcall_b200.h"
#include "mcall_kernels.cuh"

using namespace mcb;

#define NCLASS 6                /* allele-count classes 1..5 + class 0 = everything else */
#define NCOUNTS (NCLASS+24)     /* class counts | +NCLASS: work counters | +NCLASS+8: fallback-list counts | +NCLASS+16: fallback work counters */
/*  one allocation per batch/slab: NCLASS class lists, NCLASS fallback lists (sites the multi-allelic kernel hands to the general one)  */
static inline size_t lists_bytes(int cap) { return sizeof(int32_t)*(size_t)(2*NCLASS)*cap; }
#define MAX_STAGE 16
#define MW_L2_SHARE 0.34        /* the 4-allele warp kernel: its grid's tails of the packed copies may take this share of L2 */

/*  Scratch of the grouped (-G) and generic (6..32 allele) kernels, indexed by blockIdx inside a launch.  One set per host
 *  slab and one for the device path: slabs run on independent streams, so their launches may overlap and must not share it.  */
struct KernelScratch
{
    void *grp = nullptr;  size_t grp_bytes = 0;
    void *gen_grp = nullptr, *gen_pl = nullptr, *gen_sum = nullptr;  int gen_grid = 0;
    double *mm_sums[6] = {};  size_t mm_sums_bytes[6] = {};     /* mcall_multi.cu: per-CTA rows of normalisers, one buffer per allele-count class (the classes run concurrently) */
    uint8_t *mw_tail[6] = {};  size_t mw_tail_bytes[6] = {};    /* mcall_multi_warp.cu: per-warp tails of the packed copies (4-allele class) */
};
static void free_scratch(KernelScratch &k)
{
    cudaFree(k.grp); cudaFree(k.gen_grp); cudaFree(k.gen_pl); cudaFree(k.gen_sum);
    for (int i=0; i<6; i++) { cudaFree(k.mm_sums[i]); cudaFree(k.mw_tail[i]); }
    k = KernelScratch();
}

#define NSLAB 3
struct HostSlab                 /* one stage of the host-path ring (H2D of slab k+1 overlaps kernels and D2H of slab k) */
{
    cudaStream_t stream = nullptr;
    cudaEvent_t  done = nullptr, cursor_ready = nullptr;
    /* compaction tail still owed by the slab in flight on this stage */
    bool pending = false;  int p_beg = 0, p_n = 0;  size_t p_plout = 0, p_gp = 0, p_pl16 = 0;
    /* the small per-site arrays of a slab travel as ONE copy each way through pinned staging buffers */
    char *h_in = nullptr, *h_out = nullptr;  size_t h_in_bytes = 0, h_out_bytes = 0;
    size_t s_out_beg = 0, s_ret = 0, s_als = 0, s_map = 0, s_qual = 0, s_ac = 0, s_an = 0, s_fl = 0, s_diag = 0, s_ploo = 0;
    void  *dev = nullptr;  size_t dev_bytes = 0;    /* one arena, carved per slab */
    int32_t *lists = nullptr, *counts = nullptr;  int list_cap = 0;
    unsigned long long *cursor = nullptr;           /* device: compacted-PL allocation cursor (int32 units) */
    unsigned long long *h_cursor = nullptr;         /* pinned host copy */
    KernelScratch scratch;
};

struct mcb_ctx
{
    mcb_params p;
    int device = 0, nsm = 0;  size_t smem_per_sm = 0, l2_bytes = 0;
    double theta_log = 0;
    double pl2p[256];
    DevTables *d_tab = nullptr;
    uint8_t  *d_ploidy = nullptr;  int nploidy = 0, ploidy_cap = 0;  bool any_nondiploid = false;
    std::vector<uint8_t> h_ploidy;
    uint32_t *d_grp_off = nullptr, *d_grp_smpl = nullptr, *d_smpl2grp = nullptr;  int ngroups = 1;
    bool grp_sorted = false;             /* every group lists its members in ascending sample order (what mcall_biallelic_groups.cu walks) */
    int64_t opt_gorder = 35421;          /* -G: launch order of the allele-count classes on their streams, one decimal digit per class (sweep: profiles/r02_groups_launch_order.log) */
    int64_t opt_bgroups = 1;             /* -G, two-allele class: the warp-per-site kernel of mcall_biallelic_groups.cu (0: mcall_groups.cu only) */
    KernelScratch scratch;              /* device path (mcb_call_device) */
    /* device-path scratch */
    int32_t *d_lists = nullptr, *d_counts = nullptr;  int list_cap = 0;
    unsigned long long *d_cursor = nullptr;
    HostSlab slab[NSLAB];
    /* options */
    int64_t opt_tile_bytes = 0, opt_ring_bytes = 0, opt_blocks_per_sm = 0, opt_slab_bytes = 64ll<<20, opt_slab_min = 8ll<<20, opt_block = 0;     /* 0 = automatic */
    int64_t opt_exact = 0;               /* 1: every site through the literal phase 1 (KArgs.exact_phase1): the general, grouped and 6..32 allele kernels */
    int64_t opt_adjudicate = 0;          /* 1: the sites flagged MCB_SITE_NEAR_TIE are evaluated again with the literal phase 1 inside the call */
    int64_t opt_multi = 1;               /* 3-5 allele classes: the CTA-per-site kernel of mcall_multi.cu (0: the general tiled kernel) */
    int64_t opt_mm_nst = 0;              /* its ring stages per warp (0 = automatic) */
    int64_t opt_mm_nst_c[NCLASS] = {0,0,0,0,0,0};       /* ... per allele-count class */
    int64_t opt_mm_block = 0;            /* its CTA size (0 = automatic) */
    int64_t opt_mm_block_c[NCLASS] = {0,0,0,0,0,0};     /* ... per allele-count class */
    int64_t opt_warp2 = -1;              /* biallelic warp-per-site kernel: -1 automatic, 0 off, n = force n warps per CTA */
    int64_t opt_warp3 = -1;              /* 3-allele warp-per-site kernel: -1 automatic, 0 off, n = at most n warps per CTA */
    int64_t opt_warp4 = -1;              /* the same for the 4-allele warp-per-site kernel */
    int64_t opt_order = 54321;           /* launch order of the allele-count classes */
    int64_t opt_time_kernels = 0, opt_concurrent = 1;    /* class kernels on their own streams: a class fills the tail of the previous one (-3.5 % per C3 step) */
    int64_t opt_ring_bytes_c[NCLASS] = {0,0,0,0,0,0};   /* per allele-count class override of ring_bytes (0 = opt_ring_bytes) */
    int64_t opt_block_c[NCLASS] = {0,0,0,0,0,0};        /* per class override of the CTA size */
    int64_t opt_tile_bytes_c[NCLASS] = {0,0,0,0,0,0};   /* per class override of tile_bytes */
    int64_t opt_bps_c[NCLASS] = {0,0,0,0,0,0};          /* per class cap of resident CTAs per SM (0 = as many as fit): lets classes share an SM */
    cudaStream_t cstream[NCLASS] = {};   /* one stream per allele-count class: their persistent grids overlap */
    cudaEvent_t  cev_fork = nullptr, cev_join[NCLASS] = {};
    cudaEvent_t kev[NCLASS+1] = {};      /* events around the per-class launches (time_kernels=1) */
    bool kev_valid = false;
    /* stats */
    int64_t stats[4] = {0,0,0,0};
    std::string cuda_err;
};

static int cuda_fail(mcb_ctx *ctx, cudaError_t e, const char *what)
{
    if ( ctx )
    {
        char buf[512];
        snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
        ctx->cuda_err = buf;
    }
    return MCB_ECUDA;
}
#define CK(call) do { cudaError_t e_ = (call); if ( e_!=cudaSuccess ) return cuda_fail(ctx, e_, #call); } while (0)

/* ---- host-built tables --------------------------------------------------------------------------- */
static inline double gq_of(double x) { return -4.34294*log(x); }       /* mcall.c:877, host libm */
static void build_tables(DevTables *t)
{
    for (int i=0; i<256; i++) t->pl2p[i] = pow(10., -i/10.);            /* mcall.c:56-61 */
    for (int i=0; i<MCB_PL2P_BIG; i++) t->pl2p_big[i] = pow(10., -i/10.);  /* mcall.c:472 */
    /*  gq_thr[k] = the largest double x in (0,1] with gq_of(x) >= k, found by bisection over the
     *  (ordered) bit patterns of positive doubles.  GQ = max{k : x <= gq_thr[k]}, capped at 127.   */
    t->gq_thr[0] = HUGE_VAL;
    for (int k=1; k<128; k++)
    {
        uint64_t lo = 1, hi;                    /* lo: smallest denormal, gq ~ 3232 >= k */
        double one = 1.0; memcpy(&hi, &one, 8); /* gq_of(1.0) = -0 < k */
        while ( hi - lo > 1 )
        {
            uint64_t mid = lo + (hi-lo)/2;
            double x; memcpy(&x, &mid, 8);
            if ( gq_of(x) >= (double)k ) lo = mid; else hi = mid;
        }
        memcpy(&t->gq_thr[k], &lo, 8);
    }
}
static double init_theta(double theta, const uint8_t *init_ploidy, int nsmpl)      /* mcall.c:397-416 */
{
    if ( !(theta>0) ) return theta;
    int n = 0;
    if ( !init_ploidy ) n = 2*nsmpl;
    else for (int i=0; i<nsmpl; i++) n += init_ploidy[i];
    double aM = 1;
    for (int i=2; i<n; i++) aM += 1./i;
    theta *= aM;
    if ( theta >= 1 )
    {
        fprintf(stderr,"The prior is too big (theta*aM=%.2f), going with 0.99\n", theta);
        theta = 0.99;
    }
    return log(theta);
}

/* ---- lifecycle ------------------------------------------------------------------------------------ */
extern "C" int mcb_version(void) { return 100; }

extern "C" const char *mcb_strerror(int code)
{
    switch ( code )
    {
        case MCB_OK:     return "ok";
        case MCB_EINVAL: return "invalid argument";
        case MCB_ENOMEM: return "out of memory";
        case MCB_ECUDA:  return "CUDA error";
        case MCB_ENODEV: return "no CUDA device (this library has no CPU fallback)";
        case MCB_EPL:    return "Wrong number of PL fields";
        case MCB_EQS:    return "The QS annotation not present / FORMAT/AD required with -G";
        case MCB_EPRIOR: return "Incorrect prior AN,AC values";
    }
    return "unknown error";
}
extern "C" const char *mcb_last_cuda_error(const mcb_ctx *ctx) { return ctx ? ctx->cuda_err.c_str() : ""; }
extern "C" double mcb_get_theta(const mcb_ctx *ctx) { return ctx->theta_log; }
extern "C" int mcb_get_pl2p(const mcb_ctx *ctx, double *out) { memcpy(out, ctx->pl2p, sizeof(double)*256); return 0; }
extern "C" int mcb_get_stats(const mcb_ctx *ctx, int64_t stats[4]) { memcpy(stats, ctx->stats, sizeof(int64_t)*4); return 0; }

extern "C" int mcb_set_option(mcb_ctx *ctx, const char *key, int64_t value)
{
    if ( !ctx || !key ) return MCB_EINVAL;
    if ( !strcmp(key,"tile_bytes") )         ctx->opt_tile_bytes = value;
    else if ( !strcmp(key,"ring_bytes") )    ctx->opt_ring_bytes = value;
    else if ( !strcmp(key,"blocks_per_sm") ) ctx->opt_blocks_per_sm = value;
    else if ( !strcmp(key,"slab_bytes") )    ctx->opt_slab_bytes = value;
    else if ( !strcmp(key,"slab_min") )      ctx->opt_slab_min = value;        /* 0 = uniform slabs of slab_bytes */
    else if ( !strcmp(key,"time_kernels") )  ctx->opt_time_kernels = value;
    else if ( !strcmp(key,"concurrent") )    ctx->opt_concurrent = value;
    else if ( !strcmp(key,"order") )         ctx->opt_order = value;
    else if ( !strcmp(key,"multi") )         ctx->opt_multi = value;
    else if ( !strcmp(key,"bgroups") )       ctx->opt_bgroups = value;
    else if ( !strcmp(key,"gorder") )
    {
        int seen = 0; int64_t v = value;
        for (int i=0; i<5; i++) { const int d = (int)(v % 10); v /= 10; if ( d<1 || d>5 ) return MCB_EINVAL; seen |= 1<<d; }
        if ( v || seen != 0x3e ) return MCB_EINVAL;      /* a permutation of 1..5 */
        ctx->opt_gorder = value;
    }
    else if ( !strcmp(key,"exact_phase1") )  { if ( value<0 || value>1 ) return MCB_EINVAL; ctx->opt_exact = value; }
    else if ( !strcmp(key,"adjudicate") )    { if ( value<0 || value>1 ) return MCB_EINVAL; ctx->opt_adjudicate = value; }
    else if ( !strcmp(key,"mm_nst") )        { if ( value<0 || value>4 ) return MCB_EINVAL; ctx->opt_mm_nst = value; }
    else if ( !strncmp(key,"mm_nst_",7) && key[7]>='3' && key[7]<='5' && !key[8] ) { if ( value<0 || value>4 ) return MCB_EINVAL; ctx->opt_mm_nst_c[key[7]-'0'] = value; }
    else if ( !strcmp(key,"mm_block") )      { if ( value!=0 && value!=64 && value!=128 && value!=256 ) return MCB_EINVAL; ctx->opt_mm_block = value; }
    else if ( !strncmp(key,"mm_block_",9) && key[9]>='3' && key[9]<='5' && !key[10] ) { if ( value!=0 && value!=64 && value!=128 && value!=256 ) return MCB_EINVAL; ctx->opt_mm_block_c[key[9]-'0'] = value; }
    else if ( !strcmp(key,"warp2") )         { if ( value<-1 || value>biallelic_max_warps() ) return MCB_EINVAL; ctx->opt_warp2 = value; }
    else if ( !strcmp(key,"warp3") )         { if ( value<-1 || value>triallelic_max_warps() ) return MCB_EINVAL; ctx->opt_warp3 = value; }
    else if ( !strcmp(key,"warp4") )         { if ( value<-1 || value>multi_warp_max_warps() ) return MCB_EINVAL; ctx->opt_warp4 = value; }
    else if ( !strncmp(key,"ring_bytes_",11) && key[11]>='1' && key[11]<='5' && !key[12] ) ctx->opt_ring_bytes_c[key[11]-'0'] = value;
    else if ( !strncmp(key,"block_",6) && key[6]>='1' && key[6]<='5' && !key[7] )
    {
        if ( value!=0 && value!=32 && value!=64 && value!=128 && value!=256 ) return MCB_EINVAL;
        ctx->opt_block_c[key[6]-'0'] = value;
    }
    else if ( !strcmp(key,"block") )         { if ( value!=0 && value!=32 && value!=64 && value!=128 && value!=256 ) return MCB_EINVAL; ctx->opt_block = value; }
    else if ( !strncmp(key,"tile_bytes_",11) && key[11]>='1' && key[11]<='5' && !key[12] ) ctx->opt_tile_bytes_c[key[11]-'0'] = value;
    else if ( !strncmp(key,"bps_",4) && key[4]>='1' && key[4]<='5' && !key[5] ) { if ( value<0 ) return MCB_EINVAL; ctx->opt_bps_c[key[4]-'0'] = value; }
    else return MCB_EINVAL;
    return MCB_OK;
}

/*  Device copy of the ploidy table.  One row is uploaded per registration; the table is only reallocated (after a device
 *  synchronisation: kernels in flight read it) when it outgrows its capacity, which starts at 64 vectors.  */
static int upload_ploidy(mcb_ctx *ctx, int first, int count)
{
    const int S = ctx->p.nsmpl;
    if ( ctx->nploidy > ctx->ploidy_cap )
    {
        CK(cudaDeviceSynchronize());
        if ( ctx->d_ploidy ) cudaFree(ctx->d_ploidy);
        ctx->ploidy_cap = std::max(64, 2*ctx->nploidy);
        CK(cudaMalloc(&ctx->d_ploidy, (size_t)ctx->ploidy_cap*S));
        first = 0; count = ctx->nploidy;
    }
    CK(cudaMemcpy(ctx->d_ploidy + (size_t)first*S, ctx->h_ploidy.data() + (size_t)first*S, (size_t)count*S, cudaMemcpyHostToDevice));
    if ( !ctx->any_nondiploid )
        for (size_t i=(size_t)first*S; i<(size_t)(first+count)*S; i++) if ( ctx->h_ploidy[i]!=2 ) { ctx->any_nondiploid = true; break; }
    return MCB_OK;
}

extern "C" int mcb_init(mcb_ctx **out, const mcb_params *params)
{
    if ( !out || !params || params->nsmpl<=0 || params->max_nals<1 || params->max_nals>MCB_MAX_NALS ) return MCB_EINVAL;
    if ( params->ngroups > 1 && (!params->grp_off || !params->grp_smpl) ) return MCB_EINVAL;
    int ndev = 0;
    if ( cudaGetDeviceCount(&ndev)!=cudaSuccess || ndev<=0 ) return MCB_ENODEV;
    if ( params->device<0 || params->device>=ndev ) return MCB_EINVAL;
    mcb_ctx *ctx = new mcb_ctx();
    ctx->p = *params;
    ctx->p.init_ploidy = nullptr; ctx->p.grp_off = nullptr; ctx->p.grp_smpl = nullptr;
    if ( !(ctx->p.tie_eps > 0) ) ctx->p.tie_eps = 1e-6;
    ctx->device = params->device;
    *out = ctx;
    CK(cudaSetDevice(ctx->device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, ctx->device));
    ctx->nsm = prop.multiProcessorCount;
    ctx->smem_per_sm = prop.sharedMemPerMultiprocessor;
    ctx->l2_bytes = prop.l2CacheSize;
    ctx->theta_log = init_theta(params->theta, params->init_ploidy, params->nsmpl);

    DevTables *t = new DevTables();
    build_tables(t);
    memcpy(ctx->pl2p, t->pl2p, sizeof ctx->pl2p);
    cudaError_t e = cudaMalloc(&ctx->d_tab, sizeof(DevTables));
    if ( e==cudaSuccess ) e = cudaMemcpy(ctx->d_tab, t, sizeof(DevTables), cudaMemcpyHostToDevice);
    delete t;
    if ( e!=cudaSuccess ) return cuda_fail(ctx, e, "tables");

    ctx->h_ploidy.assign(params->nsmpl, 2);     /* id 0: all diploid */
    ctx->nploidy = 1;
    int rc = upload_ploidy(ctx, 0, 1);
    if ( rc ) return rc;
    CK(cudaMalloc(&ctx->d_counts, sizeof(int32_t)*NCOUNTS));     /* + work counter of the warp-per-site kernel */
    CK(cudaMalloc(&ctx->d_cursor, sizeof(unsigned long long)));
    if ( params->ngroups > 1 )         /* smpl_grp_t.smpl lists (mcall.c:250-349): every sample in exactly one group */
    {
        const int Q = params->ngroups, S = params->nsmpl;
        if ( params->grp_off[0]!=0 || params->grp_off[Q]!=(uint32_t)S ) return MCB_EINVAL;
        std::vector<uint32_t> s2g(S, 0xffffffffu);
        for (int g=0; g<Q; g++)
            for (uint32_t i=params->grp_off[g]; i<params->grp_off[g+1]; i++)
            {
                uint32_t smp = params->grp_smpl[i];
                if ( smp>=(uint32_t)S || s2g[smp]!=0xffffffffu ) return MCB_EINVAL;
                s2g[smp] = g;
            }
        ctx->ngroups = Q;
        ctx->grp_sorted = true;
        for (int g=0; g<Q; g++)
            for (uint32_t i=params->grp_off[g]+1; i<params->grp_off[g+1]; i++)
                if ( params->grp_smpl[i] <= params->grp_smpl[i-1] ) ctx->grp_sorted = false;
        CK(cudaMalloc(&ctx->d_grp_off, sizeof(uint32_t)*(Q+1)));
        CK(cudaMalloc(&ctx->d_grp_smpl, sizeof(uint32_t)*S));
        CK(cudaMalloc(&ctx->d_smpl2grp, sizeof(uint32_t)*S));
        CK(cudaMemcpy(ctx->d_grp_off, params->grp_off, sizeof(uint32_t)*(Q+1), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(ctx->d_grp_smpl, params->grp_smpl, sizeof(uint32_t)*S, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(ctx->d_smpl2grp, s2g.data(), sizeof(uint32_t)*S, cudaMemcpyHostToDevice));
    }
    for (int i=0; i<NSLAB; i++)
    {
        CK(cudaStreamCreateWithFlags(&ctx->slab[i].stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ctx->slab[i].done, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->slab[i].cursor_ready, cudaEventDisableTiming));
        CK(cudaMalloc(&ctx->slab[i].counts, sizeof(int32_t)*NCOUNTS));
        CK(cudaMalloc(&ctx->slab[i].cursor, sizeof(unsigned long long)));
        CK(cudaHostAlloc(&ctx->slab[i].h_cursor, sizeof(unsigned long long), cudaHostAllocDefault));
    }
    return MCB_OK;
}

extern "C" void mcb_destroy(mcb_ctx *ctx)
{
    if ( !ctx ) return;
    cudaSetDevice(ctx->device);
    cudaFree(ctx->d_tab); cudaFree(ctx->d_ploidy); cudaFree(ctx->d_grp_off); cudaFree(ctx->d_grp_smpl); cudaFree(ctx->d_smpl2grp); free_scratch(ctx->scratch);
    cudaFree(ctx->d_lists); cudaFree(ctx->d_counts); cudaFree(ctx->d_cursor);
    for (int i=0; i<NSLAB; i++)
    {
        if ( ctx->slab[i].stream ) cudaStreamDestroy(ctx->slab[i].stream);
        if ( ctx->slab[i].done ) cudaEventDestroy(ctx->slab[i].done);
        if ( ctx->slab[i].cursor_ready ) cudaEventDestroy(ctx->slab[i].cursor_ready);
        free_scratch(ctx->slab[i].scratch);
        cudaFree(ctx->slab[i].dev); cudaFree(ctx->slab[i].lists); cudaFree(ctx->slab[i].counts); cudaFree(ctx->slab[i].cursor);
        if ( ctx->slab[i].h_cursor ) cudaFreeHost(ctx->slab[i].h_cursor);
        if ( ctx->slab[i].h_in ) cudaFreeHost(ctx->slab[i].h_in);
        if ( ctx->slab[i].h_out ) cudaFreeHost(ctx->slab[i].h_out);
    }
    for (int i=0; i<=NCLASS; i++) if ( ctx->kev[i] ) cudaEventDestroy(ctx->kev[i]);
    for (int i=1; i<NCLASS; i++) { if ( ctx->cstream[i] ) cudaStreamDestroy(ctx->cstream[i]); if ( ctx->cev_join[i] ) cudaEventDestroy(ctx->cev_join[i]); }
    if ( ctx->cev_fork ) cudaEventDestroy(ctx->cev_fork);
    delete ctx;
}

extern "C" int mcb_set_ploidy(mcb_ctx *ctx, int id, const uint8_t *ploidy)
{
    if ( !ctx || id<0 || id>65535 || !ploidy ) return MCB_EINVAL;
    int S = ctx->p.nsmpl;
    for (int i=0; i<S; i++) if ( ploidy[i]>2 ) return MCB_EINVAL;
    CK(cudaSetDevice(ctx->device));
    const int old_n = ctx->nploidy;
    if ( id >= ctx->nploidy )
    {
        ctx->h_ploidy.resize((size_t)(id+1)*S, 2);
        ctx->nploidy = id+1;
    }
    const bool rewrite = id < old_n && memcmp(ctx->h_ploidy.data() + (size_t)id*S, ploidy, S);
    memcpy(ctx->h_ploidy.data() + (size_t)id*S, ploidy, S);
    if ( rewrite )
    {
        /* an id that batches already referred to changes its meaning: nothing in flight may still read the old row,
           and the "every sample diploid" shortcut is re-derived from the whole table */
        CK(cudaDeviceSynchronize());
        ctx->any_nondiploid = false;
        return upload_ploidy(ctx, 0, ctx->nploidy);
    }
    const int first = std::min(id, old_n);      /* ids skipped over are filled with all-diploid rows */
    return upload_ploidy(ctx, first, ctx->nploidy - first);
}

extern "C" void *mcb_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if ( cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault)!=cudaSuccess ) return nullptr;
    return p;
}
extern "C" void mcb_host_free(void *ptr) { if ( ptr ) cudaFreeHost(ptr); }

/*  Device time of the site kernel of each allele-count class in the last mcb_call_device (needs option
 *  time_kernels=1; synchronises the events).  ms[k] for k=1..5; ms[0] = sum.                              */
extern "C" int mcb_get_kernel_times(mcb_ctx *ctx, float ms[6])
{
    if ( !ctx || !ms || !ctx->kev_valid ) return MCB_EINVAL;
    CK(cudaSetDevice(ctx->device));
    CK(cudaEventSynchronize(ctx->kev[5]));
    ms[0] = 0;
    for (int k=1; k<=5; k++) { CK(cudaEventElapsedTime(&ms[k], ctx->kev[k-1], ctx->kev[k])); ms[0] += ms[k]; }
    return MCB_OK;
}

/*  Sites of each allele-count class (n[k], k=3..5; the other entries are 0) that the multi-allelic kernels of the last
 *  mcb_call_device handed back to the general kernel through their fallback lists (synchronises the device).              */
extern "C" int mcb_get_fallback_counts(mcb_ctx *ctx, int32_t n[6])
{
    if ( !ctx || !n || !ctx->d_counts ) return MCB_EINVAL;
    CK(cudaSetDevice(ctx->device));
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(n, ctx->d_counts + NCLASS + 8, sizeof(int32_t)*6, cudaMemcpyDeviceToHost));
    return MCB_OK;
}

/*  Self-test of the shared-reciprocal division used by phase 2 (see rcp_shared/div_shared in mcall_kernels.cu):
 *  mode 0 = exhaustive biallelic domain (256^3 PL triples), mode 6/10/15 = n random multi-allelic vectors.
 *  Writes the number of quotients that differ from IEEE a/b; must be 0.                                     */
extern "C" int mcb_selftest_div(mcb_ctx *ctx, int mode, uint64_t n, uint64_t seed, uint64_t *mismatch)
{
    if ( !ctx || !mismatch ) return MCB_EINVAL;
    CK(cudaSetDevice(ctx->device));
    unsigned long long *d = nullptr;
    CK(cudaMalloc(&d, 8));
    CK(cudaMemset(d, 0, 8));
    if ( mode==0 || mode==20 || mode==21 ) n = 1ull<<24;
    CK(launch_selftest_div(ctx->d_tab, mode, n, seed, d, 0));
    CK(cudaDeviceSynchronize());
    unsigned long long h = 0;
    CK(cudaMemcpy(&h, d, 8, cudaMemcpyDeviceToHost));
    cudaFree(d);
    *mismatch = h;
    return MCB_OK;
}

/* ---- launch geometry -------------------------------------------------------------------------------- */
/*  CTA size, tile size and ring size per allele-count class.  Explicit options win; the defaults below are the best
 *  settings of the sweeps in profiles/ (measured at 2,504 samples) plus smaller CTAs for small sample counts, where a
 *  128-thread CTA would have mostly idle lanes.                                                                    */
static int class_block(const mcb_ctx *ctx, int nals)
{
    if ( ctx->opt_block_c[nals] ) return (int)ctx->opt_block_c[nals];
    if ( ctx->opt_block ) return (int)ctx->opt_block;
    const int S = ctx->p.nsmpl;
    int b = S<=192 ? 32 : (S<=768 ? 64 : 128);
    if ( (nals==3 || nals==4) && b>64 ) b = 64;
    return b;
}
static int64_t class_tile_bytes(const mcb_ctx *ctx, int nals)
{
    if ( ctx->opt_tile_bytes_c[nals] ) return ctx->opt_tile_bytes_c[nals];
    if ( ctx->opt_tile_bytes ) return ctx->opt_tile_bytes;
    return (nals==3 || nals==4) ? 8192 : 32768;
}
static int64_t class_ring_bytes(const mcb_ctx *ctx, int nals)
{
    if ( ctx->opt_ring_bytes_c[nals] ) return ctx->opt_ring_bytes_c[nals];
    if ( ctx->opt_ring_bytes ) return ctx->opt_ring_bytes;
    return (nals==3 || nals==4) ? 16384 : 65536;
}

static void tile_geometry(const mcb_ctx *ctx, int nals, int es, int *tile_smpl, int *nstage, size_t *ring_bytes)
{
    int G = nals*(nals+1)/2, S = ctx->p.nsmpl;
    const int64_t tile_target = class_tile_bytes(ctx, nals);
    int ts = (int)(tile_target/(es*G));
    ts = std::max(256, ts/256*256);
    ts = std::min(ts, 32*class_block(ctx, nals));      /* the AC counters of phase 2 allow at most 63 samples per thread and tile */
    ts = std::max(ts, class_block(ctx, nals));      /* the AC counters of phase 2 allow at most 63 samples per thread and tile */
    int ntiles = (S + ts - 1)/ts;
    size_t tile_bytes = (size_t)ts*G*es;
    const int64_t ring_cap = class_ring_bytes(ctx, nals);
    int cap = (int)std::max<int64_t>(2, ring_cap/(int64_t)tile_bytes);
    int ns = std::min(MAX_STAGE, std::min(ntiles, cap));
    if ( ns<1 ) ns = 1;
    *tile_smpl = ts; *nstage = ns; *ring_bytes = tile_bytes*ns;
}

/*  Sites with 0 or more than 5 alleles (class 0).  With max_nals <= 5 they cannot be legal input and are reported
 *  unsupported; otherwise the generic kernel of mcall_generic.cu handles 6..32 alleles (int32 PLs).            */
static int enqueue_class0(mcb_ctx *ctx, KArgs &a, const mcb_batch *b, const mcb_result *r, int32_t *lists, int32_t *counts, int pl_es, KernelScratch &sc, cudaStream_t st)
{
    if ( ctx->p.max_nals <= 5 || pl_es != 4 )
    {
        CK(launch_unsupported(lists, counts, r->ret, r->site_flags, b->nals, r->pl_off_out, st));
        return MCB_OK;
    }
    if ( !sc.gen_grid )
    {
        size_t g1, g2, g3;
        generic_scratch_bytes(1, ctx->ngroups, ctx->p.nsmpl, &g1, &g2, &g3);
        int grid = (int)std::max<int64_t>(1, std::min<int64_t>(ctx->nsm, (int64_t)(768ll<<20)/(int64_t)(g1+g2+g3)));
        generic_scratch_bytes(grid, ctx->ngroups, ctx->p.nsmpl, &g1, &g2, &g3);
        CK(cudaMalloc(&sc.gen_grp, g1)); CK(cudaMalloc(&sc.gen_pl, g2)); CK(cudaMalloc(&sc.gen_sum, g3));
        sc.gen_grid = grid;
    }
    a.site_list = lists; a.site_count = counts;
    a.grp_off = ctx->d_grp_off; a.grp_smpl = ctx->d_grp_smpl; a.smpl2grp = ctx->d_smpl2grp; a.ngroups = ctx->ngroups;
    CK(launch_generic_kernel(a, sc.gen_grp, sc.gen_pl, sc.gen_sum, std::min(sc.gen_grid, std::max(1, b->nsites)), st));
    return MCB_OK;
}

/*  one stream per allele-count class (their persistent grids overlap) + fork / join events, created on first use  */
static int ensure_class_streams(mcb_ctx *ctx)
{
    if ( ctx->cev_fork ) return MCB_OK;
    CK(cudaEventCreateWithFlags(&ctx->cev_fork, cudaEventDisableTiming));
    /* concurrent=2: stream priorities in launch order (5 alleles first = highest), so that a later class only
       fills the SMs the earlier one leaves idle in the tail of its persistent grid */
    int plo = 0, phi = 0;
    CK(cudaDeviceGetStreamPriorityRange(&plo, &phi));       /* numerically lower = higher priority */
    for (int i=1; i<NCLASS; i++)
    {
        int pos = 0; { int64_t v = ctx->opt_order; int d[5] = {5,4,3,2,1}; for (int k=4; k>=0 && v>0; k--, v/=10) d[k] = (int)(v%10); for (int k=0; k<5; k++) if ( d[k]==i ) pos = k; }
        int prio = std::min(plo, phi + pos);
        if ( ctx->opt_concurrent>=2 ) CK(cudaStreamCreateWithPriority(&ctx->cstream[i], cudaStreamNonBlocking, prio));
        else
        CK(cudaStreamCreateWithFlags(&ctx->cstream[i], cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ctx->cev_join[i], cudaEventDisableTiming));
    }
    return MCB_OK;
}

/*  In-call adjudication (option "adjudicate"), enqueued on `st` behind every site kernel of the call (the class streams have
 *  joined it).  A scan of site_flags lists the sites flagged MCB_SITE_NEAR_TIE per allele-count class, in the class lists of
 *  the first evaluation, which no longer needs them; then each class is launched over its list with the literal phase 1: the
 *  general kernel (pooled, int32 or int16 PLs), the grouped kernel, the 6..32 allele kernel.  The grids are persistent and
 *  read the list's count on the device, so an empty list costs one short launch and the host never waits.  Every output
 *  of a listed site is overwritten, in place (KArgs.adj_pass; compacted blocks were reserved at full size, compact_out_off).
 *  The fallback-list counts of the first evaluation (mcb_get_fallback_counts) are left as they are.
 *  ggrid / gper_class: the grid and the per-class scratch stride of the grouped kernel (grouped calling only).  */
static int enqueue_adjudication(mcb_ctx *ctx, const KArgs &a1, const mcb_batch *b, int32_t *lists, int32_t *counts, int list_stride, int pl_es,
                                KernelScratch &sc, int ggrid, size_t gper_class, cudaStream_t st, int *launches)
{
    CK(cudaMemsetAsync(counts, 0, sizeof(int32_t)*2*NCLASS, st));          /* class counts + work counters */
    CK(launch_collect_near_ties(b->nals, b->nsites, a1.site_flags, lists, counts, list_stride, st));
    KArgs a = a1;
    a.exact_phase1 = 1; a.adj_pass = 1; a.adj_reserve = 0;
    a.fb_list = nullptr; a.fb_count = nullptr; a.mm_sums = nullptr;
    const bool ploidy = ctx->any_nondiploid, gpk = a.gp && (a.output_tags & MCB_CALL_FMT_GP);
    int n = 1;
    for (int nals=1; nals<=5; nals++, n++)
    {
        a.site_list = lists + (size_t)nals*list_stride; a.site_count = counts + nals;
        a.work_counter = counts + NCLASS + nals;
        if ( ctx->ngroups > 1 ) { CK(launch_groups_kernel(nals, a, (char*)sc.grp + (size_t)(nals-1)*gper_class, ggrid, st)); continue; }
        size_t ring; tile_geometry(ctx, nals, pl_es, &a.tile_smpl, &a.nstage, &ring);
        const int block = (pl_es==2 || gpk) ? 128 : class_block(ctx, nals);
        int nb = 1;
        CK(site_kernel_occupancy(nals, ploidy, gpk, block, pl_es, ring, &nb));
        if ( nb<1 ) return cuda_fail(ctx, cudaErrorLaunchOutOfResources, "site kernel does not fit on an SM");
        const int grid = (int)std::min<int64_t>((int64_t)b->nsites, (int64_t)ctx->nsm*nb);
        cudaError_t le = launch_site_kernel(nals, ploidy, gpk, block, pl_es, a, grid, ring, st);
        if ( le!=cudaSuccess ) return cuda_fail(ctx, le, "near-tie adjudication: site kernel");
    }
    if ( ctx->p.max_nals > 5 && pl_es == 4 )        /* 6..32 alleles (class 0) */
    {
        int rc = enqueue_class0(ctx, a, b, nullptr, lists, counts, pl_es, sc, st);
        if ( rc ) return rc;
        n++;
    }
    *launches += n;
    return MCB_OK;
}

static int enqueue(mcb_ctx *ctx, const mcb_batch *b, const mcb_result *r, int32_t *lists, int32_t *counts, int list_stride, unsigned long long *cursor, KernelScratch &sc, cudaStream_t st)
{
    CK(cudaMemsetAsync(counts, 0, sizeof(int32_t)*NCOUNTS, st));
    if ( r->pl_off_out ) CK(cudaMemsetAsync(cursor, 0, sizeof(unsigned long long), st));
    CK(launch_classify(b->nals, b->nsites, lists, counts, list_stride, ctx->p.max_nals, r->ret, r->site_flags, r->pl_off_out, st));
    int launches = 1;
    KArgs a;
    memset(&a, 0, sizeof a);
    a.pl = b->pl; a.pl_off = b->pl_off; a.nals = b->nals; a.unseen = b->unseen; a.ploidy_id = b->ploidy_id;
    a.qs = b->qs; a.nqs = b->nqs; a.ad = b->ad; a.ad_off = b->ad_off; a.nad = b->nad;
    a.prior_an = b->prior_an; a.prior_ac = b->prior_ac;
    a.ret = r->ret; a.als_new = r->als_new; a.als_map = r->als_map; a.qual = r->qual; a.ac = r->ac; a.an = r->an;
    a.site_flags = r->site_flags; a.diag = r->diag; a.gt = r->gt; a.gq = r->gq; a.gp = r->gp; a.out_pl = r->pl;
    a.pl_off_out = r->pl_off_out; a.pl_cursor = r->pl_off_out ? cursor : nullptr;
    a.tab = ctx->d_tab; a.ploidy_tab = ctx->d_ploidy; a.nploidy = ctx->nploidy;
    a.nsmpl = ctx->p.nsmpl; a.max_nals = ctx->p.max_nals; a.flag = ctx->p.flag; a.output_tags = ctx->p.output_tags;
    a.theta = ctx->theta_log; a.tie_eps = ctx->p.tie_eps; a.use_prior = ctx->p.use_prior;
    a.exact_phase1 = (int)ctx->opt_exact;
    a.adj_reserve = ctx->opt_adjudicate && r->pl_off_out;     /* flagged sites reserve their full-G compacted block (compact_out_off) */
    const bool ploidy = ctx->any_nondiploid;
    const int pl_es = b->pl_type==2 ? 2 : 4;
    if ( b->pl_type!=0 && b->pl_type!=4 && b->pl_type!=2 ) return MCB_EINVAL;
    if ( ctx->ngroups > 1 && pl_es!=4 ) return MCB_EINVAL;        /* grouped calling takes int32 PLs only */
    if ( ctx->ngroups > 1 )         /* grouped calling (-G): the correctness-first kernel of mcall_groups.cu */
    {
        if ( !b->ad || !b->ad_off || !b->nad ) return MCB_EQS;      /* mcall.c:1476 */
        a.grp_off = ctx->d_grp_off; a.grp_smpl = ctx->d_grp_smpl; a.smpl2grp = ctx->d_smpl2grp; a.ngroups = ctx->ngroups;
        int grid = std::min(b->nsites, ctx->nsm*8);
        const size_t per_cta = groups_scratch_bytes(1, ctx->ngroups, a.nsmpl);
        grid = (int)std::max<int64_t>(1, std::min<int64_t>(grid, (int64_t)(512ll<<20)/(int64_t)per_cta));
        const size_t per_class = (groups_scratch_bytes(grid, ctx->ngroups, a.nsmpl) + 255) & ~(size_t)255, need = 5*per_class;
        if ( need > sc.grp_bytes )
        {
            CK(cudaStreamSynchronize(st));
            if ( sc.grp ) CK(cudaFree(sc.grp));
            CK(cudaMalloc(&sc.grp, need));
            sc.grp_bytes = need;
        }
        /* the classes run on their own streams (each with its own stretch of the per-CTA group records): the multi-allelic
           ones are a few hundred sites per batch, i.e. a single wave bound by the latency of one site */
        /* time_kernels=1: the classes one after the other on the caller's stream, in ascending order, an event after each */
        const bool gtiming = ctx->opt_time_kernels && lists==ctx->d_lists;
        const bool gfork = ctx->opt_concurrent != 0 && !gtiming;
        if ( gfork )
        {
            { int src = ensure_class_streams(ctx); if ( src ) return src; }
            CK(cudaEventRecord(ctx->cev_fork, st));
        }
        if ( gtiming )
        {
            for (int i=0; i<=NCLASS; i++) if ( !ctx->kev[i] ) CK(cudaEventCreate(&ctx->kev[i]));
            CK(cudaEventRecord(ctx->kev[0], st));
        }
        for (int step=0; step<5; step++)
        {
            int nals = step+1;
            if ( !gtiming ) { int64_t v = ctx->opt_gorder; for (int i=0; i<4-step; i++) v /= 10; nals = (int)(v % 10); }
            a.site_list = lists + (size_t)nals*list_stride; a.site_count = counts + nals;
            a.work_counter = counts + NCLASS + nals;
            cudaStream_t cs = gfork ? ctx->cstream[nals] : st;
            if ( gfork ) CK(cudaStreamWaitEvent(cs, ctx->cev_fork, 0));
            /* two alleles, up to 32 groups with ascending member lists, no FORMAT/GP: the warp-per-site kernel; what it has no
               code for comes back on a fallback list that the general grouped kernel walks */
            if ( nals==2 && ctx->opt_bgroups && !ctx->opt_exact && ctx->grp_sorted && biallelic_groups_ok(a.nsmpl, ctx->ngroups) && !(a.gp && (a.output_tags & MCB_CALL_FMT_GP)) )
            {
                KArgs ab = a;
                ab.fb_list = lists + (size_t)(NCLASS + nals)*list_stride;
                ab.fb_count = counts + NCLASS + 8 + nals;
                const int w = biallelic_groups_warps();
                const int bgrid = (int)std::min<int64_t>(((int64_t)b->nsites + w - 1)/w, (int64_t)ctx->nsm*biallelic_groups_ctas_per_sm());
                cudaError_t le = launch_biallelic_groups_kernel(ab, std::max(1, bgrid), cs);
                if ( le!=cudaSuccess ) return cuda_fail(ctx, le, "two-allele grouped kernel");
                launches++;
                a.site_list = ab.fb_list; a.site_count = ab.fb_count;
            }
            CK(launch_groups_kernel(nals, a, (char*)sc.grp + (size_t)(nals-1)*per_class, grid, cs));
            if ( gfork ) { CK(cudaEventRecord(ctx->cev_join[nals], cs)); CK(cudaStreamWaitEvent(st, ctx->cev_join[nals], 0)); }
            if ( gtiming ) CK(cudaEventRecord(ctx->kev[nals], st));
            launches++;
        }
        { int rc0 = enqueue_class0(ctx, a, b, r, lists, counts, pl_es, sc, st); if ( rc0 ) return rc0; }
        if ( ctx->opt_adjudicate ) { int rca = enqueue_adjudication(ctx, a, b, lists, counts, list_stride, pl_es, sc, grid, per_class, st, &launches); if ( rca ) return rca; }
        ctx->stats[0] += launches + 1;
        ctx->stats[1] += b->nsites;
        ctx->kev_valid = gtiming;
        return MCB_OK;
    }
    const bool timing = ctx->opt_time_kernels && lists==ctx->d_lists;
    /*  timing mode serialises the classes on the caller's stream (per-class events); otherwise every class runs on
     *  its own stream so that the small persistent grids of the 3-5 allele classes overlap the biallelic one  */
    const bool fork = ctx->opt_concurrent && !timing;
    if ( timing )
    {
        for (int i=0; i<=NCLASS; i++) if ( !ctx->kev[i] ) CK(cudaEventCreate(&ctx->kev[i]));
        CK(cudaEventRecord(ctx->kev[0], st));
    }
    if ( fork )
    {
        { int src = ensure_class_streams(ctx); if ( src ) return src; }
        CK(cudaEventRecord(ctx->cev_fork, st));
    }
    /* launch order of the allele-count classes: digits of opt_order, first digit first (timing mode: ascending) */
    int order[5] = {5,4,3,2,1};
    {
        int64_t v = ctx->opt_order; int seen = 0, tmp[5], k = 4;
        for (; k>=0 && v>0; k--, v/=10) { tmp[k] = (int)(v%10); if ( tmp[k]>=1 && tmp[k]<=5 ) seen |= 1<<tmp[k]; }
        if ( k<0 && v==0 && seen==0x3e ) for (int i=0; i<5; i++) order[i] = tmp[i];
    }
    for (int io=0; io<5; io++)
    {
        int nals = order[io];
        if ( timing ) nals = io + 1;        /* timing mode keeps the ascending order of the event list */
        size_t ring; tile_geometry(ctx, nals, pl_es, &a.tile_smpl, &a.nstage, &ring);
        const bool gpk = a.gp && (a.output_tags & MCB_CALL_FMT_GP);
        const int block = (pl_es==2 || gpk) ? 128 : class_block(ctx, nals);
        a.site_list = lists + (size_t)nals*list_stride; a.site_count = counts + nals;
        a.work_counter = counts + NCLASS + nals;    /* zeroed with the class counts: sites are claimed dynamically */
        /* two alleles, int32 PLs, no GP: one warp per site over a byte-packed shared-memory copy */
        int bw_warps = 0;
        if ( nals==2 && pl_es==4 && !(a.gp && (a.output_tags & MCB_CALL_FMT_GP)) && ctx->opt_warp2!=0 && a.nsmpl<=8192 && !ctx->opt_exact )
        {
            const int ncta = biallelic_ctas_per_sm();
            const size_t per_cta = (size_t)(ctx->smem_per_sm/ncta) - 1024;  /* the kernel is compiled for ncta CTAs per SM */
            int w = biallelic_max_warps();
            while ( w>0 && biallelic_smem_bytes(a.nsmpl, w) > per_cta ) w--;
            if ( ctx->opt_warp2>0 ) w = std::min<int>(w, (int)ctx->opt_warp2);
            const bool tiled_forced = ctx->opt_block || ctx->opt_block_c[2];  /* an explicit CTA size asks for the tiled kernel */
            if ( ctx->opt_warp2>0 ? w>0 : (w*ncta>=16 && !tiled_forced) ) bw_warps = w;   /* few resident warps: the tiled kernel wins */
        }
        if ( bw_warps )
        {
            int grid = (int)std::min<int64_t>(((int64_t)b->nsites + bw_warps - 1)/bw_warps, (int64_t)ctx->nsm*biallelic_ctas_per_sm());
            if ( ctx->opt_blocks_per_sm>0 ) grid = std::min<int>(grid, ctx->nsm*(int)std::min<int64_t>(biallelic_ctas_per_sm(), ctx->opt_blocks_per_sm));
            if ( ctx->opt_bps_c[2]>0 ) grid = std::min<int>(grid, ctx->nsm*(int)std::min<int64_t>(biallelic_ctas_per_sm(), ctx->opt_bps_c[2]));
            cudaStream_t cs = fork ? ctx->cstream[nals] : st;
            if ( fork ) CK(cudaStreamWaitEvent(cs, ctx->cev_fork, 0));
            cudaError_t le = launch_biallelic_warp_kernel(a, ploidy, grid, bw_warps, cs);
            if ( le==cudaSuccess && getenv("MCB_DEBUG_SYNC") ) le = cudaStreamSynchronize(cs);
            if ( le!=cudaSuccess )
            {
                char what[160];
                snprintf(what, sizeof what, "biallelic warp kernel warps=%d grid=%d smem=%zu", bw_warps, grid, biallelic_smem_bytes(a.nsmpl, bw_warps));
                return cuda_fail(ctx, le, what);
            }
            launches++;
            if ( fork ) { CK(cudaEventRecord(ctx->cev_join[nals], cs)); CK(cudaStreamWaitEvent(st, ctx->cev_join[nals], 0)); }
            if ( timing ) CK(cudaEventRecord(ctx->kev[nals], st));
            continue;
        }
        int nb = 1;
        CK(site_kernel_occupancy(nals, ploidy, gpk, block, pl_es, ring, &nb));
        if ( nb<1 ) return cuda_fail(ctx, cudaErrorLaunchOutOfResources, "site kernel does not fit on an SM");
        if ( ctx->opt_blocks_per_sm>0 ) nb = std::min<int>(nb, (int)ctx->opt_blocks_per_sm);
        if ( ctx->opt_bps_c[nals]>0 ) nb = std::min<int>(nb, (int)ctx->opt_bps_c[nals]);
        int grid = (int)std::min<int64_t>((int64_t)b->nsites, (int64_t)ctx->nsm*nb);
        cudaStream_t cs = fork ? ctx->cstream[nals] : st;
        if ( fork ) CK(cudaStreamWaitEvent(cs, ctx->cev_fork, 0));
        /*  3-5 alleles, int32 PLs, every sample diploid, GT + GQ + PL requested: the CTA-per-site kernel of mcall_multi.cu, or the
         *  warp-per-site kernels of mcall_triallelic.cu (3 alleles) and mcall_multi_warp.cu (4 alleles).  Sites they have no
         *  straight-line code for come back on a fallback list, which the general kernel below walks.  */
        const bool multi_ok = nals>=3 && ctx->opt_multi && !ctx->opt_exact && !ctx->opt_block && !ctx->opt_block_c[nals] && pl_es==4 && !ploidy && !gpk && a.gt && a.gq && a.out_pl && !(a.flag & MCB_CALL_KEEPALT)
             && (a.output_tags & (MCB_CALL_FMT_GQ|MCB_CALL_FMT_GP))
             && !((reinterpret_cast<uintptr_t>(a.gt) | reinterpret_cast<uintptr_t>(a.gq) | reinterpret_cast<uintptr_t>(a.out_pl)) & 15);
        int tw_warps = 0, mw_warps = 0, mw_head = 0;
        const int64_t opt_mw = ctx->opt_warp4;
        if ( multi_ok && nals==4 && opt_mw!=0 && multi_block_for(a.nsmpl) )
        {
            /* as many warps as the registers allow; the packed copy that does not fit their shares of shared memory goes to an
               L2-resident tail, which the whole grid must keep within MW_L2_SHARE of L2 (above it the CTA kernel wins) */
            const int ncta = multi_warp_ctas_per_sm();
            const size_t per_cta = (size_t)(ctx->smem_per_sm/ncta) - 1024;
            int w = multi_warp_max_warps();
            if ( opt_mw>0 ) w = std::min<int>(w, (int)opt_mw);
            const int head = multi_warp_head(a.nsmpl, w, per_cta);
            const double tail_all = (double)ctx->nsm*ncta*w*(double)multi_warp_tail_bytes(a.nsmpl, head);
            const bool cta_forced = ctx->opt_mm_block || ctx->opt_mm_block_c[nals] || ctx->opt_mm_nst || ctx->opt_mm_nst_c[nals];
            if ( head>0 && (opt_mw>0 || (!cta_forced && tail_all <= MW_L2_SHARE*(double)ctx->l2_bytes)) ) { mw_warps = w; mw_head = head; }
        }
        if ( multi_ok && nals==3 && ctx->opt_warp3!=0 && multi_block_for(a.nsmpl) )
        {
            const int ncta = triallelic_ctas_per_sm();
            const size_t per_cta = (size_t)(ctx->smem_per_sm/ncta) - 1024;  /* the kernel is compiled for ncta CTAs per SM */
            int w = triallelic_max_warps();
            while ( w>0 && triallelic_smem_bytes(a.nsmpl, w) > per_cta ) w--;
            if ( ctx->opt_warp3>0 ) w = std::min<int>(w, (int)ctx->opt_warp3);
            /* an explicit CTA size or ring depth of the class asks for the CTA kernel; below 12 resident warps per SM it wins */
            const bool cta_forced = ctx->opt_mm_block || ctx->opt_mm_block_c[3] || ctx->opt_mm_nst || ctx->opt_mm_nst_c[3];
            if ( ctx->opt_warp3>0 ? w>0 : (w*ncta>=12 && !cta_forced) ) tw_warps = w;
        }
        if ( tw_warps )
        {
            const int tgrid = (int)std::min<int64_t>(((int64_t)b->nsites + tw_warps - 1)/tw_warps, (int64_t)ctx->nsm*triallelic_ctas_per_sm());
            KArgs am = a;
            am.fb_list = lists + (size_t)(NCLASS + nals)*list_stride;
            am.fb_count = counts + NCLASS + 8 + nals;
            cudaError_t le = launch_triallelic_warp_kernel(am, tgrid, tw_warps, cs);
            if ( le==cudaSuccess && getenv("MCB_DEBUG_SYNC") ) le = cudaStreamSynchronize(cs);
            if ( le!=cudaSuccess )
            {
                char what[160];
                snprintf(what, sizeof what, "3-allele warp kernel warps=%d grid=%d smem=%zu", tw_warps, tgrid, triallelic_smem_bytes(a.nsmpl, tw_warps));
                return cuda_fail(ctx, le, what);
            }
            launches++;
            /* the general kernel now walks the fallback list only */
            a.site_list = am.fb_list; a.site_count = am.fb_count;
            a.work_counter = counts + NCLASS + 16 + nals;
            grid = std::min(grid, ctx->nsm);
        }
        else if ( mw_warps )
        {
            const int ncta = multi_warp_ctas_per_sm();
            const int mgrid = (int)std::min<int64_t>(((int64_t)b->nsites + mw_warps - 1)/mw_warps, (int64_t)ctx->nsm*ncta);
            const size_t tail = multi_warp_tail_bytes(a.nsmpl, mw_head);
            if ( tail && (size_t)ctx->nsm*ncta*mw_warps*tail > sc.mw_tail_bytes[nals] )
            {
                CK(cudaStreamSynchronize(cs));
                if ( sc.mw_tail[nals] ) CK(cudaFree(sc.mw_tail[nals]));
                const size_t want = (size_t)ctx->nsm*ncta*mw_warps*tail;      /* full grid: no regrowth with the next, larger batch */
                CK(cudaMalloc(&sc.mw_tail[nals], want));
                sc.mw_tail_bytes[nals] = want;
            }
            KArgs am = a;
            am.fb_list = lists + (size_t)(NCLASS + nals)*list_stride;
            am.fb_count = counts + NCLASS + 8 + nals;
            cudaError_t le = launch_multi_warp_kernel(am, mgrid, mw_warps, mw_head, sc.mw_tail[nals], cs);
            if ( le==cudaSuccess && getenv("MCB_DEBUG_SYNC") ) le = cudaStreamSynchronize(cs);
            if ( le!=cudaSuccess )
            {
                char what[160];
                snprintf(what, sizeof what, "4-allele warp kernel warps=%d grid=%d head=%d smem=%zu", mw_warps, mgrid, mw_head, multi_warp_smem_bytes(mw_head, mw_warps));
                return cuda_fail(ctx, le, what);
            }
            launches++;
            /* the general kernel now walks the fallback list only */
            a.site_list = am.fb_list; a.site_count = am.fb_count;
            a.work_counter = counts + NCLASS + 16 + nals;
            grid = std::min(grid, ctx->nsm);
        }
        else if ( multi_ok )
        {
            /* CTA size: explicit option, else the class default (sweeps in profiles/), never below what the 12-bit allele counters allow */
            const int minblock = multi_block_for(a.nsmpl);
            int mblock = ctx->opt_mm_block_c[nals] ? (int)ctx->opt_mm_block_c[nals] : (ctx->opt_mm_block ? (int)ctx->opt_mm_block : 128);
            if ( !minblock ) mblock = 0;
            else mblock = std::max(mblock, minblock);
            int nst = ctx->opt_mm_nst_c[nals] ? (int)ctx->opt_mm_nst_c[nals] : (ctx->opt_mm_nst ? (int)ctx->opt_mm_nst : (nals==4 ? 1 : 2));
            const size_t cap = 227u*1024u;
            while ( mblock && nst>1 && multi_smem_bytes(nals, mblock, a.nsmpl, nst) > cap ) nst--;
            if ( mblock && multi_smem_bytes(nals, mblock, a.nsmpl, nst) <= cap )
            {
                int mnb = 0;
                CK(multi_kernel_occupancy(nals, mblock, a.nsmpl, nst, &mnb));
                if ( mnb >= 1 )
                {
                    if ( ctx->opt_bps_c[nals]>0 ) mnb = std::min<int>(mnb, (int)ctx->opt_bps_c[nals]);
                    const int mgrid = (int)std::min<int64_t>((int64_t)b->nsites, (int64_t)ctx->nsm*mnb);
                    const size_t need = multi_scratch_bytes(a.nsmpl, mgrid);
                    if ( need > sc.mm_sums_bytes[nals] )
                    {
                        CK(cudaStreamSynchronize(cs));
                        if ( sc.mm_sums[nals] ) CK(cudaFree(sc.mm_sums[nals]));
                        const size_t want = multi_scratch_bytes(a.nsmpl, ctx->nsm*mnb);      /* full grid: no regrowth with the next, larger batch */
                        CK(cudaMalloc(&sc.mm_sums[nals], want));
                        sc.mm_sums_bytes[nals] = want;
                    }
                    KArgs am = a;
                    am.nstage = nst;
                    am.mm_sums = sc.mm_sums[nals];
                    am.fb_list = lists + (size_t)(NCLASS + nals)*list_stride;
                    am.fb_count = counts + NCLASS + 8 + nals;
                    cudaError_t le = launch_multi_kernel(nals, mblock, am, mgrid, cs);
                    if ( le==cudaSuccess && getenv("MCB_DEBUG_SYNC") ) le = cudaStreamSynchronize(cs);
                    if ( le!=cudaSuccess )
                    {
                        char what[160];
                        snprintf(what, sizeof what, "multi-allelic kernel nals=%d block=%d grid=%d nst=%d smem=%zu", nals, mblock, mgrid, nst, multi_smem_bytes(nals, mblock, a.nsmpl, nst));
                        return cuda_fail(ctx, le, what);
                    }
                    launches++;
                    /* the general kernel now walks the fallback list only */
                    a.site_list = am.fb_list; a.site_count = am.fb_count;
                    a.work_counter = counts + NCLASS + 16 + nals;
                    grid = std::min(grid, ctx->nsm);
                }
            }
        }
        {
            cudaError_t le = launch_site_kernel(nals, ploidy, gpk, block, pl_es, a, grid, ring, cs);
            if ( le==cudaSuccess && getenv("MCB_DEBUG_SYNC") ) le = cudaStreamSynchronize(cs);
            if ( le!=cudaSuccess )
            {
                char what[160];
                snprintf(what, sizeof what, "site kernel nals=%d block=%d pl_es=%d grid=%d ring=%zu tile_smpl=%d nstage=%d", nals, block, pl_es, grid, ring, a.tile_smpl, a.nstage);
                return cuda_fail(ctx, le, what);
            }
        }
        launches++;
        if ( fork ) { CK(cudaEventRecord(ctx->cev_join[nals], cs)); CK(cudaStreamWaitEvent(st, ctx->cev_join[nals], 0)); }
        if ( timing ) CK(cudaEventRecord(ctx->kev[nals], st));
    }
    ctx->kev_valid = timing;
    { int rc0 = enqueue_class0(ctx, a, b, r, lists, counts, pl_es, sc, st); if ( rc0 ) return rc0; }
    launches++;
    if ( ctx->opt_adjudicate ) { int rca = enqueue_adjudication(ctx, a, b, lists, counts, list_stride, pl_es, sc, 0, 0, st, &launches); if ( rca ) return rca; }
    ctx->stats[0] += launches;
    ctx->stats[1] += b->nsites;
    return MCB_OK;
}

extern "C" int mcb_call_device(mcb_ctx *ctx, const mcb_batch *b, const mcb_result *r, void *cuda_stream)
{
    if ( !ctx || !b || !r || !r->ret || b->nsites<0 || !b->pl || !b->pl_off || !b->nals ) return MCB_EINVAL;
    if ( ctx->opt_adjudicate && !r->site_flags ) return MCB_EINVAL;     /* the flagged sites are found from site_flags */
    if ( b->nsites==0 ) return MCB_OK;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t) cuda_stream;
    if ( b->nsites > ctx->list_cap )
    {
        CK(cudaStreamSynchronize(st));
        if ( ctx->d_lists ) CK(cudaFree(ctx->d_lists));
        ctx->list_cap = b->nsites;
        CK(cudaMalloc(&ctx->d_lists, lists_bytes(ctx->list_cap)));
    }
    ctx->stats[0] = ctx->stats[1] = 0;
    return enqueue(ctx, b, r, ctx->d_lists, ctx->d_counts, ctx->list_cap, ctx->d_cursor, ctx->scratch, st);
}

/* ---- host path: slabs double-buffered over two streams ---------------------------------------------- */
static inline size_t pad256(size_t n) { return (n + 255) & ~(size_t)255; }

/*  BCF typed-vector outputs (mcb_result.gt8 / gq8 / pl16): the int32 arrays the kernels wrote are narrowed on the device before
 *  they cross PCIe.  One pass over data that is still in L2 / HBM costs ~1 % of the transfer it shortens.  */
template<typename T> __device__ __forceinline__ T narrow_one(int v)
{
    constexpr int LO = sizeof(T)==1 ? INT8_MIN : INT16_MIN, HI = sizeof(T)==1 ? INT8_MAX : INT16_MAX;
    if ( v==INT32_MIN ) return (T)LO;               /* bcf_int32_missing    -> bcf_int8/16_missing */
    if ( v==INT32_MIN+1 ) return (T)(LO+1);         /* bcf_int32_vector_end -> bcf_int8/16_vector_end */
    return (T)(v > HI ? HI : (v < LO+2 ? LO+2 : v));
}
template<typename T> __global__ void narrow_kernel(const int32_t *src, T *dst, size_t n)
{
    const size_t n4 = n >> 2, stride = (size_t)gridDim.x*blockDim.x;
    for (size_t i = (size_t)blockIdx.x*blockDim.x + threadIdx.x; i < n4; i += stride)
    {
        const int4 v = reinterpret_cast<const int4*>(src)[i];
        T o[4] = { narrow_one<T>(v.x), narrow_one<T>(v.y), narrow_one<T>(v.z), narrow_one<T>(v.w) };
        if ( sizeof(T)==1 ) reinterpret_cast<uint32_t*>(dst)[i] = *reinterpret_cast<uint32_t*>(o);
        else reinterpret_cast<uint2*>(dst)[i] = *reinterpret_cast<uint2*>(o);
    }
    for (size_t i = (n4<<2) + (size_t)blockIdx.x*blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = narrow_one<T>(src[i]);
}
template<typename T> static cudaError_t launch_narrow(const int32_t *src, T *dst, size_t n, int nsm, cudaStream_t st)
{
    if ( !n ) return cudaSuccess;
    const int grid = (int)std::min<size_t>((size_t)nsm*8, (n/4 + 255)/256 + 1);
    narrow_kernel<T><<<grid, 256, 0, st>>>(src, dst, n);
    return cudaGetLastError();
}

extern "C" int mcb_call_host(mcb_ctx *ctx, const mcb_batch *b, const mcb_result *r)
{
    if ( !ctx || !b || !r || !r->ret || b->nsites<0 || !b->pl || !b->pl_off || !b->nals ) return MCB_EINVAL;
    if ( ctx->opt_adjudicate && !r->site_flags ) return MCB_EINVAL;     /* the flagged sites are found from site_flags */
    if ( b->nsites==0 ) return MCB_OK;
    CK(cudaSetDevice(ctx->device));
    const int S = ctx->p.nsmpl, M = ctx->p.max_nals, R = b->nsites;
    ctx->stats[0] = ctx->stats[1] = 0;

    /* per-site PL extents (host knows nals) and a monotonicity check: slabs copy one contiguous PL range */
    if ( b->pl_type!=0 && b->pl_type!=4 && b->pl_type!=2 ) return MCB_EINVAL;
    const int es = b->pl_type==2 ? 2 : 4;               /* bytes per input PL element */
    const int64_t amask = 16/es - 1;                    /* sites start on 16-byte boundaries */
    std::vector<int64_t> ext(R);
    for (int i=0; i<R; i++)
    {
        int n = b->nals[i];
        if ( n > M && n <= MCB_MAX_NALS ) return MCB_EINVAL;    /* the per-site allele arrays (qs, prior_ac, ac, als_map) have stride max_nals */
        ext[i] = (( (int64_t)S*n*(n+1)/2 ) + amask) & ~amask;
        if ( (b->pl_off[i] & amask) || (i && b->pl_off[i] < b->pl_off[i-1] + ext[i-1]) ) return MCB_EINVAL;
    }
    const bool have_ad = ctx->ngroups>1 && b->ad && b->ad_off && b->nad;
    std::vector<int64_t> aext(have_ad ? R : 0);
    for (int i=0; have_ad && i<R; i++)
    {
        aext[i] = (((int64_t)S*b->nad[i]) + 3) & ~(int64_t)3;
        if ( i && b->ad_off[i] < b->ad_off[i-1] + aext[i-1] ) return MCB_EINVAL;
    }
    const bool want_pl = r->pl || r->pl16, want_gt = r->gt || r->gt8;
    const bool want_gq = (r->gq || r->gq8) && (ctx->p.output_tags & (MCB_CALL_FMT_GQ|MCB_CALL_FMT_GP));
    const bool gt8 = r->gt8 != nullptr, gq8 = r->gq8 != nullptr, pl16 = r->pl16 != nullptr;     /* BCF typed outputs */
    const bool want_gp = r->gp && (ctx->p.output_tags & MCB_CALL_FMT_GP);
    const bool compact = r->pl_off_out != nullptr;      /* trimmed PL/GP leave the device compacted */
    int64_t out_total = 0;                              /* int32 units already placed in r->pl */
    std::vector<std::pair<int,int64_t>> slab_base;      /* (first site, base) per slab, applied to pl_off_out at the end */

    /* Compacted output: the PL/GP extent of a slab is known only after its kernels ran.  The host reads the cursor of
       slab k-1 AFTER it has queued the uploads and kernels of slab k, so the copy engines never wait for the host. */
    auto finish = [&](HostSlab &sl) -> int
    {
        if ( !sl.pending ) return MCB_OK;
        sl.pending = false;
        CK(cudaEventSynchronize(sl.cursor_ready));      /* kernels ran, the small outputs (and the cursor) are in h_out */
        const int beg = sl.p_beg, n = sl.p_n;
        const char *ho = sl.h_out - sl.s_out_beg;
        memcpy(r->ret + beg, ho + sl.s_ret, 4*(size_t)n);
        if ( r->als_new ) memcpy(r->als_new + beg, ho + sl.s_als, 4*(size_t)n);
        if ( r->als_map ) memcpy(r->als_map + (size_t)beg*M, ho + sl.s_map, (size_t)n*M);
        if ( r->qual ) memcpy(r->qual + beg, ho + sl.s_qual, 4*(size_t)n);
        if ( r->ac ) memcpy(r->ac + (size_t)beg*M, ho + sl.s_ac, 4*(size_t)n*M);
        if ( r->an ) memcpy(r->an + beg, ho + sl.s_an, 4*(size_t)n);
        if ( r->site_flags ) memcpy(r->site_flags + beg, ho + sl.s_fl, 4*(size_t)n);
        if ( r->diag ) memcpy(r->diag + (size_t)beg*4, ho + sl.s_diag, 32*(size_t)n);
        if ( !compact ) return MCB_OK;
        memcpy(r->pl_off_out + beg, ho + sl.s_ploo, sizeof(int64_t)*(size_t)n);
        const int64_t used = (int64_t)*sl.h_cursor;
        char *base = (char*) sl.dev;
        if ( want_pl && used && pl16 )
        {
            CK(launch_narrow<int16_t>((const int32_t*)(base + sl.p_plout), (int16_t*)(base + sl.p_pl16), (size_t)used, ctx->nsm, sl.stream));
            CK(cudaMemcpyAsync(r->pl16 + out_total, base + sl.p_pl16, (size_t)used*2, cudaMemcpyDeviceToHost, sl.stream));
        }
        else
        if ( want_pl && used ) CK(cudaMemcpyAsync(r->pl + out_total, base + sl.p_plout, (size_t)used*4, cudaMemcpyDeviceToHost, sl.stream));
        if ( want_gp && used ) CK(cudaMemcpyAsync(r->gp + out_total, base + sl.p_gp, (size_t)used*4, cudaMemcpyDeviceToHost, sl.stream));
        slab_base.push_back(std::make_pair(sl.p_beg, out_total));
        out_total += used;
        CK(cudaEventRecord(sl.done, sl.stream));
        return MCB_OK;
    };
    for (int i=0; i<NSLAB; i++) ctx->slab[i].pending = false;

    int beg = 0, islab = 0;
    while ( beg < R )
    {
        /* slab = as many sites as fit the slab budget of PL bytes.  The budget ramps up geometrically from opt_slab_min
           at the start of the call and down again towards its end: the first upload and the last download are the only
           transfers that overlap nothing, so they are kept short; the slabs in between are large (few launches). */
        const int64_t done_bytes = (b->pl_off[beg] - b->pl_off[0])*es;
        const int64_t left_bytes = (b->pl_off[R-1] + ext[R-1] - b->pl_off[beg])*es;
        int64_t budget = std::min<int64_t>(ctx->opt_slab_bytes, std::max<int64_t>(ctx->opt_slab_min, std::min<int64_t>(done_bytes, left_bytes/2)));
        if ( ctx->opt_slab_min<=0 ) budget = ctx->opt_slab_bytes;
        int end = beg; int64_t pl_ints = 0;
        while ( end < R && (end==beg || (pl_ints + ext[end])*es <= budget) ) { pl_ints = b->pl_off[end] + ext[end] - b->pl_off[beg]; end++; }
        const int n = end - beg;
        HostSlab &sl = ctx->slab[islab % NSLAB];
        { int frc = finish(sl); if ( frc ) return frc; }
        CK(cudaEventSynchronize(sl.done));      /* previous use of this stage finished (event starts signalled) */

        /* carve the arena */
        size_t off = 0;
        auto carve = [&](size_t bytes) { size_t o = off; off += pad256(bytes); return o; };
        size_t o_pl = carve((size_t)pl_ints*es), o_plout = want_pl ? carve((size_t)pl_ints*4) : 0;
        size_t o_gp = want_gp ? carve((size_t)pl_ints*4) : 0;
        const int64_t ad0 = have_ad ? b->ad_off[beg] : 0, ad_ints = have_ad ? b->ad_off[end-1] + aext[end-1] - ad0 : 0;
        size_t o_ad = have_ad ? carve((size_t)ad_ints*4) : 0;
        size_t o_gt = want_gt ? carve(8*(size_t)n*S) : 0, o_gq = want_gq ? carve(4*(size_t)n*S) : 0;
        size_t o_gt8 = (want_gt && gt8) ? carve(2*(size_t)n*S) : 0, o_gq8 = (want_gq && gq8) ? carve((size_t)n*S) : 0;
        size_t o_pl16 = (want_pl && pl16) ? carve((size_t)pl_ints*2) : 0;
        /* small inputs, contiguous: one upload */
        const size_t in_beg = off;
        size_t o_ploff = carve(sizeof(int64_t)*n), o_nals = carve(n), o_unseen = carve(n), o_pid = carve(2*(size_t)n);
        size_t o_qs = carve(sizeof(float)*(size_t)n*M), o_nqs = carve(n);
        size_t o_pan = carve(sizeof(int32_t)*n), o_pac = carve(sizeof(int32_t)*(size_t)n*M);
        size_t o_adoff = have_ad ? carve(sizeof(int64_t)*n) : 0, o_nad = have_ad ? carve(n) : 0;
        const size_t in_end = off;
        /* small outputs, contiguous: one download */
        const size_t out_beg = off;
        size_t o_ret = carve(4*(size_t)n), o_als = carve(4*(size_t)n), o_map = carve((size_t)n*M), o_qual = carve(4*(size_t)n);
        size_t o_ac = carve(4*(size_t)n*M), o_an = carve(4*(size_t)n), o_fl = carve(4*(size_t)n), o_diag = carve(32*(size_t)n);
        size_t o_ploo = compact ? carve(sizeof(int64_t)*n) : 0;
        const size_t out_end = off;
        if ( in_end - in_beg > sl.h_in_bytes )
        {
            if ( sl.h_in ) CK(cudaFreeHost(sl.h_in));
            sl.h_in_bytes = (in_end - in_beg) + (in_end - in_beg)/4;
            CK(cudaHostAlloc(&sl.h_in, sl.h_in_bytes, cudaHostAllocDefault));
        }
        if ( out_end - out_beg > sl.h_out_bytes )
        {
            if ( sl.h_out ) CK(cudaFreeHost(sl.h_out));
            sl.h_out_bytes = (out_end - out_beg) + (out_end - out_beg)/4;
            CK(cudaHostAlloc(&sl.h_out, sl.h_out_bytes, cudaHostAllocDefault));
        }
        if ( off > sl.dev_bytes )
        {
            if ( sl.dev ) CK(cudaFree(sl.dev));
            sl.dev_bytes = off + off/8;
            CK(cudaMalloc(&sl.dev, sl.dev_bytes));
        }
        if ( n > sl.list_cap )
        {
            if ( sl.lists ) CK(cudaFree(sl.lists));
            sl.list_cap = n + n/8;
            CK(cudaMalloc(&sl.lists, lists_bytes(sl.list_cap)));
        }
        char *base = (char*) sl.dev;
        cudaStream_t st = sl.stream;
        const int64_t pl0 = b->pl_off[beg];
#define H2D(dst,src,bytes) CK(cudaMemcpyAsync(base+(dst), (src), (bytes), cudaMemcpyHostToDevice, st))
        H2D(o_pl, (const char*)b->pl + (size_t)pl0*es, (size_t)pl_ints*es);
        if ( have_ad ) H2D(o_ad, b->ad + ad0, (size_t)ad_ints*4);
        {
            char *hi = sl.h_in - in_beg;
            memcpy(hi + o_ploff, b->pl_off + beg, sizeof(int64_t)*n);
            memcpy(hi + o_nals, b->nals + beg, n);
            if ( b->unseen ) memcpy(hi + o_unseen, b->unseen + beg, n);
            if ( b->ploidy_id ) memcpy(hi + o_pid, b->ploidy_id + beg, 2*(size_t)n);
            if ( b->qs ) memcpy(hi + o_qs, b->qs + (size_t)beg*M, sizeof(float)*(size_t)n*M);
            if ( b->nqs ) memcpy(hi + o_nqs, b->nqs + beg, n);
            if ( b->prior_an ) memcpy(hi + o_pan, b->prior_an + beg, sizeof(int32_t)*n);
            if ( b->prior_ac ) memcpy(hi + o_pac, b->prior_ac + (size_t)beg*M, sizeof(int32_t)*(size_t)n*M);
            if ( have_ad ) { memcpy(hi + o_adoff, b->ad_off + beg, sizeof(int64_t)*n); memcpy(hi + o_nad, b->nad + beg, n); }
            H2D(in_beg, sl.h_in, in_end - in_beg);
        }
#undef H2D
        /* device views: pl pointers are biased by -pl0 so that the absolute pl_off[] stay valid */
        mcb_batch db; memset(&db, 0, sizeof db);
        db.nsites = n;
        db.pl = (const int32_t*)((const char*)(base+o_pl) - (size_t)pl0*es); db.pl_off = (const int64_t*)(base+o_ploff);
        db.pl_type = b->pl_type;
        db.nals = (const uint8_t*)(base+o_nals);
        db.unseen = b->unseen ? (const uint8_t*)(base+o_unseen) : nullptr;
        db.ploidy_id = b->ploidy_id ? (const uint16_t*)(base+o_pid) : nullptr;
        db.qs = b->qs ? (const float*)(base+o_qs) : nullptr;
        db.nqs = b->nqs ? (const uint8_t*)(base+o_nqs) : nullptr;
        db.prior_an = b->prior_an ? (const int32_t*)(base+o_pan) : nullptr;
        db.prior_ac = b->prior_ac ? (const int32_t*)(base+o_pac) : nullptr;
        if ( have_ad )
        {
            db.ad = (const int32_t*)(base+o_ad) - ad0; db.ad_off = (const int64_t*)(base+o_adoff); db.nad = (const uint8_t*)(base+o_nad);
        }
        mcb_result dr; memset(&dr, 0, sizeof dr);
        dr.ret = (int32_t*)(base+o_ret); dr.als_new = (uint32_t*)(base+o_als); dr.als_map = (int8_t*)(base+o_map);
        dr.qual = (float*)(base+o_qual); dr.ac = (int32_t*)(base+o_ac); dr.an = (int32_t*)(base+o_an);
        dr.site_flags = (uint32_t*)(base+o_fl); dr.diag = (double*)(base+o_diag);
        dr.gt = want_gt ? (int32_t*)(base+o_gt) : nullptr;
        dr.gq = want_gq ? (int32_t*)(base+o_gq) : nullptr;
        dr.pl = want_pl ? (int32_t*)(base+o_plout) - pl0 : nullptr;
        dr.gp = want_gp ? (float*)(base+o_gp) - pl0 : nullptr;
        if ( compact )
        {
            dr.pl = want_pl ? (int32_t*)(base+o_plout) : nullptr;
            dr.gp = want_gp ? (float*)(base+o_gp) : nullptr;
            dr.pl_off_out = (int64_t*)(base+o_ploo);
        }

        int rc = enqueue(ctx, &db, &dr, sl.lists, sl.counts, sl.list_cap, sl.cursor, sl.scratch, st);
        if ( rc ) return rc;

#define D2H(dst,src,bytes) CK(cudaMemcpyAsync((dst), base+(src), (bytes), cudaMemcpyDeviceToHost, st))
        if ( compact ) CK(cudaMemcpyAsync(sl.h_cursor, sl.cursor, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        D2H(sl.h_out, out_beg, out_end - out_beg);
        CK(cudaEventRecord(sl.cursor_ready, st));
        sl.s_out_beg = out_beg; sl.s_ret = o_ret; sl.s_als = o_als; sl.s_map = o_map; sl.s_qual = o_qual; sl.s_ac = o_ac;
        sl.s_an = o_an; sl.s_fl = o_fl; sl.s_diag = o_diag; sl.s_ploo = o_ploo;
        sl.pending = true; sl.p_beg = beg; sl.p_n = n; sl.p_plout = o_plout; sl.p_gp = o_gp; sl.p_pl16 = o_pl16;
        if ( want_gt && gt8 )
        {
            CK(launch_narrow<int8_t>((const int32_t*)(base+o_gt), (int8_t*)(base+o_gt8), 2*(size_t)n*S, ctx->nsm, st));
            D2H(r->gt8 + (size_t)beg*S*2, o_gt8, 2*(size_t)n*S);
        }
        else
        if ( want_gt ) D2H(r->gt + (size_t)beg*S*2, o_gt, 8*(size_t)n*S);
        if ( want_gq && gq8 )
        {
            CK(launch_narrow<int8_t>((const int32_t*)(base+o_gq), (int8_t*)(base+o_gq8), (size_t)n*S, ctx->nsm, st));
            D2H(r->gq8 + (size_t)beg*S, o_gq8, (size_t)n*S);
        }
        else
        if ( want_gq ) D2H(r->gq + (size_t)beg*S, o_gq, 4*(size_t)n*S);
        if ( !compact )
        {
            if ( want_pl && pl16 )
            {
                CK(launch_narrow<int16_t>((const int32_t*)(base+o_plout), (int16_t*)(base+o_pl16), (size_t)pl_ints, ctx->nsm, st));
                D2H(r->pl16 + pl0, o_pl16, (size_t)pl_ints*2);
            }
            else
            if ( want_pl ) D2H(r->pl + pl0, o_plout, (size_t)pl_ints*4);
            if ( want_gp ) D2H(r->gp + pl0, o_gp, (size_t)pl_ints*4);
            CK(cudaEventRecord(sl.done, st));
        }
        /* the host-side tail of the PREVIOUS slab (scatter of its small outputs, compacted PL download): its kernels
           have had the whole upload of this one to finish */
        if ( islab ) { int frc = finish(ctx->slab[(islab-1) % NSLAB]); if ( frc ) return frc; }
#undef D2H
        beg = end; islab++;
    }
    for (int k=0; k<NSLAB; k++) { int frc = finish(ctx->slab[(islab + k) % NSLAB]); if ( frc ) return frc; }   /* oldest first */
    for (int k=0; k<NSLAB; k++) CK(cudaStreamSynchronize(ctx->slab[k].stream));
    for (size_t k=0; k<slab_base.size(); k++)           /* slab-local offsets -> offsets into r->pl */
    {
        const int first = slab_base[k].first, last = k+1<slab_base.size() ? slab_base[k+1].first : R;
        for (int i=first; i<last; i++) if ( r->pl_off_out[i] >= 0 ) r->pl_off_out[i] += slab_base[k].second;
    }
    ctx->stats[2] = out_total;
    return MCB_OK;
}
