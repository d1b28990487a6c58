"""ctypes mirror of include/mcall_b200.h (the C-ABI structs) plus numpy holders for one batch.

These are plain data definitions; nothing here computes.  The same struct layout is used by the
product library (bcftools_b200/csrc -> libmcall_b200.so) and, in tests only, by the oracle
libraries, so that parity tests hand identical bytes to both sides.
"""
import ctypes as C
import numpy as np

# flags, identical to call.h:32-39 in the reference
CALL_KEEPALT = 1 << 0
CALL_VARONLY = 1 << 1
CALL_FMT_GQ = 1 << 6
CALL_FMT_GP = 1 << 7

INT32_MISSING = -2**31            # bcf_int32_missing  [htslib]
INT32_VECTOR_END = -2**31 + 1     # bcf_int32_vector_end
FLOAT_MISSING_BITS = 0x7F800001
FLOAT_VECTOR_END_BITS = 0x7F800002

SITE_PL_DROPPED = 1 << 0
SITE_NEAR_TIE = 1 << 1
SITE_UNSEEN_SEL = 1 << 2
SITE_TOO_MANY_ALS = 1 << 3
SITE_NO_QS = 1 << 4
SITE_REF_GT = 1 << 5
SITE_ADJUDICATED = 1 << 9        # near tie evaluated again with the literal phase 1 (option "adjudicate"); with SITE_NEAR_TIE

MCB_OK, MCB_EINVAL, MCB_ENOMEM, MCB_ECUDA, MCB_ENODEV, MCB_EPL, MCB_EQS, MCB_EPRIOR = 0, -1, -2, -3, -4, -5, -6, -7


class McbParams(C.Structure):
    _fields_ = [
        ("nsmpl", C.c_int32), ("max_nals", C.c_int32),
        ("theta", C.c_double),
        ("init_ploidy", C.c_void_p),
        ("flag", C.c_uint32), ("output_tags", C.c_uint32),
        ("ngroups", C.c_int32),
        ("grp_off", C.c_void_p), ("grp_smpl", C.c_void_p),
        ("use_prior", C.c_int32), ("device", C.c_int32),
        ("tie_eps", C.c_double),
    ]


class McbBatch(C.Structure):
    _fields_ = [
        ("nsites", C.c_int32),
        ("pl", C.c_void_p), ("pl_off", C.c_void_p),
        ("nals", C.c_void_p), ("unseen", C.c_void_p), ("ploidy_id", C.c_void_p),
        ("qs", C.c_void_p), ("nqs", C.c_void_p),
        ("ad", C.c_void_p), ("ad_off", C.c_void_p), ("nad", C.c_void_p),
        ("prior_an", C.c_void_p), ("prior_ac", C.c_void_p),
        ("pl_type", C.c_int32),
    ]


class McbResult(C.Structure):
    _fields_ = [
        ("ret", C.c_void_p), ("als_new", C.c_void_p), ("als_map", C.c_void_p), ("qual", C.c_void_p),
        ("ac", C.c_void_p), ("an", C.c_void_p), ("site_flags", C.c_void_p), ("diag", C.c_void_p),
        ("gt", C.c_void_p), ("gq", C.c_void_p), ("gp", C.c_void_p), ("pl", C.c_void_p), ("pl_off_out", C.c_void_p),
        ("gt8", C.c_void_p), ("gq8", C.c_void_p), ("pl16", C.c_void_p),
    ]


BATCH_FIELDS = {  # name -> numpy dtype
    "pl": np.int32, "pl_off": np.int64, "nals": np.uint8, "unseen": np.uint8, "ploidy_id": np.uint16,
    "qs": np.float32, "nqs": np.uint8, "ad": np.int32, "ad_off": np.int64, "nad": np.uint8,
    "prior_an": np.int32, "prior_ac": np.int32,
}
RESULT_FIELDS = {
    "ret": np.int32, "als_new": np.uint32, "als_map": np.int8, "qual": np.float32, "ac": np.int32,
    "an": np.int32, "site_flags": np.uint32, "diag": np.float64, "gt": np.int32, "gq": np.int32,
    "gp": np.float32, "pl": np.int32, "pl_off_out": np.int64,
    "gt8": np.int8, "gq8": np.int8, "pl16": np.int16,
}


def _ptr(a):
    return None if a is None else a.ctypes.data


class CallParams:
    """Host-side description of what mcall_init() reads from call_t (mcall.c:361-417)."""

    def __init__(self, nsmpl, max_nals=5, theta=1.1e-3, init_ploidy=None, flag=0, output_tags=0,
                 groups=None, use_prior=False, device=0, tie_eps=0.0):
        self.nsmpl, self.max_nals, self.theta = int(nsmpl), int(max_nals), float(theta)
        self.init_ploidy = None if init_ploidy is None else np.ascontiguousarray(init_ploidy, np.uint8)
        self.flag, self.output_tags = int(flag), int(output_tags)
        self.use_prior, self.device, self.tie_eps = bool(use_prior), int(device), float(tie_eps)
        # groups: list of lists of sample indices (smpl_grp_t.smpl), or None = pooled
        self.groups = None
        self.grp_off = self.grp_smpl = None
        if groups is not None and len(groups) > 1:
            self.groups = [list(map(int, g)) for g in groups]
            self.grp_off = np.zeros(len(groups) + 1, np.uint32)
            self.grp_off[1:] = np.cumsum([len(g) for g in self.groups])
            self.grp_smpl = np.array([s for g in self.groups for s in g], np.uint32)
            assert len(self.grp_smpl) == self.nsmpl and len(set(self.grp_smpl.tolist())) == self.nsmpl

    @property
    def ngroups(self):
        return 1 if self.groups is None else len(self.groups)

    def c_struct(self):
        p = McbParams()
        p.nsmpl, p.max_nals, p.theta = self.nsmpl, self.max_nals, self.theta
        p.init_ploidy = _ptr(self.init_ploidy)
        p.flag, p.output_tags = self.flag, self.output_tags
        p.ngroups = self.ngroups
        p.grp_off, p.grp_smpl = _ptr(self.grp_off), _ptr(self.grp_smpl)
        p.use_prior, p.device, p.tie_eps = int(self.use_prior), self.device, self.tie_eps
        return p


def pad4(n):
    return (int(n) + 3) & ~3


class HostBatch:
    """numpy arrays of one mcb_batch (host memory)."""

    def __init__(self, nsmpl, max_nals, nals, pl_blocks=None, pl=None, pl_off=None, unseen=None, ploidy_id=None,
                 qs=None, nqs=None, ad_blocks=None, prior_an=None, prior_ac=None):
        self.nsmpl, self.max_nals = int(nsmpl), int(max_nals)
        self.nals = np.ascontiguousarray(nals, np.uint8)
        R = self.nsites = len(self.nals)
        ngt = self.nals.astype(np.int64) * (self.nals.astype(np.int64) + 1) // 2
        if pl is None:
            sizes = np.array([pad4(nsmpl * g) for g in ngt], np.int64)
            self.pl_off = np.zeros(R, np.int64)
            if R:
                self.pl_off[1:] = np.cumsum(sizes)[:-1]
            self.pl = np.full(int(sizes.sum()) if R else 0, INT32_VECTOR_END, np.int32)
            for i, blk in enumerate(pl_blocks):
                blk = np.asarray(blk, np.int32).reshape(-1)
                assert blk.size == nsmpl * ngt[i], (i, blk.size, nsmpl, ngt[i])
                self.pl[self.pl_off[i]:self.pl_off[i] + blk.size] = blk
        else:
            self.pl = np.ascontiguousarray(pl, np.int32)
            self.pl_off = np.ascontiguousarray(pl_off, np.int64)
        self.ngt = ngt
        self.unseen = np.zeros(R, np.uint8) if unseen is None else np.ascontiguousarray(unseen, np.uint8)
        self.ploidy_id = None if ploidy_id is None else np.ascontiguousarray(ploidy_id, np.uint16)
        self.qs = None
        if qs is not None:
            self.qs = np.zeros((R, max_nals), np.float32)
            q = np.asarray(qs, np.float32)
            self.qs[:, :q.shape[1]] = q
        self.nqs = None if nqs is None else np.ascontiguousarray(nqs, np.uint8)
        self.ad = self.ad_off = self.nad = None
        if ad_blocks is not None:
            self.nad = np.array([np.asarray(a).reshape(nsmpl, -1).shape[1] for a in ad_blocks], np.uint8)
            sizes = np.array([pad4(nsmpl * int(n)) for n in self.nad], np.int64)
            self.ad_off = np.zeros(R, np.int64)
            if R:
                self.ad_off[1:] = np.cumsum(sizes)[:-1]
            self.ad = np.full(int(sizes.sum()) if R else 0, INT32_VECTOR_END, np.int32)
            for i, blk in enumerate(ad_blocks):
                blk = np.asarray(blk, np.int32).reshape(-1)
                self.ad[self.ad_off[i]:self.ad_off[i] + blk.size] = blk
        self.prior_an = None if prior_an is None else np.ascontiguousarray(prior_an, np.int32)
        self.prior_ac = None
        if prior_ac is not None:
            self.prior_ac = np.full((R, max_nals), INT32_VECTOR_END, np.int32)
            a = np.asarray(prior_ac, np.int32)
            self.prior_ac[:, :a.shape[1]] = a

    pl_type = 0

    def site_pl(self, i):
        return self.pl[self.pl_off[i]:self.pl_off[i] + self.nsmpl * int(self.ngt[i])].reshape(self.nsmpl, -1)

    def c_struct(self):
        b = McbBatch()
        b.nsites = self.nsites
        for name in BATCH_FIELDS:
            setattr(b, name, _ptr(getattr(self, name)))
        b.pl_type = getattr(self, "pl_type", 0)
        return b

    def to_int16(self):
        """Same batch with the PL slab as BCF-style int16 typed vectors (sentinels INT16_MIN / INT16_MIN+1), sites on
        16-byte boundaries.  Values must fit (PL <= 32767)."""
        import copy
        nb = copy.copy(self)
        S = self.nsmpl
        sizes = (S * self.ngt + 7) & ~7
        nb.pl_off = np.zeros(self.nsites, np.int64)
        if self.nsites:
            nb.pl_off[1:] = np.cumsum(sizes)[:-1]
        nb.pl = np.full(int(sizes.sum()) if self.nsites else 0, -32767, np.int16)
        for i in range(self.nsites):
            src = self.pl[self.pl_off[i]:self.pl_off[i] + S * int(self.ngt[i])]
            dst = np.where(src == INT32_MISSING, -32768, np.where(src == INT32_VECTOR_END, -32767, src))
            assert dst.max(initial=0) <= 32767
            nb.pl[nb.pl_off[i]:nb.pl_off[i] + src.size] = dst.astype(np.int16)
        nb.pl_type = 2
        return nb

    def subset(self, idx):
        """Batch restricted to the given sites (copies)."""
        idx = list(map(int, idx))
        return HostBatch(self.nsmpl, self.max_nals, self.nals[idx], pl_blocks=[self.site_pl(i) for i in idx],
                         unseen=self.unseen[idx], ploidy_id=None if self.ploidy_id is None else self.ploidy_id[idx],
                         qs=None if self.qs is None else self.qs[idx], nqs=None if self.nqs is None else self.nqs[idx],
                         ad_blocks=None if self.ad is None else [self.site_ad(i) for i in idx],
                         prior_an=None if self.prior_an is None else self.prior_an[idx],
                         prior_ac=None if self.prior_ac is None else self.prior_ac[idx])

    def site_ad(self, i):
        return self.ad[self.ad_off[i]:self.ad_off[i] + self.nsmpl * int(self.nad[i])].reshape(self.nsmpl, -1)


class HostResult:
    """numpy arrays of one mcb_result (host memory), sized for a HostBatch."""

    def __init__(self, batch, want_gp=False, fill=True, compact=False, typed=False):
        R, S, M = batch.nsites, batch.nsmpl, batch.max_nals
        self.typed = typed
        self.batch = batch
        self.ret = np.zeros(R, np.int32)
        self.als_new = np.zeros(R, np.uint32)
        self.als_map = np.full((R, M), -1, np.int8)
        self.qual = np.zeros(R, np.float32)
        self.ac = np.zeros((R, M), np.int32)
        self.an = np.zeros(R, np.int32)
        self.site_flags = np.zeros(R, np.uint32)
        self.diag = np.zeros((R, 4), np.float64)
        self.gt = np.zeros((R, S, 2), np.int32)
        self.gq = np.zeros((R, S), np.int32)
        self.gp = np.zeros(batch.pl.size, np.float32) if want_gp else None
        self.pl = np.zeros(batch.pl.size, np.int32)
        # compact=True: trimmed PL/GP blocks are packed at the front of pl/gp, site i at pl_off_out[i]
        self.pl_off_out = np.full(R, -1, np.int64) if compact else None
        # typed=True (mcb_call_host): GT/GQ/PL arrive as BCF typed vectors (int8/int8/int16) instead of int32
        self.gt8 = self.gq8 = self.pl16 = None
        if typed:
            self.gt8 = np.zeros((R, S, 2), np.int8)
            self.gq8 = np.zeros((R, S), np.int8)
            self.pl16 = np.zeros(batch.pl.size, np.int16)
            self.gt = self.gq = self.pl = None

    def widen(self):
        """typed results -> the int32 arrays of the reference interface (BCF sentinels mapped to the int32 ones)."""
        def w(a, bits):
            lo = -(1 << (bits - 1))
            o = a.astype(np.int32)
            o[a == lo] = np.iinfo(np.int32).min
            o[a == lo + 1] = np.iinfo(np.int32).min + 1
            return o
        self.gt, self.gq, self.pl = w(self.gt8, 8), w(self.gq8, 8), w(self.pl16, 16)
        return self

    def _out_off(self, i):
        return self.batch.pl_off[i] if self.pl_off_out is None else self.pl_off_out[i]

    def c_struct(self):
        r = McbResult()
        for name in RESULT_FIELDS:
            setattr(r, name, _ptr(getattr(self, name)))
        return r

    def site_pl(self, i):
        """Trimmed PL block of site i: [nsmpl][G'] with G' from ret[i]."""
        n = int(self.ret[i])
        g = n * (n + 1) // 2
        o = self._out_off(i)
        return self.pl[o:o + self.batch.nsmpl * g].reshape(self.batch.nsmpl, g)

    def site_gp(self, i):
        n = int(self.ret[i])
        g = n * (n + 1) // 2
        o = self._out_off(i)
        return self.gp[o:o + self.batch.nsmpl * g].reshape(self.batch.nsmpl, g)
