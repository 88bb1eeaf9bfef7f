"""ctypes binding of libhomulator_b200.so + host-side mirror of the reference's operation objects.

The reference exposes `OP(label, maxLevel, currentLevel, alpha, Config*, Arch*)` + `simulate()` for
OP in {HMULT, HROTATE, HADD, PMULT, PADD} (reference include/Operation.h:200-319).  The classes at the
bottom keep that constructor shape; `simulate()` runs the operation on seeded synthetic data on the GPU
and returns measured microseconds and the reference-shaped instruction counts.
"""
import ctypes as C
import math
import os

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

HML_MAX_STAGES = 48


class HmlError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("homulator_b200 error %d: %s" % (code, msg))
        self.code = code


class _StageCount(C.Structure):
    _fields_ = [("label", C.c_char * 48), ("opcode", C.c_char * 16), ("limb_ops", C.c_uint64), ("instructions", C.c_uint64)]


class _Counts(C.Structure):
    _fields_ = [("ntt", C.c_uint64), ("intt", C.c_uint64), ("mult", C.c_uint64), ("bconv_step2", C.c_uint64),
                ("automorph", C.c_uint64), ("total", C.c_uint64), ("driver_total", C.c_uint64), ("n_stages", C.c_uint32),
                ("stages", _StageCount * HML_MAX_STAGES)]


class _ShardInfo(C.Structure):
    _fields_ = [("gather1_slots", C.c_uint32), ("gather2_slots", C.c_uint32), ("n_own_q", C.c_uint32), ("n_own_p", C.c_uint32),
                ("own_q", C.c_uint32 * 128), ("own_p", C.c_uint32 * 128), ("owner", C.c_uint32 * 128), ("slot", C.c_uint32 * 128)]


class _ExecCounts(C.Structure):
    _fields_ = [("ntt_limbs", C.c_uint64), ("intt_limbs", C.c_uint64), ("ewe_limbs", C.c_uint64),
                ("bconv_limb_macs", C.c_uint64), ("automorph_limbs", C.c_uint64), ("kernel_launches", C.c_uint64)]


class _TraceOp(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("dst", C.c_uint32), ("a", C.c_uint32), ("b", C.c_uint32)]


class _Profile(C.Structure):
    _fields_ = [("us", C.c_double * 5), ("launches", C.c_uint64 * 5), ("total_us", C.c_double)]


def lib_path():
    return os.path.join(HERE, "libhomulator_b200.so")


# every symbol include/homulator_b200.h declares (tests check the library exports all of them)
EXPORTS = [
    "hml_ctx_create", "hml_ctx_create_params", "hml_ctx_destroy", "hml_last_error", "hml_last_create_error",
    "hml_ring_degree", "hml_n_moduli", "hml_get_moduli", "hml_get_roots", "hml_dev_alloc", "hml_dev_free", "hml_h2d",
    "hml_d2h", "hml_sync", "hml_key_pack", "hml_ntt", "hml_intt", "hml_ntt_batch", "hml_intt_batch", "hml_ewe", "hml_automorph", "hml_bconv", "hml_bconv_batch", "hml_keyswitch", "hml_rescale",
    "hml_hmult", "hml_hrotate", "hml_hadd", "hml_pmult", "hml_padd", "hml_pmult_add", "hml_hmult_batch", "hml_hrotate_batch",
    "hml_hmult_host", "hml_hrotate_host", "hml_hmult_host_packed", "hml_hrotate_host_packed", "hml_packed_bytes", "hml_pack_host",
    "hml_unpack_host", "hml_host_alloc_pinned", "hml_host_free_pinned", "hml_trace_counts",
    "hml_get_counts", "hml_buffer_plan", "hml_exec_counts_get", "hml_exec_counts_reset", "hml_cli_main", "hml_profile_begin", "hml_profile_end",
    "hml_shard_layout", "hml_keyswitch_shard_begin", "hml_keyswitch_shard_mid", "hml_keyswitch_shard_end",
    "hml_keyswitch_shard_mid_p2p", "hml_keyswitch_shard_end_p2p", "hml_shard_signal", "hml_shard_wait", "hml_shard_sync",
    "hml_ipc_export", "hml_ipc_import", "hml_ipc_close", "hml_rescale_shard_begin", "hml_rescale_shard_end",
    "hml_shard_status", "hml_shard_create", "hml_shard_destroy", "hml_shard_handles", "hml_shard_connect_ipc",
    "hml_shard_connect_local", "hml_shard_prepare", "hml_shard_check", "hml_shard_own_limbs", "hml_keyswitch_sharded",
    "hml_hrotate_sharded", "hml_hmult_sharded", "hml_rescale_sharded", "hml_ew_sharded", "hml_group_op", "hml_hrotate_hoisted",
    "hml_replay_create", "hml_replay_bind", "hml_replay_run", "hml_replay_slot", "hml_replay_slot_level", "hml_replay_destroy",
    "hml_shard_create_ex", "hml_hrotate_hoisted_sharded", "hml_group_hrotate_hoisted", "hml_hrotate_sum_hoisted",
    "hml_hrotate_bsgs_hoisted", "hml_hmult_sum", "hml_hrotate_sum_hoisted_sharded", "hml_group_hrotate_sum_hoisted",
    "hml_hmult_sum_sharded", "hml_group_hmult_sum",
]


KEY_PACKED = 0x80000000  # HML_KEY_PACKED: OR into evk_q_limbs when the key went through Context.key_pack


def load_library():
    """Load the in-tree C-ABI library (building it first when a toolkit is present).  Raises if absent."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    from .build import build
    build()  # mtime-guarded: rebuilds only when a source is newer than the library (no-op on a box without nvcc)
    L = C.CDLL(path)
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
    L.hml_ctx_create.argtypes = [C.c_char_p, u32, u32, i32, C.POINTER(vp)]
    L.hml_ctx_create_params.argtypes = [u32, u32, u32, u32, u32, i32, C.POINTER(vp)]
    L.hml_ctx_destroy.argtypes = [vp]
    L.hml_ctx_destroy.restype = None
    L.hml_last_error.argtypes = [vp]
    L.hml_last_error.restype = C.c_char_p
    L.hml_last_create_error.restype = C.c_char_p
    L.hml_ring_degree.argtypes = [vp]
    L.hml_ring_degree.restype = u32
    L.hml_n_moduli.argtypes = [vp]
    L.hml_n_moduli.restype = u32
    L.hml_get_moduli.argtypes = [vp, C.POINTER(u64), u32]
    L.hml_get_roots.argtypes = [vp, C.POINTER(u64), u32]
    L.hml_ntt.argtypes = [vp, vp, vp, C.POINTER(u32), u32, vp]
    L.hml_intt.argtypes = [vp, vp, vp, C.POINTER(u32), u32, vp]
    L.hml_ntt_batch.argtypes = [vp, vp, vp, C.POINTER(u32), u32, u32, vp]
    L.hml_intt_batch.argtypes = [vp, vp, vp, C.POINTER(u32), u32, u32, vp]
    L.hml_ewe.argtypes = [vp, vp, vp, vp, vp, i32, vp, C.POINTER(u32), u32, vp]
    L.hml_automorph.argtypes = [vp, vp, vp, u64, u32, vp]
    L.hml_bconv.argtypes = [vp, vp, C.POINTER(u32), u32, vp, C.POINTER(u32), u32, vp]
    L.hml_bconv_batch.argtypes = [vp, vp, C.POINTER(u32), u32, vp, C.POINTER(u32), u32, u32, vp]
    L.hml_keyswitch.argtypes = [vp, u32, vp, vp, u32, vp, vp, vp]
    L.hml_rescale.argtypes = [vp, u32, vp, vp, vp]
    L.hml_hmult.argtypes = [vp, u32, vp, vp, vp, u32, vp, vp]
    L.hml_hrotate.argtypes = [vp, u32, vp, vp, u32, u64, vp, vp]
    for f in ("hml_hadd", "hml_pmult", "hml_padd"):
        getattr(L, f).argtypes = [vp, u32, vp, vp, vp, vp]
    L.hml_pmult_add.argtypes = [vp, u32, vp, vp, vp, vp, vp]
    L.hml_hmult_batch.argtypes = [vp, u32, u32, vp, vp, vp, u32, vp, vp]
    L.hml_hmult_sum.argtypes = [vp, u32, u32, C.POINTER(vp), C.POINTER(vp), u32, vp, u32, vp, vp]
    L.hml_hrotate_batch.argtypes = [vp, u32, u32, vp, vp, u32, u64, vp, vp]
    L.hml_hmult_host.argtypes = [vp, u32, u32, vp, vp, vp, u32, vp]
    L.hml_hrotate_host.argtypes = [vp, u32, u32, vp, vp, u32, u64, vp]
    L.hml_hmult_host_packed.argtypes = [vp, u32, u32, vp, vp, vp, u32, vp]
    L.hml_hrotate_host_packed.argtypes = [vp, u32, u32, vp, vp, u32, u64, vp]
    L.hml_packed_bytes.argtypes = [vp, u64]
    L.hml_packed_bytes.restype = u64
    L.hml_pack_host.argtypes = [vp, vp, u64, vp]
    L.hml_unpack_host.argtypes = [vp, vp, u64, vp]
    L.hml_host_alloc_pinned.argtypes = [vp, u64, C.POINTER(vp)]
    L.hml_host_free_pinned.argtypes = [vp, vp]
    L.hml_trace_counts.argtypes = [C.c_char_p, u32, u32, u32, u32, u32, u32, u32, C.POINTER(_Counts)]
    L.hml_get_counts.argtypes = [vp, C.c_char_p, u32, C.POINTER(_Counts)]
    L.hml_buffer_plan.argtypes = [vp, C.c_char_p, u32, C.c_char_p, u64]
    L.hml_exec_counts_get.argtypes = [vp, C.POINTER(_ExecCounts)]
    L.hml_exec_counts_reset.argtypes = [vp]
    L.hml_cli_main.argtypes = [i32, C.POINTER(C.c_char_p)]
    L.hml_shard_layout.argtypes = [u32, u32, u32, u32, C.POINTER(_ShardInfo)]
    L.hml_keyswitch_shard_begin.argtypes = [vp, u32, u32, u32, vp, vp, vp]
    L.hml_keyswitch_shard_mid.argtypes = [vp, u32, u32, u32, vp, vp, vp, vp, vp]
    L.hml_keyswitch_shard_end.argtypes = [vp, u32, u32, u32, vp, vp, vp, vp]
    L.hml_keyswitch_shard_mid_p2p.argtypes = [vp, u32, u32, u32, vp, C.POINTER(vp), vp, vp, vp]
    L.hml_keyswitch_shard_end_p2p.argtypes = [vp, u32, u32, u32, C.POINTER(vp), vp, vp, vp]
    L.hml_shard_signal.argtypes = [vp, vp, u32, u64, u32, vp]
    L.hml_shard_wait.argtypes = [vp, vp, u32, u64, u32, vp]
    L.hml_shard_sync.argtypes = [vp, vp, u32, vp, u32, u64, u32, vp]
    L.hml_rescale_shard_begin.argtypes = [vp, u32, u32, u32, vp, vp, vp]
    L.hml_rescale_shard_end.argtypes = [vp, u32, u32, u32, vp, vp, vp, vp]
    L.hml_ipc_export.argtypes = [vp, vp, C.c_char_p]
    L.hml_ipc_import.argtypes = [vp, C.c_char_p, C.POINTER(vp)]
    L.hml_ipc_close.argtypes = [vp, vp]
    L.hml_shard_status.argtypes = [vp, vp, u32, vp]
    L.hml_shard_create.argtypes = [vp, u32, u32, u32, C.POINTER(vp)]
    L.hml_shard_create_ex.argtypes = [vp, u32, u32, u32, u32, C.POINTER(vp)]
    L.hml_shard_destroy.argtypes = [vp]
    L.hml_shard_handles.argtypes = [vp, C.c_char_p]
    L.hml_shard_connect_ipc.argtypes = [vp, C.c_char_p]
    L.hml_shard_connect_local.argtypes = [C.POINTER(vp), u32]
    L.hml_shard_prepare.argtypes = [vp, u32]
    L.hml_shard_check.argtypes = [vp, vp]
    L.hml_shard_own_limbs.argtypes = [vp, u32, C.POINTER(u32), C.POINTER(u32)]
    L.hml_keyswitch_sharded.argtypes = [vp, u32, vp, vp, vp, vp, vp]
    L.hml_hrotate_sharded.argtypes = [vp, u32, vp, vp, u64, vp, vp]
    L.hml_hmult_sharded.argtypes = [vp, u32, vp, vp, vp, vp, vp]
    L.hml_rescale_sharded.argtypes = [vp, u32, vp, vp, vp]
    L.hml_ew_sharded.argtypes = [vp, u32, i32, vp, vp, vp, vp]
    L.hml_group_op.argtypes = [C.POINTER(vp), u32, i32, u32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), u64,
                               C.POINTER(vp)]
    L.hml_hrotate_hoisted.argtypes = [vp, u32, vp, u32, C.POINTER(vp), u32, C.POINTER(u64), C.POINTER(vp), vp]
    L.hml_hrotate_sum_hoisted.argtypes = [vp, u32, vp, u32, C.POINTER(vp), u32, C.POINTER(u64), C.POINTER(vp), u32, vp, vp]
    L.hml_hrotate_bsgs_hoisted.argtypes = [vp, u32, vp, u32, C.POINTER(u64), C.POINTER(vp), u32, C.POINTER(u64), C.POINTER(vp), u32,
                                           C.POINTER(vp), u32, vp, vp]
    L.hml_hrotate_hoisted_sharded.argtypes = [vp, u32, vp, u32, C.POINTER(vp), C.POINTER(u64), C.POINTER(vp), vp]
    L.hml_group_hrotate_hoisted.argtypes = [C.POINTER(vp), u32, u32, C.POINTER(vp), u32, C.POINTER(vp), C.POINTER(u64), C.POINTER(vp),
                                            C.POINTER(vp)]
    L.hml_hrotate_sum_hoisted_sharded.argtypes = [vp, u32, vp, u32, C.POINTER(vp), C.POINTER(u64), C.POINTER(vp), vp, vp]
    L.hml_group_hrotate_sum_hoisted.argtypes = [C.POINTER(vp), u32, u32, C.POINTER(vp), u32, C.POINTER(vp), C.POINTER(u64), C.POINTER(vp),
                                                C.POINTER(vp), C.POINTER(vp)]
    L.hml_hmult_sum_sharded.argtypes = [vp, u32, u32, C.POINTER(vp), C.POINTER(vp), vp, vp, vp]
    L.hml_group_hmult_sum.argtypes = [C.POINTER(vp), u32, u32, u32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    L.hml_replay_create.argtypes = [vp, vp, u32, C.POINTER(_TraceOp), u32, u32, C.POINTER(vp)]
    L.hml_replay_bind.argtypes = [vp, vp, C.POINTER(vp), u32, C.POINTER(u32), C.POINTER(vp), u32, vp, u32]
    L.hml_replay_run.argtypes = [vp, vp]
    L.hml_replay_slot.argtypes = [vp, u32, C.POINTER(vp), C.POINTER(u32)]
    L.hml_replay_slot_level.argtypes = [vp, u32, C.POINTER(u32)]
    L.hml_replay_destroy.argtypes = [vp]
    L.hml_dev_alloc.argtypes = [vp, u64, C.POINTER(vp)]
    L.hml_dev_free.argtypes = [vp, vp]
    L.hml_h2d.argtypes = [vp, vp, vp, u64, vp]
    L.hml_d2h.argtypes = [vp, vp, vp, u64, vp]
    L.hml_key_pack.argtypes = [vp, vp, u64, vp, vp]
    L.hml_profile_begin.argtypes = [vp, vp]
    L.hml_profile_end.argtypes = [vp, C.POINTER(_Profile)]
    L.hml_sync.argtypes = [vp, vp]
    _LIB = L
    return L


def _counts_to_dict(c):
    return {
        "NTT": c.ntt, "INTT": c.intt, "MULT": c.mult, "BCONV_STEP2": c.bconv_step2, "AUTO": c.automorph,
        "total": c.total, "driverTotal": c.driver_total,
        "stages": [{"label": c.stages[i].label.decode(), "opcode": c.stages[i].opcode.decode(),
                    "limb_ops": c.stages[i].limb_ops, "instructions": c.stages[i].instructions} for i in range(c.n_stages)],
    }


def trace_counts(op, N, batch_size, max_level, L, alpha, bconv_high=2, bconv_width=6):
    """Reference-shaped instruction counts of one op (pure host code in the library; no GPU needed)."""
    lib = load_library()
    c = _Counts()
    rc = lib.hml_trace_counts(op.encode(), N, batch_size, max_level, L, alpha, bconv_high, bconv_width, C.byref(c))
    if rc:
        raise HmlError(rc, lib.hml_last_create_error().decode())
    return _counts_to_dict(c)


def shard_layout(L, alpha, rank, world):
    """Ownership / gather-slot layout of the limb-sharded key switch (pure host code in the library)."""
    lib = load_library()
    s = _ShardInfo()
    rc = lib.hml_shard_layout(L, alpha, rank, world, C.byref(s))
    if rc:
        raise HmlError(rc, "bad shard layout arguments")
    E = L + alpha
    return {"gather1_slots": s.gather1_slots, "gather2_slots": s.gather2_slots,
            "own_q": [s.own_q[i] for i in range(s.n_own_q)], "own_p": [s.own_p[i] for i in range(s.n_own_p)],
            "owner": [s.owner[e] for e in range(E)], "slot": [s.slot[e] for e in range(E)]}


def algorithmic_words(op, L, alpha):
    """Algorithmic traffic of one op in limb-sized words W = 8N bytes (SURVEY.md 8d, unfused schedule)."""
    E, beta = L + alpha, math.ceil(L / alpha)
    ks = 2 * L + 2 * L + beta * E + 2 * beta * E + (3 * beta + 2) * E + 4 * alpha + 4 * alpha + 2 * (alpha + L) + 4 * L + 6 * L
    if op == "keyswitch":
        return ks
    if op == "hmult":
        return ks + 7 * L + 6 * L + 2 * (4 + 5 * (L - 1))
    if op == "hrotate":
        return ks + 4 * L + 3 * L
    if op in ("hadd", "pmult", "padd"):
        return 6 * L
    if op in ("ntt", "intt", "auto"):
        return 2
    raise ValueError(op)


def _ptr(t):
    if t is None or t.numel() == 0:
        return None
    if not t.is_cuda or not t.is_contiguous() or t.element_size() != 8:
        raise ValueError("expected a contiguous 64-bit CUDA tensor")
    return t.data_ptr()


def _u32arr(v):
    return (C.c_uint32 * len(v))(*[int(x) for x in v])


class Context:
    """One hml_ctx: replaces `new Config(path)` + `new Arch(config)` (reference bench_micro24.cpp:16-27)."""

    def __init__(self, cfg_path=None, max_level=None, alpha=None, device=0, N=None, element_bit_width=36, batch_size=256):
        import torch
        self.lib = load_library()
        self.h = C.c_void_p()
        if not torch.cuda.is_available():
            raise HmlError(3, "no CUDA device: homulator_b200 has no CPU fallback")
        if cfg_path is not None:
            rc = self.lib.hml_ctx_create(str(cfg_path).encode(), max_level, alpha, device, C.byref(self.h))
        else:
            rc = self.lib.hml_ctx_create_params(N, element_bit_width, min(batch_size, N), max_level, alpha, device, C.byref(self.h))
        if rc:
            raise HmlError(rc, self.lib.hml_last_create_error().decode())
        self.device = torch.device("cuda", device)
        self.N = self.lib.hml_ring_degree(self.h)
        self.max_level, self.alpha = max_level, alpha
        n = self.lib.hml_n_moduli(self.h)
        buf = (C.c_uint64 * n)()
        self._chk(self.lib.hml_get_moduli(self.h, buf, n))
        self.moduli = [int(x) for x in buf]
        self._chk(self.lib.hml_get_roots(self.h, buf, n))
        self.psi = [int(x) for x in buf]

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.lib.hml_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc:
            raise HmlError(rc, self.lib.hml_last_error(self.h).decode())

    def _stream(self):
        import torch
        return torch.cuda.current_stream(self.device).cuda_stream

    def ext_mod_idx(self, L):
        return list(range(L)) + [self.max_level + j for j in range(self.alpha)]

    def beta(self, L):
        return -(-L // self.alpha)

    def empty(self, *shape):
        import torch
        return torch.empty(*shape, dtype=torch.int64, device=self.device)

    # ---- primitives (one per reference instruction class)
    def ntt(self, x, mod_idx, out=None, inverse=False):
        out = self.empty(*x.shape) if out is None else out
        n = len(mod_idx)
        assert x.numel() == n * self.N
        f = self.lib.hml_intt if inverse else self.lib.hml_ntt
        self._chk(f(self.h, _ptr(x), _ptr(out), _u32arr(mod_idx), n, self._stream()))
        return out

    def intt(self, x, mod_idx, out=None):
        return self.ntt(x, mod_idx, out, inverse=True)

    def ntt_batch(self, x, mod_idx, out=None, inverse=False):
        """x [n_batch][len(mod_idx)][N]: one launch pair for the whole batch (hml_ntt_batch / hml_intt_batch)"""
        out = self.empty(*x.shape) if out is None else out
        n = len(mod_idx)
        nb = x.numel() // (n * self.N)
        assert x.numel() == nb * n * self.N
        f = self.lib.hml_intt_batch if inverse else self.lib.hml_ntt_batch
        self._chk(f(self.h, _ptr(x), _ptr(out), _u32arr(mod_idx), n, nb, self._stream()))
        return out

    def ewe(self, x1, x2, x3, x4, mod_idx, subtract=False, out=None):
        ref = x1 if x1 is not None else x3
        out = self.empty(*ref.shape) if out is None else out
        self._chk(self.lib.hml_ewe(self.h, _ptr(x1), _ptr(x2), _ptr(x3), _ptr(x4), int(subtract), _ptr(out),
                                   _u32arr(mod_idx), len(mod_idx), self._stream()))
        return out

    def automorph(self, x, galois_elt, out=None):
        out = self.empty(*x.shape) if out is None else out
        self._chk(self.lib.hml_automorph(self.h, _ptr(x), _ptr(out), galois_elt, x.numel() // self.N, self._stream()))
        return out

    def bconv(self, x, src_idx, dst_idx, out=None):
        out = self.empty(len(dst_idx), self.N) if out is None else out
        self._chk(self.lib.hml_bconv(self.h, _ptr(x), _u32arr(src_idx), len(src_idx), _ptr(out), _u32arr(dst_idx),
                                     len(dst_idx), self._stream()))
        return out

    def bconv_batch(self, x, src_idx, dst_idx, out=None):
        """x [n_batch][n_src][N] -> [n_batch][n_dst][N] in one launch."""
        nb = x.shape[0]
        out = self.empty(nb, len(dst_idx), self.N) if out is None else out
        self._chk(self.lib.hml_bconv_batch(self.h, _ptr(x), _u32arr(src_idx), len(src_idx), _ptr(out), _u32arr(dst_idx),
                                           len(dst_idx), nb, self._stream()))
        return out

    # ---- sub-operations and operations
    def keyswitch(self, L, d, evk, evk_q_limbs=None):
        o0, o1 = self.empty(L, self.N), self.empty(L, self.N)
        self._chk(self.lib.hml_keyswitch(self.h, L, _ptr(d), _ptr(evk), evk_q_limbs or L, _ptr(o0), _ptr(o1), self._stream()))
        return o0, o1

    def rescale(self, L, x):
        out = self.empty(L - 1, self.N)
        self._chk(self.lib.hml_rescale(self.h, L, _ptr(x), _ptr(out), self._stream()))
        return out

    def hmult(self, L, ct_a, ct_b, evk, evk_q_limbs=None, out=None):
        out = self.empty(2, L - 1, self.N) if out is None else out
        self._chk(self.lib.hml_hmult(self.h, L, _ptr(ct_a), _ptr(ct_b), _ptr(evk), evk_q_limbs or L, _ptr(out), self._stream()))
        return out

    def key_pack(self, key):
        """Packed copy of an evaluation / rotation key (hml_key_pack): same shape, every limb slot holds N 32-bit low words + N high
        bytes.  Pass it with evk_q_limbs = limbs | KEY_PACKED."""
        import torch
        out = torch.empty_like(key)
        self._chk(self.lib.hml_key_pack(self.h, _ptr(key), key.numel() // self.N, _ptr(out), self._stream()))
        return out

    def hrotate(self, L, ct, rotkey, galois_elt=5, evk_q_limbs=None, out=None):
        out = self.empty(2, L, self.N) if out is None else out
        self._chk(self.lib.hml_hrotate(self.h, L, _ptr(ct), _ptr(rotkey), evk_q_limbs or L, galois_elt, _ptr(out), self._stream()))
        return out

    def hrotate_hoisted(self, L, ct, rotkeys, galois_elts, evk_q_limbs=None, outs=None):
        """Rotations of ONE ciphertext sharing one ModUp (hml_hrotate_hoisted); returns the list of outputs."""
        n = len(galois_elts)
        outs = [self.empty(2, L, self.N) for _ in range(n)] if outs is None else outs
        keys = (C.c_void_p * n)(*[_ptr(k) for k in rotkeys])
        po = (C.c_void_p * n)(*[_ptr(o) for o in outs])
        gs = (C.c_uint64 * n)(*[int(g) for g in galois_elts])
        self._chk(self.lib.hml_hrotate_hoisted(self.h, L, _ptr(ct), n, keys, evk_q_limbs or L, gs, po, self._stream()))
        return outs

    def hrotate_sum_hoisted(self, L, ct, rotkeys, galois_elts, pts, evk_q_limbs=None, pt_q_limbs=None, out=None):
        """sum_i pts[i] * rotate(ct, galois_elts[i]) with one ModUp and one ModDown (hml_hrotate_sum_hoisted).  pts[i] is
        [pt_q_limbs + alpha][N]: Q-limbs first, P-limb j at row pt_q_limbs + j (pt_q_limbs defaults to L)."""
        n = len(galois_elts)
        if len(rotkeys) != n or len(pts) != n:
            raise ValueError("one key and one plaintext per galois element")
        out = self.empty(2, L, self.N) if out is None else out
        keys = (C.c_void_p * max(n, 1))(*[_ptr(k) for k in rotkeys])
        pa = (C.c_void_p * max(n, 1))(*[_ptr(p) for p in pts])
        gs = (C.c_uint64 * max(n, 1))(*[int(g) for g in galois_elts])
        self._chk(self.lib.hml_hrotate_sum_hoisted(self.h, L, _ptr(ct), n, keys, evk_q_limbs or L, gs, pa, pt_q_limbs or L, _ptr(out),
                                                   self._stream()))
        return out

    def hrotate_bsgs_hoisted(self, L, ct, baby_galois, baby_keys, giant_galois, giant_keys, pts, evk_q_limbs=None, pt_q_limbs=None,
                             out=None):
        """sum_j rotate(sum_i pts[j][i] * rotate(ct, baby_galois[i]), giant_galois[j]) with one ModUp for every baby step and one
        final ModDown (hml_hrotate_bsgs_hoisted).  pts is n2 lists of n1 plaintexts [pt_q_limbs + alpha][N] (P-limb m at row
        pt_q_limbs + m); a key may be None for an identity element (galois 1)."""
        n1, n2 = len(baby_galois), len(giant_galois)
        if len(baby_keys) != n1 or len(giant_keys) != n2 or len(pts) != n2 or any(len(row) != n1 for row in pts):
            raise ValueError("one key per galois element and n2 rows of n1 plaintexts")
        out = self.empty(2, L, self.N) if out is None else out
        bk = (C.c_void_p * max(n1, 1))(*[_ptr(k) for k in baby_keys])
        gk = (C.c_void_p * max(n2, 1))(*[_ptr(k) for k in giant_keys])
        bg = (C.c_uint64 * max(n1, 1))(*[int(g) for g in baby_galois])
        gg = (C.c_uint64 * max(n2, 1))(*[int(g) for g in giant_galois])
        pa = (C.c_void_p * max(n1 * n2, 1))(*[_ptr(p) for row in pts for p in row])
        self._chk(self.lib.hml_hrotate_bsgs_hoisted(self.h, L, _ptr(ct), n1, bg, bk, n2, gg, gk, evk_q_limbs or L, pa, pt_q_limbs or L,
                                                    _ptr(out), self._stream()))
        return out

    def hadd(self, L, a, b, out=None):
        out = self.empty(2, L, self.N) if out is None else out
        self._chk(self.lib.hml_hadd(self.h, L, _ptr(a), _ptr(b), _ptr(out), self._stream()))
        return out

    def pmult(self, L, ct, pt, out=None):
        out = self.empty(2, L, self.N) if out is None else out
        self._chk(self.lib.hml_pmult(self.h, L, _ptr(ct), _ptr(pt), _ptr(out), self._stream()))
        return out

    def padd(self, L, ct, pt, out=None):
        out = self.empty(2, L, self.N) if out is None else out
        self._chk(self.lib.hml_padd(self.h, L, _ptr(ct), _ptr(pt), _ptr(out), self._stream()))
        return out

    def pmult_add(self, L, ct, pt, ct_add, out=None):
        out = self.empty(2, L, self.N) if out is None else out
        self._chk(self.lib.hml_pmult_add(self.h, L, _ptr(ct), _ptr(pt), _ptr(ct_add), _ptr(out), self._stream()))
        return out

    def hmult_batch(self, L, ct_a, ct_b, evk, evk_q_limbs=None, out=None):
        n = ct_a.shape[0]
        out = self.empty(n, 2, L - 1, self.N) if out is None else out
        self._chk(self.lib.hml_hmult_batch(self.h, L, n, _ptr(ct_a), _ptr(ct_b), _ptr(evk), evk_q_limbs or L, _ptr(out), self._stream()))
        return out

    def hmult_sum(self, L, cts_a, cts_b, evk, evk_q_limbs=None, out=None):
        """sum_i cts_a[i] * cts_b[i] with one key switch and one rescale per output (hml_hmult_sum).  cts_a / cts_b are equally long
        lists of [2][L][N] tensors (one output, [2][L-1][N]) or of [n_out][2][L][N] tensors (n_out outputs, [n_out][2][L-1][N]);
        passing the same tensor as cts_a[i] and cts_b[i] squares it and reads it once."""
        n = len(cts_a)
        if len(cts_b) != n or n == 0:
            raise ValueError("cts_a and cts_b must be equally long and not empty")
        shape = tuple(cts_a[0].shape)
        if len(shape) not in (3, 4) or any(tuple(t.shape) != shape for t in list(cts_a) + list(cts_b)):
            raise ValueError("every term must have the shape [2][L][N] or the same [n_out][2][L][N]")
        n_out = shape[0] if len(shape) == 4 else 1
        if out is None:
            out = self.empty(*shape[:-3], 2, L - 1, self.N)
        pa = (C.c_void_p * n)(*[_ptr(t) for t in cts_a])
        pb = (C.c_void_p * n)(*[_ptr(t) for t in cts_b])
        self._chk(self.lib.hml_hmult_sum(self.h, L, n, pa, pb, n_out, _ptr(evk), evk_q_limbs or L, _ptr(out), self._stream()))
        return out

    def hrotate_batch(self, L, ct, rotkey, galois_elt=5, evk_q_limbs=None, out=None):
        n = ct.shape[0]
        out = self.empty(n, 2, L, self.N) if out is None else out
        self._chk(self.lib.hml_hrotate_batch(self.h, L, n, _ptr(ct), _ptr(rotkey), evk_q_limbs or L, galois_elt, _ptr(out), self._stream()))
        return out

    def hmult_host(self, L, ct_a_host, ct_b_host, evk_dev, out_host, evk_q_limbs=None):
        """ct_*_host / out_host: CPU tensors (pinned for full speed) [n][2][L][N] / [n][2][L-1][N]."""
        n = ct_a_host.shape[0]
        self._chk(self.lib.hml_hmult_host(self.h, L, n, ct_a_host.data_ptr(), ct_b_host.data_ptr(), _ptr(evk_dev),
                                          evk_q_limbs or L, out_host.data_ptr()))
        return out_host

    def hrotate_host(self, L, ct_host, rotkey_dev, out_host, galois_elt=5, evk_q_limbs=None):
        n = ct_host.shape[0]
        self._chk(self.lib.hml_hrotate_host(self.h, L, n, ct_host.data_ptr(), _ptr(rotkey_dev), evk_q_limbs or L, galois_elt,
                                            out_host.data_ptr()))
        return out_host

    def pack_host(self, words_host):
        """CPU tensor of uint64 words [.., N] -> uint8 CPU tensor of packed limbs (5N bytes per limb), pinned."""
        import torch
        n_limbs = words_host.numel() // self.N
        out = torch.empty(self.lib.hml_packed_bytes(self.h, n_limbs), dtype=torch.uint8).pin_memory()
        self._chk(self.lib.hml_pack_host(self.h, words_host.data_ptr(), n_limbs, out.data_ptr()))
        return out

    def unpack_host(self, packed_host, shape):
        import torch
        out = torch.empty(*shape, dtype=torch.int64)
        self._chk(self.lib.hml_unpack_host(self.h, packed_host.data_ptr(), out.numel() // self.N, out.data_ptr()))
        return out

    def hmult_host_packed(self, L, n, a_packed, b_packed, evk_dev, out_packed, evk_q_limbs=None):
        self._chk(self.lib.hml_hmult_host_packed(self.h, L, n, a_packed.data_ptr(), b_packed.data_ptr(), _ptr(evk_dev), evk_q_limbs or L,
                                                 out_packed.data_ptr()))
        return out_packed

    def hrotate_host_packed(self, L, n, ct_packed, rotkey_dev, out_packed, galois_elt=5, evk_q_limbs=None):
        self._chk(self.lib.hml_hrotate_host_packed(self.h, L, n, ct_packed.data_ptr(), _ptr(rotkey_dev), evk_q_limbs or L, galois_elt,
                                                   out_packed.data_ptr()))
        return out_packed

    def keyswitch_sharded(self, L, d_own, evk_own, rank, world, all_gather):
        """Limb-sharded key switch (SURVEY.md 8e mode 2).  `all_gather(buf)` must all-gather, in place along dim 0,
        a tensor whose slice [rank] this rank has filled (torch.distributed.all_gather_into_tensor(buf, buf[rank]))."""
        lay = shard_layout(L, self.alpha, rank, world)
        nq = len(lay["own_q"])
        g1 = self.empty(world, lay["gather1_slots"], self.N)
        g2 = self.empty(world, 2, lay["gather2_slots"], self.N)
        o0, o1 = self.empty(max(nq, 1), self.N), self.empty(max(nq, 1), self.N)
        st = self._stream()
        self._chk(self.lib.hml_keyswitch_shard_begin(self.h, L, rank, world, _ptr(d_own), _ptr(g1), st))
        all_gather(g1)
        self._chk(self.lib.hml_keyswitch_shard_mid(self.h, L, rank, world, _ptr(d_own), _ptr(g1), _ptr(evk_own), _ptr(g2), st))
        all_gather(g2)
        self._chk(self.lib.hml_keyswitch_shard_end(self.h, L, rank, world, _ptr(g2), _ptr(o0), _ptr(o1), st))
        return o0[:nq], o1[:nq]

    # ---- peer-direct limb-sharded key switch (no collective; NVLink loads inside the base conversion)
    def dev_alloc(self, n_words, zero=True):
        """Plain cudaMalloc through the ABI (shareable with cudaIpc, unlike a slice of torch's caching allocator)."""
        p = C.c_void_p()
        self._chk(self.lib.hml_dev_alloc(self.h, n_words, C.byref(p)))
        if zero:
            import numpy as np
            z = np.zeros(n_words, dtype=np.uint64)
            self._chk(self.lib.hml_h2d(self.h, p.value, z.ctypes.data, n_words, None))
            self._chk(self.lib.hml_sync(self.h, None))
        return p.value

    def ipc_export(self, ptr):
        buf = C.create_string_buffer(64)
        self._chk(self.lib.hml_ipc_export(self.h, ptr, buf))
        return bytes(buf.raw)

    def ipc_import(self, handle):
        p = C.c_void_p()
        self._chk(self.lib.hml_ipc_import(self.h, handle, C.byref(p)))
        return p.value

    def counts(self, op, L):
        c = _Counts()
        rc = self.lib.hml_get_counts(self.h, op.encode(), L, C.byref(c))
        if rc:
            raise HmlError(rc, self.lib.hml_last_create_error().decode())
        return _counts_to_dict(c)

    def buffer_plan(self, op, L):
        """the op's device workspace as `Malloc <name> from A to B` lines (reference include/Addr.h:29-48)"""
        buf = C.create_string_buffer(8192)
        self._chk(self.lib.hml_buffer_plan(self.h, op.encode(), L, buf, len(buf)))
        return buf.value.decode()

    def profile(self, fn):
        """Run fn() in measuring mode: device microseconds per kernel class (the reference's per-unit statistics)."""
        self._chk(self.lib.hml_profile_begin(self.h, self._stream()))
        try:
            fn()
        finally:
            pr = _Profile()
            self._chk(self.lib.hml_profile_end(self.h, C.byref(pr)))
        names = ("NTT", "INTT", "BCONV", "EWE", "AUTO")
        return {"us": {n: pr.us[i] for i, n in enumerate(names)}, "launches": {n: pr.launches[i] for i, n in enumerate(names)},
                "total_us": pr.total_us}

    def exec_counts(self, reset=False):
        e = _ExecCounts()
        self._chk(self.lib.hml_exec_counts_get(self.h, C.byref(e)))
        if reset:
            self._chk(self.lib.hml_exec_counts_reset(self.h))
        return {k: getattr(e, k) for k, _ in _ExecCounts._fields_}

    # ---- seeded synthetic operands (SURVEY.md 8d)
    def uniform(self, mod_idx, tensor_id, lead=()):
        """int64 CUDA tensor [*lead, len(mod_idx), N] of uniform residues, generated on the device."""
        import torch
        g = torch.Generator(device=self.device)
        g.manual_seed(0x486F6D75 + 7919 * tensor_id)
        n_lead = 1
        for d in lead:
            n_lead *= d
        out = self.empty(n_lead, len(mod_idx), self.N)
        for i, mi in enumerate(mod_idx):
            out[:, i].random_(0, self.moduli[mi], generator=g)
        return out.view(*lead, len(mod_idx), self.N)


class Shard:
    """One rank's view of a limb-shard group (hml_shard, homulator_b200/csrc/shard.cu): every sharded op is ONE C-ABI call.
    Build with Shard.ipc(ctx, max_L, rank, world, exchange) (one process per GPU) or Shard.local_group(ctxs, max_L)
    (one process driving all ranks; emulation on a single GPU when the ctxs share a device).  max_rot (1..16, the same on
    every rank) is the number of hoisted rotations that share one exchange (hrotate_hoisted)."""

    def __init__(self, ctx, max_L, rank, world, max_rot=1):
        self.ctx, self.max_L, self.rank, self.world, self.max_rot = ctx, max_L, rank, world, max_rot
        self.h = C.c_void_p()
        ctx._chk(ctx.lib.hml_shard_create_ex(ctx.h, max_L, rank, world, max_rot, C.byref(self.h)))

    @classmethod
    def ipc(cls, ctx, max_L, rank, world, exchange, max_rot=1):
        """`exchange(obj)` returns the list of every rank's obj (torch.distributed.all_gather_object)."""
        sh = cls(ctx, max_L, rank, world, max_rot)
        buf = C.create_string_buffer(256)
        ctx._chk(ctx.lib.hml_shard_handles(sh.h, buf))
        allh = exchange(bytes(buf.raw))
        if world > 1:
            ctx._chk(ctx.lib.hml_shard_connect_ipc(sh.h, b"".join(allh)))
        return sh

    @classmethod
    def local_group(cls, ctxs, max_L, max_rot=1):
        world = len(ctxs)
        group = [cls(c, max_L, r, world, max_rot) for r, c in enumerate(ctxs)]
        if world > 1:
            arr = (C.c_void_p * world)(*[g.h for g in group])
            ctxs[0]._chk(ctxs[0].lib.hml_shard_connect_local(arr, world))
        return group

    def close(self):
        if self.h:
            self.ctx.lib.hml_shard_destroy(self.h)
            self.h = C.c_void_p()

    def own(self, L):
        a, b = C.c_uint32(), C.c_uint32()
        self.ctx._chk(self.ctx.lib.hml_shard_own_limbs(self.h, L, C.byref(a), C.byref(b)))
        return a.value, b.value

    def own_q(self, L):
        return list(range(self.rank, L, self.world))

    def own_ext(self, L):
        return [e for e in range(L + self.ctx.alpha) if e % self.world == self.rank]

    def prepare(self, L):
        self.ctx._chk(self.ctx.lib.hml_shard_prepare(self.h, L))

    def check(self):
        self.ctx._chk(self.ctx.lib.hml_shard_check(self.h, self.ctx._stream()))

    def keyswitch(self, L, d_own, evk_own, o0=None, o1=None):
        c = self.ctx
        nq, _ = self.own(L)
        o0 = c.empty(max(nq, 1), c.N) if o0 is None else o0
        o1 = c.empty(max(nq, 1), c.N) if o1 is None else o1
        c._chk(c.lib.hml_keyswitch_sharded(self.h, L, _ptr(d_own), _ptr(evk_own), _ptr(o0), _ptr(o1), c._stream()))
        return o0[:nq], o1[:nq]

    def hrotate(self, L, ct_own, rk_own, g, out=None):
        c = self.ctx
        nq, _ = self.own(L)
        out = c.empty(2, max(nq, 1), c.N) if out is None else out
        c._chk(c.lib.hml_hrotate_sharded(self.h, L, _ptr(ct_own), _ptr(rk_own), g, _ptr(out), c._stream()))
        return out

    def hrotate_hoisted(self, L, ct_own, rk_owns, galois_elts, outs=None):
        """Rotations of ONE sharded ciphertext sharing one ModUp (hml_hrotate_hoisted_sharded); rk_owns[i] is this rank's key
        slice for galois_elts[i] (None on a rank that owns no extended limb).  Returns the list of outputs [2][nq][N]."""
        c = self.ctx
        nq, _ = self.own(L)
        n = len(galois_elts)
        if len(rk_owns) != n:
            raise ValueError("one key slice per galois element")
        outs = [c.empty(2, max(nq, 1), c.N) for _ in range(n)] if outs is None else outs
        keys = (C.c_void_p * max(n, 1))(*[(_ptr(k) if k is not None else None) for k in rk_owns])
        po = (C.c_void_p * max(n, 1))(*[_ptr(o) for o in outs])
        gs = (C.c_uint64 * max(n, 1))(*[int(g) for g in galois_elts])
        c._chk(c.lib.hml_hrotate_hoisted_sharded(self.h, L, _ptr(ct_own), n, keys, gs, po, c._stream()))
        return outs

    def hrotate_sum_hoisted(self, L, ct_own, rk_owns, galois_elts, pt_owns, out=None):
        """sum_i pt_owns[i] * rotate(ct, galois_elts[i]) on this rank's limbs with one ModUp, one ModDown and two exchanges
        (hml_hrotate_sum_hoisted_sharded).  rk_owns[i] / pt_owns[i] are this rank's key and plaintext slices (the plaintext's
        owned rows of the extended basis, own_ext(L) order: replay.shard_plaintexts); None on a rank that owns no extended limb.
        Returns the output [2][nq][N]."""
        c = self.ctx
        nq, _ = self.own(L)
        n = len(galois_elts)
        if len(rk_owns) != n or len(pt_owns) != n:
            raise ValueError("one key slice and one plaintext slice per galois element")
        out = c.empty(2, max(nq, 1), c.N) if out is None else out
        keys = (C.c_void_p * max(n, 1))(*[(_ptr(k) if k is not None else None) for k in rk_owns])
        pa = (C.c_void_p * max(n, 1))(*[(_ptr(p) if p is not None else None) for p in pt_owns])
        gs = (C.c_uint64 * max(n, 1))(*[int(g) for g in galois_elts])
        c._chk(c.lib.hml_hrotate_sum_hoisted_sharded(self.h, L, _ptr(ct_own), n, keys, gs, pa, _ptr(out), c._stream()))
        return out

    def hmult_sum(self, L, a_owns, b_owns, evk_own, out=None):
        """sum_i a_owns[i] * b_owns[i] on this rank's limbs with one key switch and one rescale (hml_hmult_sum_sharded); the
        same tensor as a_owns[i] and b_owns[i] squares it.  Returns the output [2][nk][N] (the owned limbs below L-1)."""
        c = self.ctx
        _, nk = self.own(L)
        n = len(a_owns)
        if len(b_owns) != n:
            raise ValueError("a_owns and b_owns must be equally long")
        out = c.empty(2, max(nk, 1), c.N) if out is None else out
        pa = (C.c_void_p * max(n, 1))(*[_ptr(t) for t in a_owns])
        pb = (C.c_void_p * max(n, 1))(*[_ptr(t) for t in b_owns])
        c._chk(c.lib.hml_hmult_sum_sharded(self.h, L, n, pa, pb, _ptr(evk_own), _ptr(out), c._stream()))
        return out

    def hmult(self, L, a_own, b_own, evk_own, out=None):
        c = self.ctx
        _, nk = self.own(L)
        out = c.empty(2, max(nk, 1), c.N) if out is None else out
        c._chk(c.lib.hml_hmult_sharded(self.h, L, _ptr(a_own), _ptr(b_own), _ptr(evk_own), _ptr(out), c._stream()))
        return out

    def rescale(self, L, x_own, out=None):
        c = self.ctx
        _, nk = self.own(L)
        out = c.empty(2, max(nk, 1), c.N) if out is None else out
        c._chk(c.lib.hml_rescale_sharded(self.h, L, _ptr(x_own), _ptr(out), c._stream()))
        return out

    def ew(self, L, kind, a_own, b_own, out=None):
        c = self.ctx
        out = c.empty(*a_own.shape) if out is None else out
        c._chk(c.lib.hml_ew_sharded(self.h, L, {"hadd": 0, "pmult": 1, "padd": 2}[kind], _ptr(a_own), _ptr(b_own), _ptr(out), c._stream()))
        return out


def group_op(group, kind, L, a, b=None, key=None, out0=None, out1=None, galois_elt=0, streams=None):
    """hml_group_op: all ranks of a local group, one host thread.  kind in keyswitch / hrotate / hmult / rescale; every
    operand is a list indexed by rank (None entries allowed for ranks that own nothing)."""
    import torch
    world = len(group)
    ctx = group[0].ctx

    def arr(lst):
        if lst is None:
            return None
        return (C.c_void_p * world)(*[(_ptr(t) if t is not None else None) for t in lst])

    if streams is None:
        st = torch.cuda.current_stream(ctx.device).cuda_stream
        streams = [st] * world
    gh = (C.c_void_p * world)(*[g.h for g in group])
    sa = (C.c_void_p * world)(*streams)
    rc = ctx.lib.hml_group_op(gh, world, {"keyswitch": 0, "hrotate": 1, "hmult": 2, "rescale": 3}[kind], L, arr(a), arr(b), arr(key),
                              arr(out0), arr(out1), galois_elt, sa)
    if rc:
        msgs = [g.ctx.lib.hml_last_error(g.ctx.h).decode() for g in group]
        raise HmlError(rc, next((m for m in msgs if m), "group op failed"))


def group_hrotate_hoisted(group, L, ct_own, keys, galois_elts, outs=None, streams=None):
    """hml_group_hrotate_hoisted: Shard.hrotate_hoisted on every rank of a local group from one host thread.  ct_own[r] is rank
    r's ciphertext slice, keys[r][i] its key slice for galois_elts[i] (None where the rank owns no extended limb); returns
    outs[r][i] (allocated when not given)."""
    import torch
    world, n = len(group), len(galois_elts)
    ctx = group[0].ctx
    if len(ct_own) != world or len(keys) != world or any(len(k) != n for k in keys):
        raise ValueError("ct_own needs one entry per rank, keys one list of len(galois_elts) key slices per rank")
    if outs is None:
        outs = [[g.ctx.empty(2, max(g.own(L)[0], 1), g.ctx.N) for _ in range(n)] for g in group]
    if streams is None:
        st = torch.cuda.current_stream(ctx.device).cuda_stream
        streams = [st] * world
    gh = (C.c_void_p * world)(*[g.h for g in group])
    ca = (C.c_void_p * world)(*[_ptr(t) for t in ct_own])
    ka = (C.c_void_p * max(world * n, 1))(*[(_ptr(k) if k is not None else None) for r in range(world) for k in keys[r]])
    oa = (C.c_void_p * max(world * n, 1))(*[_ptr(o) for r in range(world) for o in outs[r]])
    gs = (C.c_uint64 * max(n, 1))(*[int(g) for g in galois_elts])
    sa = (C.c_void_p * world)(*streams)
    rc = ctx.lib.hml_group_hrotate_hoisted(gh, world, L, ca, n, ka, gs, oa, sa)
    if rc:
        msgs = [g.ctx.lib.hml_last_error(g.ctx.h).decode() for g in group]
        raise HmlError(rc, next((m for m in msgs if m), "group hoisted rotation failed"))
    return outs


def _group_call(group, streams, fn, what):
    """fn(group handle array, stream array) -> return code of a hml_group_* call; raises with the first rank's message"""
    import torch
    world = len(group)
    if streams is None:
        streams = [torch.cuda.current_stream(group[0].ctx.device).cuda_stream] * world
    rc = fn((C.c_void_p * world)(*[g.h for g in group]), (C.c_void_p * world)(*streams))
    if rc:
        msgs = [g.ctx.lib.hml_last_error(g.ctx.h).decode() for g in group]
        raise HmlError(rc, next((m for m in msgs if m), what + " failed"))


def group_hrotate_sum_hoisted(group, L, ct_own, keys, galois_elts, pts, outs=None, streams=None):
    """hml_group_hrotate_sum_hoisted: Shard.hrotate_sum_hoisted on every rank of a local group from one host thread.  ct_own[r]
    is rank r's ciphertext slice, keys[r][i] / pts[r][i] its key and plaintext slices for galois_elts[i] (None where the rank owns
    no extended limb); returns outs[r] (allocated when not given)."""
    world, n = len(group), len(galois_elts)
    if len(ct_own) != world or len(keys) != world or len(pts) != world or any(len(k) != n for k in keys) or any(len(p) != n for p in pts):
        raise ValueError("ct_own needs one entry per rank, keys and pts one list of len(galois_elts) slices per rank")
    if outs is None:
        outs = [g.ctx.empty(2, max(g.own(L)[0], 1), g.ctx.N) for g in group]
    opt = lambda t: _ptr(t) if t is not None else None  # noqa: E731
    ca = (C.c_void_p * world)(*[opt(t) for t in ct_own])
    ka = (C.c_void_p * max(world * n, 1))(*[opt(k) for r in range(world) for k in keys[r]])
    pa = (C.c_void_p * max(world * n, 1))(*[opt(p) for r in range(world) for p in pts[r]])
    oa = (C.c_void_p * world)(*[opt(o) for o in outs])
    gs = (C.c_uint64 * max(n, 1))(*[int(g) for g in galois_elts])
    lib = group[0].ctx.lib
    _group_call(group, streams, lambda gh, sa: lib.hml_group_hrotate_sum_hoisted(gh, world, L, ca, n, ka, gs, pa, oa, sa), "group rotation sum")
    return outs


def group_hmult_sum(group, L, a_own, b_own, evk_own, outs=None, streams=None):
    """hml_group_hmult_sum: Shard.hmult_sum on every rank of a local group from one host thread.  a_own[r][i] / b_own[r][i] are
    rank r's slices of term i, evk_own[r] its key slice (None where the rank owns no extended limb); returns outs[r]
    [2][nk][N] (allocated when not given)."""
    world = len(group)
    n = len(a_own[0]) if a_own else 0
    if len(a_own) != world or len(b_own) != world or len(evk_own) != world or any(len(x) != n for x in list(a_own) + list(b_own)):
        raise ValueError("a_own / b_own need one list of n_terms slices per rank, evk_own one key slice per rank")
    if outs is None:
        outs = [g.ctx.empty(2, max(g.own(L)[1], 1), g.ctx.N) for g in group]
    opt = lambda t: _ptr(t) if t is not None else None  # noqa: E731
    pa = (C.c_void_p * max(world * n, 1))(*[opt(t) for r in range(world) for t in a_own[r]])
    pb = (C.c_void_p * max(world * n, 1))(*[opt(t) for r in range(world) for t in b_own[r]])
    ea = (C.c_void_p * world)(*[opt(k) for k in evk_own])
    oa = (C.c_void_p * world)(*[opt(o) for o in outs])
    lib = group[0].ctx.lib
    _group_call(group, streams, lambda gh, sa: lib.hml_group_hmult_sum(gh, world, L, n, pa, pb, ea, oa, sa), "group product sum")
    return outs


class Replay:
    """hml_replay: a trace of (kind, dst, a, b) tuples over named ciphertexts, run through the C ABI (optionally as one CUDA
    graph, optionally with hoisted rotations, optionally limb-sharded).  `trace` uses the tuple format of
    homulator_b200.replay; names are mapped to slots here ("x" = slot 0 = the input).  hoist_sum=True turns a hoistable run of
    rotations whose outputs are summed with plaintext weights into one double-hoisted sum (HML_REPLAY_HOIST_SUM); the
    plaintexts are then bound as [L + alpha][N] (P-limbs at rows L..).  hmult_sum=True turns a chain of products summed as they
    are formed into one lazily relinearised sum (HML_REPLAY_HMULT_SUM, hml_hmult_sum)."""
    KINDS = {"hrotate": 0, "pmult": 1, "hadd": 2, "padd": 3, "hmult": 4}

    def __init__(self, ctx, L, trace, shard=None, graph=False, hoist=False, hoist_sum=False, hmult_sum=False):
        self.ctx, self.L, self.shard = ctx, L, shard
        self.names = {"x": 0}
        ops = []
        for op in trace:
            kind, dst, a, b = op
            if a not in self.names:
                raise ValueError("trace reads %r before it is written" % (a,))
            if kind in ("hadd", "hmult"):
                if b not in self.names:
                    raise ValueError("trace reads %r before it is written" % (b,))
                bb = self.names[b]
            else:
                bb = int(b)
            if dst not in self.names:
                self.names[dst] = len(self.names)
            ops.append((self.KINDS[kind], self.names[dst], self.names[a], bb))
        arr = (_TraceOp * len(ops))(*[_TraceOp(*o) for o in ops])
        self.h = C.c_void_p()
        flags = (1 if graph else 0) | (2 if hoist else 0) | (4 if hoist_sum else 0) | (8 if hmult_sum else 0)
        ctx._chk(ctx.lib.hml_replay_create(ctx.h, shard.h if shard is not None else None, L, arr, len(ops), flags, C.byref(self.h)))
        self._keep = None

    def bind(self, x, plaintexts, rot_keys, evk, evk_q_limbs=None):
        """plaintexts: dict / list idx -> tensor; rot_keys: dict rotation amount -> key tensor."""
        c = self.ctx
        n_pt = (max(plaintexts.keys()) + 1) if isinstance(plaintexts, dict) and plaintexts else len(plaintexts or [])
        get = (lambda i: plaintexts.get(i)) if isinstance(plaintexts, dict) else (lambda i: plaintexts[i])
        pts = (C.c_void_p * max(n_pt, 1))(*[(_ptr(get(i)) if get(i) is not None else None) for i in range(n_pt)])
        rots = sorted(rot_keys.keys())
        ra = (C.c_uint32 * max(len(rots), 1))(*rots)
        ka = (C.c_void_p * max(len(rots), 1))(*[_ptr(rot_keys[r]) for r in rots])
        self._keep = (x, plaintexts, rot_keys, evk)
        c._chk(c.lib.hml_replay_bind(self.h, _ptr(x), pts, n_pt, ra, ka, len(rots), _ptr(evk), evk_q_limbs or self.L))
        return self

    def run(self):
        self.ctx._chk(self.ctx.lib.hml_replay_run(self.h, self.ctx._stream()))
        return self

    def result(self, name):
        """Device tensor view [2][n_limbs][N] of a named ciphertext (owned by the replay object; valid until close())."""
        import torch
        p, n = C.c_void_p(), C.c_uint32()
        self.ctx._chk(self.ctx.lib.hml_replay_slot(self.h, self.names[name], C.byref(p), C.byref(n)))
        return _tensor_view(p.value, (2, n.value, self.ctx.N), self.ctx.device, self)

    def close(self):
        if self.h:
            self.ctx.lib.hml_replay_destroy(self.h)
            self.h = C.c_void_p()


class _DevArray:
    """__cuda_array_interface__ holder so torch can view library-owned device memory without copying."""

    def __init__(self, ptr, shape, owner):
        self.owner = owner
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<i8", "data": (ptr, False), "version": 3, "strides": None}


def _tensor_view(ptr, shape, device, owner):
    import torch
    if 0 in shape:
        return torch.empty(*shape, dtype=torch.int64, device=device)
    return torch.as_tensor(_DevArray(ptr, shape, owner), device=device)


class _Op:
    """Mirror of the reference's op objects: OP(label, maxLevel, currentLevel, alpha, cfg, arch)."""
    name = None

    def __init__(self, label, max_level, current_level, alpha, cfg, arch=None, device=0):
        self.label, self.L = label, current_level
        self.ctx = cfg if isinstance(cfg, Context) else Context(cfg, max_level, alpha, device)
        self.counts = self.ctx.counts(self.name, current_level)  # the reference builds its trace in the constructor

    def _operands(self):
        c, L = self.ctx, self.L
        q = list(range(L))
        ct_a = c.uniform(q, 1, lead=(2,))
        ct_b = c.uniform(q, 2, lead=(2,))
        key = c.uniform(c.ext_mod_idx(L), 3, lead=(c.beta(L), 2)) if self.name in ("hmult", "hrotate") else None
        return ct_a, ct_b, key

    def execute(self, *args, **kw):
        raise NotImplementedError

    def simulate(self, iters=10, warmup=3):
        """Run on seeded synthetic data; returns dict(us_median=..., counts=...)."""
        import torch
        ct_a, ct_b, key = self._operands()
        args = {"hmult": (ct_a, ct_b, key), "hrotate": (ct_a, key), "hadd": (ct_a, ct_b), "pmult": (ct_a, ct_b[0]),
                "padd": (ct_a, ct_b[0])}[self.name]
        for _ in range(warmup):
            self.execute(*args)
        torch.cuda.synchronize()
        times = []
        for _ in range(iters):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            self.execute(*args)
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1) * 1e3)
        times.sort()
        return {"op": self.name, "us_median": times[len(times) // 2], "us_min": times[0], "counts": self.counts}


class HMULT(_Op):
    name = "hmult"

    def execute(self, ct_a, ct_b, evk, evk_q_limbs=None):
        return self.ctx.hmult(self.L, ct_a, ct_b, evk, evk_q_limbs)


class HROTATE(_Op):
    name = "hrotate"

    def execute(self, ct, rotkey, galois_elt=5, evk_q_limbs=None):
        return self.ctx.hrotate(self.L, ct, rotkey, galois_elt, evk_q_limbs)


class HADD(_Op):
    name = "hadd"

    def execute(self, a, b):
        return self.ctx.hadd(self.L, a, b)


class PMULT(_Op):
    name = "pmult"

    def execute(self, ct, pt):
        return self.ctx.pmult(self.L, ct, pt)


class PADD(_Op):
    name = "padd"

    def execute(self, ct, pt):
        return self.ctx.padd(self.L, ct, pt)
