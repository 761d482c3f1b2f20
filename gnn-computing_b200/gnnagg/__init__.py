"""gnnagg -- Python host side of libgnnagg.so (the C ABI declared in include/gnnagg.h).

PyTorch is used only for device memory, streams and torch.distributed; every computation goes
through the C ABI with raw device pointers.  There is no CPU or PyTorch fallback: if the shared
library is missing, or a device entry point is called without a GPU, an exception is raised.

`gnnagg.plugin` mirrors the reference's PyTorch extension (Figure7/kernel.cpp:37-179).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
LIB_PATH = os.path.join(_ROOT, "lib", "libgnnagg.so")
CSRC = os.path.join(_ROOT, "csrc")

SCHED_LOCALITY, SCHED_NEIGHBOR_GROUPING, SCHED_LOCALITY_NEIGHBOR_GROUPING, SCHED_NOP = 0, 1, 2, 3


class GnnaggError(RuntimeError):
    pass


def build(verbose=False):
    """compile libgnnagg.so for sm_100a (nvcc cross-compiles without a GPU)"""
    cmd = ["make", "-C", CSRC, "-j8"] + ([] if verbose else ["-s"])
    subprocess.check_call(cmd)


_lib = None

_SIGS = {
    # name: (restype, argtypes)
    "gnnagg_version": (C.c_int, []),
    "gnnagg_last_error": (C.c_char_p, []),
    "gnnagg_device_info": (C.c_int, [C.POINTER(C.c_int)] * 3 + [C.c_char_p, C.c_int]),
    "gnnagg_schedule_build": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "gnnagg_schedule_num_target": (C.c_int64, [C.c_void_p]),
    "gnnagg_schedule_num_edges": (C.c_int64, [C.c_void_p]),
    "gnnagg_schedule_ptr": (C.c_void_p, [C.c_void_p]),
    "gnnagg_schedule_idx": (C.c_void_p, [C.c_void_p]),
    "gnnagg_schedule_target": (C.c_void_p, [C.c_void_p]),
    "gnnagg_schedule_val": (C.c_void_p, [C.c_void_p]),
    "gnnagg_schedule_free": (None, [C.c_void_p]),
    "gnnagg_reorder_csr": (C.c_int, [C.c_void_p] * 4 + [C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "gnnagg_graph_config": (C.c_int, [C.c_char_p, C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "gnnagg_graph_load": (C.c_int, [C.c_char_p, C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]),
    "gnnagg_graph_write": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "gnnagg_lsh_reorder": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_uint64, C.c_void_p]),
    "gnnagg_reorder_write": (C.c_int, [C.c_char_p, C.c_void_p, C.c_int]),
    "gnnagg_create": (C.c_int, [C.c_void_p] * 4 + [C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "gnnagg_create_on": (C.c_int, [C.c_void_p] * 4 + [C.c_int, C.c_int, C.POINTER(C.c_void_p), C.c_void_p]),
    "gnnagg_set_val_on": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "gnnagg_destroy": (C.c_int, [C.c_void_p]),
    "gnnagg_set_val": (C.c_int, [C.c_void_p, C.c_void_p]),
    "gnnagg_schedule_apply": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.c_int, C.c_int]),
    "gnnagg_num_target": (C.c_int, [C.c_void_p]),
    "gnnagg_schedule_kind": (C.c_int, [C.c_void_p]),
    "gnnagg_sched_to_csr_order": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gnnagg_sched_dev_ptr": (C.c_void_p, [C.c_void_p]),
    "gnnagg_sched_dev_idx": (C.c_void_p, [C.c_void_p]),
    "gnnagg_sched_dev_target": (C.c_void_p, [C.c_void_p]),
    "gnnagg_sched_dev_val": (C.c_void_p, [C.c_void_p]),
    "gnnagg_prepare": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "gnnagg_gcn_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_gcn_run_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_gcn_run_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_gcn_run_acc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_gcn_run_rows_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_gcn_run_acc_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_gcn_run_edgewise": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "gnnagg_csr2edgelist": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "gnnagg_gcn_layer": (C.c_int, [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_gcn_layer_bf16": (C.c_int, [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_dense_nn": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_gat_run": (C.c_int, [C.c_void_p] * 4 + [C.c_int, C.c_float, C.c_int, C.c_void_p]),
    "gnnagg_gat_edge_weights": (C.c_void_p, [C.c_void_p]),
    "gnnagg_edge_softmax": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p]),
    "gnnagg_u_add_v": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gnnagg_add_to_center": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gnnagg_each_div": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gnnagg_mlp_run": (C.c_int, [C.c_void_p] * 4 + [C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_sddmm": (C.c_int, [C.c_void_p] * 4 + [C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_transpose_build": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "gnnagg_transpose_dev": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)] + [C.POINTER(C.c_void_p)] * 3),
    "gnnagg_gcn_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "gnnagg_gcn_backward_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "gnnagg_gat_backward": (C.c_int, [C.c_void_p] * 9 + [C.c_int, C.c_float, C.c_void_p]),
    "gnnagg_sample_subgraph": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint64] + [C.POINTER(C.c_void_p)] * 3 +
                               [C.POINTER(C.c_int)] * 2 + [C.c_void_p]),
    "gnnagg_device_free": (C.c_int, [C.c_void_p]),
    "gnnagg_gather_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "gnnagg_spmm_naive": (C.c_int, [C.c_int] + [C.c_void_p] * 5 + [C.c_int, C.c_void_p]),
    "gnnagg_validate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int), C.c_void_p]),
    "gnnagg_validate_reordered": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                            C.POINTER(C.c_int), C.c_void_p]),
    "gnnagg_gcn_run_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_gcn_layer_host": (C.c_int, [C.c_void_p] * 4 + [C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_gat_run_host": (C.c_int, [C.c_void_p] * 4 + [C.c_int, C.c_float, C.c_int, C.c_void_p]),
    "gnnagg_launch_count": (C.c_int64, [C.c_void_p]),
    "gnnagg_set_warp_edges": (C.c_int, [C.c_void_p, C.c_int]),
    "gnnagg_set_host_pipeline": (C.c_int, [C.c_void_p, C.c_int]),
    "gnnagg_set_locality_slices": (C.c_int, [C.c_void_p, C.c_int]),
    "gnnagg_set_merge_duplicates": (C.c_int, [C.c_void_p, C.c_int]),
    "gnnagg_merged_edges": (C.c_int, [C.c_void_p]),
    "gnnagg_merged_dev": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "gnnagg_profile_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "gnnagg_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "gnnagg_memcpy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64]),
    # multi-GPU over NVLink peer memory (dist.cu)
    "gnnagg_dist_create": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int64), C.c_int, C.POINTER(C.c_void_p)]),
    "gnnagg_dist_create_rank": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_int64), C.c_int, C.POINTER(C.c_void_p)]),
    "gnnagg_dist_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "gnnagg_dist_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "gnnagg_dist_destroy": (C.c_int, [C.c_void_p]),
    "gnnagg_dist_set_graph": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "gnnagg_dist_prepare": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "gnnagg_dist_x": (C.c_void_p, [C.c_void_p, C.c_int]),
    "gnnagg_dist_gcn_run": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_dist_gcn_layer": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_dist_gcn_layer_host": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_dist_gcn_run_bf16": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_dist_gcn_layer_bf16": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "gnnagg_dist_gcn_layer_host_bf16": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                                  C.c_void_p]),
    "gnnagg_dist_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int),
                                   C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "gnnagg_dist_connect_local": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "gnnagg_dist_disconnect": (C.c_int, [C.c_void_p]),
    "gnnagg_dist_profile_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "gnnagg_dist_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "gnnagg_dist_check": (C.c_int, [C.c_void_p]),
    "gnnagg_dist_launch_count": (C.c_int64, [C.c_void_p]),
}

DIST_BLOB_BYTES = 256
DIST_MAX_WORLD = 16
DIST_NO_EXCHANGE = 1


def lib():
    """the loaded libgnnagg.so; raises when it has not been built (no fallback)"""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GnnaggError("libgnnagg.so not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "or `make -C gnn-computing_b200/csrc`")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def exported_symbols():
    return sorted(_SIGS)


def check(rc):
    if rc != 0:
        raise GnnaggError("gnnagg rc=%d: %s" % (rc, lib().gnnagg_last_error().decode(errors="replace")))


def _np(a):
    return None if a is None else a.ctypes.data


# ------------------------------------------------------------------ host preprocessing (numpy)
def schedule_build(kind, ptr, idx, val=None, par_num=0, neighbor_num=0, total_num_v=None):
    """host schedule -> (ptr_vec, idx_vec, target_vec, val_vec|None) as numpy arrays"""
    L = lib()
    ptr = np.ascontiguousarray(ptr, np.int32)
    idx = np.ascontiguousarray(idx, np.int32)
    val = None if val is None else np.ascontiguousarray(val, np.float32)
    n, m = len(ptr) - 1, len(idx)
    h = C.c_void_p()
    check(L.gnnagg_schedule_build(kind, _np(ptr), _np(idx), _np(val), n, m, par_num, neighbor_num,
                                  n if total_num_v is None else total_num_v, C.byref(h)))
    try:
        g, e = L.gnnagg_schedule_num_target(h), L.gnnagg_schedule_num_edges(h)

        def view(p, count, dt):
            if not p or count == 0:
                return np.empty(0, dt)
            return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_int32 if dt == np.int32 else C.c_float)),
                                         shape=(count,)).copy()

        out_ptr = view(L.gnnagg_schedule_ptr(h), g + 1, np.int32)
        out_idx = view(L.gnnagg_schedule_idx(h), e, np.int32)
        out_tgt = view(L.gnnagg_schedule_target(h), g, np.int32)
        pv = L.gnnagg_schedule_val(h)
        out_val = view(pv, e, np.float32) if (val is not None and kind != SCHED_NEIGHBOR_GROUPING) else None
    finally:
        L.gnnagg_schedule_free(h)
    return out_ptr, out_idx, out_tgt, out_val


def reorder_csr(ptr, idx, rows, reverse_rows):
    ptr = np.ascontiguousarray(ptr, np.int32)
    idx = np.ascontiguousarray(idx, np.int32)
    rows = np.ascontiguousarray(rows, np.int32)
    reverse_rows = np.ascontiguousarray(reverse_rows, np.int32)
    newptr, newidx = np.empty_like(ptr), np.empty_like(idx)
    check(lib().gnnagg_reorder_csr(_np(ptr), _np(idx), _np(rows), _np(reverse_rows), len(ptr) - 1, len(idx),
                                   _np(newptr), _np(newidx)))
    return newptr, newidx


def load_graph(dset, datadir="../data/", reorder_subfix=""):
    """reference load_graph(dset, ..., reorder_subfix) (src/data.cu:31): returns
    (indptr, indices, rows|None, reverse_rows|None)"""
    L = lib()
    nv, ne = C.c_int(), C.c_int()
    check(L.gnnagg_graph_config(datadir.encode(), dset.encode(), C.byref(nv), C.byref(ne)))
    ptr, idx = np.empty(nv.value + 1, np.int32), np.empty(ne.value, np.int32)
    rows, rev = np.empty(nv.value, np.int32), np.empty(nv.value, np.int32)
    reordered = C.c_int(0)
    rpath = (datadir + dset + ".reorder" + reorder_subfix) if reorder_subfix else ""
    check(L.gnnagg_graph_load(datadir.encode(), dset.encode(), rpath.encode(), nv.value, ne.value, _np(ptr), _np(idx),
                              _np(rows), _np(rev), C.byref(reordered)))
    if not reordered.value:
        rows = rev = None
    return ptr, idx, rows, rev


def write_graph(dset, ptr, idx, datadir="../data/"):
    ptr = np.ascontiguousarray(ptr, np.int32)
    idx = np.ascontiguousarray(idx, np.int32)
    check(lib().gnnagg_graph_write(datadir.encode(), dset.encode(), len(ptr) - 1, len(idx), _np(ptr), _np(idx)))


def lsh_reorder(ptr, idx, num_perm=0, bands=0, rows_per_band=0, cluster_cap=0, seed=1):
    ptr = np.ascontiguousarray(ptr, np.int32)
    idx = np.ascontiguousarray(idx, np.int32)
    rows = np.empty(len(ptr) - 1, np.int32)
    check(lib().gnnagg_lsh_reorder(_np(ptr), _np(idx), len(ptr) - 1, len(idx), num_perm, bands, rows_per_band,
                                   cluster_cap, seed, _np(rows)))
    return rows


def write_reorder(path, rows):
    rows = np.ascontiguousarray(rows, np.int32)
    check(lib().gnnagg_reorder_write(path.encode(), _np(rows), len(rows)))


# ------------------------------------------------------------------ device side (torch tensors)
def _stream():
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dp(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _f32(t, name, cuda=True):
    """device (or host) float32 operand of a C-ABI call: the library only sees a raw pointer, so a float64 tensor,
    a column-sliced view or a tensor on the wrong side would silently compute garbage -- reject them here"""
    import torch

    if t is None:
        return None
    if isinstance(t, np.ndarray):
        if cuda:
            raise GnnaggError("%s: expected a CUDA tensor, got a numpy array" % name)
        if t.dtype != np.float32 or not t.flags["C_CONTIGUOUS"]:
            raise GnnaggError("%s: numpy operand must be C-contiguous float32" % name)
        return C.c_void_p(t.ctypes.data)
    if t.dtype != torch.float32:
        raise GnnaggError("%s: expected float32, got %s" % (name, t.dtype))
    if not t.is_contiguous():
        raise GnnaggError("%s: expected a contiguous row-major tensor (got strides %s)" % (name, tuple(t.stride())))
    if bool(t.is_cuda) != bool(cuda):
        raise GnnaggError("%s: expected a %s tensor" % (name, "CUDA" if cuda else "host"))
    return C.c_void_p(t.data_ptr())


def _bf16(t, name, cuda=True):
    """bfloat16 torch operand (the gathered X / dY of the bf16 GCN entry points, or the host X shard of
    gnnagg_dist_gcn_layer_host_bf16 with cuda=False); numpy has no bf16, so numpy arrays are not accepted"""
    import torch

    if isinstance(t, np.ndarray) or t.dtype != torch.bfloat16:
        raise GnnaggError("%s: expected bfloat16, got %s" % (name, t.dtype))
    if not t.is_contiguous():
        raise GnnaggError("%s: expected a contiguous row-major tensor (got strides %s)" % (name, tuple(t.stride())))
    if bool(t.is_cuda) != bool(cuda):
        raise GnnaggError("%s: expected a %s tensor" % (name, "CUDA" if cuda else "host"))
    return C.c_void_p(t.data_ptr())


def _is_bf16(t):
    import torch

    return not isinstance(t, np.ndarray) and t.dtype == torch.bfloat16


def device_info():
    sm, ma, mi = C.c_int(), C.c_int(), C.c_int()
    name = C.create_string_buffer(256)
    check(lib().gnnagg_device_info(C.byref(sm), C.byref(ma), C.byref(mi), name, 256))
    return {"sm_count": sm.value, "cc": (ma.value, mi.value), "name": name.value.decode()}


class Aggregator:
    """Owner of a gnnagg_aggregator handle.  ptr/idx/val are int32/int32/float32 CUDA tensors that
    stay referenced for the lifetime of the object (the C ABI borrows them)."""

    def __init__(self, ptr, idx, val=None, h_ptr=None, h_idx=None):
        import torch

        if not (ptr.is_cuda and idx.is_cuda):
            raise GnnaggError("Aggregator needs CUDA tensors (there is no CPU path)")
        assert ptr.dtype == torch.int32 and idx.dtype == torch.int32
        self.ptr, self.idx, self.val = ptr.contiguous(), idx.contiguous(), None
        self._h_ptr = None if h_ptr is None else np.ascontiguousarray(h_ptr, np.int32)
        self._h_idx = None if h_idx is None else np.ascontiguousarray(h_idx, np.int32)
        self.n, self.m = ptr.numel() - 1, idx.numel()
        h = C.c_void_p()
        # set-up kernels go on torch's current stream: ptr/idx may still be in flight there, and the runs follow on it
        check(lib().gnnagg_create_on(_dp(self.ptr), _dp(self.idx), _np(self._h_ptr), _np(self._h_idx), self.n, self.m,
                                     C.byref(h), _stream()))
        self.h = h
        if val is not None:
            self.set_val(val)

    def close(self):
        if getattr(self, "h", None):
            lib().gnnagg_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_val(self, val):
        import torch

        if val.dtype != torch.float32 or not val.is_cuda or val.numel() != self.m:
            raise GnnaggError("set_val: expected a float32 CUDA tensor with one value per edge")
        self.val = val.contiguous()
        check(lib().gnnagg_set_val_on(self.h, _dp(self.val), _stream()))

    def schedule(self, kind, params, total_num_v=None):
        import torch

        torch.cuda.current_stream().synchronize()  # the schedule is built on the legacy stream from ptr/idx/val
        arr = (C.c_int * len(params))(*params)
        check(lib().gnnagg_schedule_apply(self.h, kind, arr, len(params), self.n if total_num_v is None else total_num_v))
        return self.num_target

    @property
    def num_target(self):
        return lib().gnnagg_num_target(self.h)

    @property
    def launches(self):
        return lib().gnnagg_launch_count(self.h)

    def set_warp_edges(self, warp_edges):
        check(lib().gnnagg_set_warp_edges(self.h, int(warp_edges)))

    def set_locality_slices(self, slices):
        check(lib().gnnagg_set_locality_slices(self.h, int(slices)))

    def set_merge_duplicates(self, mode):
        """0 automatic, 1 off, 2 on (gnnagg_set_merge_duplicates)"""
        check(lib().gnnagg_set_merge_duplicates(self.h, int(mode)))

    @property
    def merged_edges(self):
        """edges the GCN aggregation walks: m' of the merged view, or m when it is off"""
        import torch

        torch.cuda.current_stream().synchronize()  # the view is built on the legacy stream from ptr/idx
        e = lib().gnnagg_merged_edges(self.h)
        if e < 0:
            raise GnnaggError("gnnagg_merged_edges: %s" % lib().gnnagg_last_error().decode(errors="replace"))
        return e

    def merged_arrays(self):
        """the merged view as the last run left it, copied back as numpy (ptr, idx, val)"""
        import torch

        L = lib()
        p, i, v = C.c_void_p(), C.c_void_p(), C.c_void_p()
        check(L.gnnagg_merged_dev(self.h, C.byref(p), C.byref(i), C.byref(v)))
        torch.cuda.synchronize()
        mp = np.empty(self.n + 1, np.int32)
        check(L.gnnagg_memcpy_d2h(mp.ctypes.data, p, mp.nbytes))
        e = int(mp[-1])
        mi, mv = np.empty(e, np.int32), np.empty(e, np.float32)
        if e:
            check(L.gnnagg_memcpy_d2h(mi.ctypes.data, i, mi.nbytes))
            check(L.gnnagg_memcpy_d2h(mv.ctypes.data, v, mv.nbytes))
        return mp, mi, mv

    def set_host_pipeline(self, slices):
        check(lib().gnnagg_set_host_pipeline(self.h, int(slices)))

    def profile(self, on=True):
        check(lib().gnnagg_profile_enable(self.h, int(on)))

    def profile_read(self):
        """ms of the last run: dict(agg, agg_rest, dense, total)"""
        ms = (C.c_float * 4)()
        check(lib().gnnagg_profile_read(self.h, ms))
        return {"agg": ms[0], "agg_rest": ms[1], "dense": ms[2], "total": ms[3]}

    def scheduled_arrays(self):
        """device schedule copied back as numpy (ptr, idx, target, val|None)"""
        L = lib()
        g = self.num_target

        def back(p, count, dt):
            out = np.empty(count, dt)
            if p and count:
                check(L.gnnagg_memcpy_d2h(out.ctypes.data, p, count * 4))
            return out

        sp = back(L.gnnagg_sched_dev_ptr(self.h), g + 1, np.int32)
        e = int(sp[-1]) if g > 0 else 0
        si = back(L.gnnagg_sched_dev_idx(self.h), e, np.int32)
        stt = back(L.gnnagg_sched_dev_target(self.h), g, np.int32)
        pv = L.gnnagg_sched_dev_val(self.h)
        sv = back(pv, e, np.float32) if pv else None
        return sp, si, stt, sv

    # --- GCN (gcn_run, gcn_layer and gcn_backward take a float32 or a bfloat16 X / dY; outputs are float32)
    def gcn_run(self, X, Y, scheduled=False):
        if _is_bf16(X):
            check(lib().gnnagg_gcn_run_bf16(self.h, _bf16(X, "X"), _f32(Y, "Y"), X.shape[1], int(scheduled), _stream()))
        else:
            check(lib().gnnagg_gcn_run(self.h, _f32(X, "X"), _f32(Y, "Y"), X.shape[1], int(scheduled), _stream()))
        return Y

    def gcn_run_acc(self, X, Y, accumulate=True):
        if _is_bf16(X):
            check(lib().gnnagg_gcn_run_acc_bf16(self.h, _bf16(X, "X"), _f32(Y, "Y"), X.shape[1], int(accumulate), _stream()))
        else:
            check(lib().gnnagg_gcn_run_acc(self.h, _f32(X, "X"), _f32(Y, "Y"), X.shape[1], int(accumulate), _stream()))
        return Y

    def gcn_run_rows(self, X, Y, row_lo, row_hi, accumulate=False):
        if _is_bf16(X):
            check(lib().gnnagg_gcn_run_rows_bf16(self.h, _bf16(X, "X"), _f32(Y, "Y"), X.shape[1], int(accumulate), int(row_lo),
                                                 int(row_hi), _stream()))
        else:
            check(lib().gnnagg_gcn_run_rows(self.h, _f32(X, "X"), _f32(Y, "Y"), X.shape[1], int(accumulate), int(row_lo), int(row_hi),
                                            _stream()))
        return Y

    def gcn_run_edgewise(self, X, Y):
        check(lib().gnnagg_gcn_run_edgewise(self.h, _dp(X), _dp(Y), X.shape[1], _stream()))
        return Y

    def csr2edgelist(self, out):
        check(lib().gnnagg_csr2edgelist(self.h, _dp(out), _stream()))
        return out

    def gcn_layer(self, X, W, H, AX=None, scheduled=False):
        if _is_bf16(X):
            check(lib().gnnagg_gcn_layer_bf16(self.h, _bf16(X, "X"), _f32(W, "W"), _f32(H, "H"), _f32(AX, "AX"), W.shape[0],
                                              W.shape[1], int(scheduled), _stream()))
        else:
            check(lib().gnnagg_gcn_layer(self.h, _f32(X, "X"), _f32(W, "W"), _f32(H, "H"), _f32(AX, "AX"), W.shape[0], W.shape[1], int(scheduled),
                                         _stream()))
        return H

    # --- GAT
    def gat_run(self, X, att, Y, slope=0.2, scheduled=False):
        check(lib().gnnagg_gat_run(self.h, _f32(X, "X"), _f32(att, "att"), _f32(Y, "Y"), X.shape[1], slope, int(scheduled), _stream()))
        return Y

    def gat_edge_weights_ptr(self):
        return lib().gnnagg_gat_edge_weights(self.h)

    def edge_softmax(self, att, out_val, slope=0.2):
        check(lib().gnnagg_edge_softmax(self.h, _dp(att), _dp(out_val), slope, _stream()))
        return out_val

    def u_add_v(self, att, out_val):
        check(lib().gnnagg_u_add_v(self.h, _dp(att), _dp(out_val), _stream()))
        return out_val

    def add_to_center(self, in_val, out_center):
        check(lib().gnnagg_add_to_center(self.h, _dp(in_val), _dp(out_center), _stream()))
        return out_center

    def each_div(self, in_center, inout_val):
        check(lib().gnnagg_each_div(self.h, _dp(in_center), _dp(inout_val), _stream()))
        return inout_val

    # --- per-edge MLP aggregator (aggr_nn.h)
    def mlp_run(self, X, W, Y, scheduled=False):
        check(lib().gnnagg_mlp_run(self.h, _f32(X, "X"), _f32(W, "W"), _f32(Y, "Y"), X.shape[1], int(scheduled), _stream()))
        return Y

    # --- SDDMM
    def sddmm(self, X1, X2, out_val, scheduled=False):
        check(lib().gnnagg_sddmm(self.h, _f32(X1, "X1"), _f32(X2, "X2"), _f32(out_val, "out_val"), X1.shape[1], int(scheduled), _stream()))
        return out_val

    # --- backward (transposed CSR built once on the GPU, then gather-side aggregation over it)
    def transpose_build(self, num_src=None):
        self.num_src = self.n if num_src is None else int(num_src)
        check(lib().gnnagg_transpose_build(self.h, self.num_src, _stream()))

    def transposed_arrays(self):
        """(t_ptr, t_idx, t_perm) copied back as numpy"""
        L = lib()
        ns, tp, ti, tq = C.c_int(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        check(L.gnnagg_transpose_dev(self.h, C.byref(ns), C.byref(tp), C.byref(ti), C.byref(tq)))

        def back(p, count):
            out = np.empty(count, np.int32)
            if p.value and count:
                check(L.gnnagg_memcpy_d2h(out.ctypes.data, p, count * 4))
            return out

        return back(tp, ns.value + 1), back(ti, self.m), back(tq, self.m)

    def gcn_backward(self, dY, dX):
        if _is_bf16(dY):
            check(lib().gnnagg_gcn_backward_bf16(self.h, _bf16(dY, "dY"), _f32(dX, "dX"), dY.shape[1], _stream()))
        else:
            check(lib().gnnagg_gcn_backward(self.h, _f32(dY, "dY"), _f32(dX, "dX"), dY.shape[1], _stream()))
        return dX

    def gat_backward(self, X, att, Y, dY, dX, datt, slope=0.2, w=None, den=None):
        check(lib().gnnagg_gat_backward(self.h, _f32(X, "X"), _f32(att, "att"), _f32(w, "w"), _f32(den, "den"), _f32(Y, "Y"), _f32(dY, "dY"), _f32(dX, "dX"), _f32(datt, "datt"),
                                        X.shape[1], slope, _stream()))
        return dX, datt

    # --- sub-graph samplers (sample.h)
    def sample_subgraph(self, active, fanout=0, layer_num=1, seed=123):
        """active: int32 CUDA tensor [n] of seed flags, updated in place to the expanded set.  Returns
        (vertexset, sub_ptr, sub_idx) as int32 CUDA tensors (copies; the library's arrays are released)."""
        import torch

        L = lib()
        vs, sp, si = C.c_void_p(), C.c_void_p(), C.c_void_p()
        nv, ne = C.c_int(), C.c_int()
        check(L.gnnagg_sample_subgraph(self.h, _dp(active), int(fanout), int(layer_num), C.c_uint64(seed), C.byref(vs),
                                       C.byref(sp), C.byref(si), C.byref(nv), C.byref(ne), _stream()))
        out = []
        for p_, count in ((vs, nv.value), (sp, nv.value + 1), (si, ne.value)):
            t = torch.empty(count, dtype=torch.int32, device=active.device)
            if count:
                h = np.empty(count, np.int32)
                check(L.gnnagg_memcpy_d2h(h.ctypes.data, p_, count * 4))
                t.copy_(torch.from_numpy(h))
            check(L.gnnagg_device_free(p_))
            out.append(t)
        return tuple(out)

    # --- host-buffer entry points (pinned CPU tensors or numpy arrays)
    def gcn_run_host(self, hX, hY, scheduled=False):
        check(lib().gnnagg_gcn_run_host(self.h, _f32(hX, "hX", cuda=False), _f32(hY, "hY", cuda=False), hX.shape[1], int(scheduled), _stream()))
        return hY

    def gcn_layer_host(self, hX, hW, hH, scheduled=False):
        check(lib().gnnagg_gcn_layer_host(self.h, _f32(hX, "hX", cuda=False), _f32(hW, "hW", cuda=False), _f32(hH, "hH", cuda=False), hW.shape[0], hW.shape[1], int(scheduled),
                                          _stream()))
        return hH

    def gat_run_host(self, hX, hatt, hY, slope=0.2, scheduled=False):
        check(lib().gnnagg_gat_run_host(self.h, _f32(hX, "hX", cuda=False), _f32(hatt, "hatt", cuda=False), _f32(hY, "hY", cuda=False), hX.shape[1], slope, int(scheduled),
                                        _stream()))
        return hY


def dense_nn(A, B, Cout):
    check(lib().gnnagg_dense_nn(_f32(A, "A"), _f32(B, "B"), _f32(Cout, "C"), A.shape[0], B.shape[1], A.shape[1], _stream()))
    return Cout


def gather_rows(X, rows, out):
    """out[i] = X[rows[i]] (rows: int64 CUDA tensor)"""
    check(lib().gnnagg_gather_rows(_dp(X), _dp(rows), _dp(out), rows.numel(), X.shape[1], _stream()))
    return out


def spmm_naive(ptr, idx, val, X, Y):
    check(lib().gnnagg_spmm_naive(ptr.numel() - 1, _dp(ptr), _dp(idx), _dp(val), _dp(X), _dp(Y), X.shape[1], _stream()))
    return Y


def validate(ref, ans):
    d = C.c_int()
    check(lib().gnnagg_validate(_dp(ref), _dp(ans), ref.numel(), C.byref(d), _stream()))
    return d.value


def validate_reordered(ref, ans, rows_map):
    d = C.c_int()
    check(lib().gnnagg_validate_reordered(_dp(ref), _dp(ans), _dp(rows_map), ref.shape[0], ref.shape[1], C.byref(d),
                                          _stream()))
    return d.value
