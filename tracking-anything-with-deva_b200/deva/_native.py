"""ctypes binding of libdeva_b200.so (C ABI declared in include/deva_b200.h).

This is the only door between the Python host code and the sm_100a kernels.  There is no
fallback: if the library is missing, was built for another ABI version, or a kernel reports an
error, a RuntimeError is raised.  PyTorch is used for device memory and streams only.
"""
import ctypes
import os
from ctypes import c_char_p, c_int, c_int32, c_int64, c_size_t, c_uint64, c_void_p, POINTER

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), 'csrc', 'libdeva_b200.so')
ABI_VERSION = 12
LIST_PITCH = 32
MAX_GROUPS = 256

_lib = None


class ConvDesc(ctypes.Structure):
    """Mirror of ``deva_b200_conv_desc`` (include/deva_b200.h)."""
    _fields_ = [('x', c_void_p), ('x2', c_void_p), ('x_lo', c_void_p), ('split_mode', c_int32), ('batch', c_int32), ('h', c_int32), ('w', c_int32), ('cin_pad', c_int32),
                ('w_packed', c_void_p), ('kh', c_int32), ('kw', c_int32), ('stride', c_int32),
                ('cout', c_int32), ('cout_pad', c_int32), ('nt', c_int32), ('th', c_int32), ('tw', c_int32),
                ('bias', c_void_p), ('res', c_void_p), ('res_lo', c_void_p), ('res_broadcast', c_int32),
                ('rank1_w', c_void_p), ('rank1_x', c_void_p),
                ('out_raw', c_void_p), ('out_relu', c_void_p), ('out_f32', c_void_p),
                ('out_raw_lo', c_void_p), ('out_relu_lo', c_void_p),
                ('head_w', c_void_p), ('head_out', c_void_p), ('head_n', c_int32),
                ('gate_h', c_void_p), ('gate_out', c_void_p), ('x_lo8', c_void_p), ('w8_packed', c_void_p),
                ('acc_scale', ctypes.c_float), ('out_relu_lo8', c_void_p), ('ksplit', c_int32)]


_SIGNATURES = {
    'deva_b200_abi_version': (c_int, []),
    'deva_b200_last_error': (c_char_p, []),
    'deva_b200_launch_count': (c_uint64, []),
    'deva_b200_device_check': (c_int, []),
    'deva_b200_pack_query': (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p,
                                     c_void_p, c_void_p]),
    'deva_b200_pack_keys': (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int, c_int, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    'deva_b200_append_values': (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int, c_int, c_void_p]),
    'deva_b200_simtopk_workspace_bytes': (c_size_t, [c_int]),
    'deva_b200_sim_topk': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int,
                                   c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                   c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    'deva_b200_merge_lists': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                      c_void_p]),
    'deva_b200_sim_dense_softmax': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p,
                                            c_void_p, c_int, c_int, c_void_p, c_int64, c_void_p, c_int64, c_void_p,
                                            c_void_p]),
    'deva_b200_readout': (c_int, [c_void_p, c_int64, c_int64, POINTER(c_int32), POINTER(c_int32), c_int, c_int,
                                  c_void_p, c_int64, c_int, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
    'deva_b200_readout_sparse_workspace_bytes': (c_size_t, [c_int, c_int]),
    'deva_b200_readout_sparse': (c_int, [c_void_p, c_int64, c_int64, POINTER(c_int32), POINTER(c_int32), c_int, c_int,
                                         c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p,
                                         c_void_p]),
    'deva_b200_readout_sparse_scatter': (c_int, [c_void_p, c_int64, c_int64, POINTER(c_int32), POINTER(c_int32),
                                                 POINTER(c_int32), c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int,
                                                 c_void_p, POINTER(c_void_p), c_int, c_int64, c_void_p]),
    'deva_b200_enable_peer_access': (c_int, [c_int, c_int]),
    'deva_b200_peer_alloc': (c_int, [c_int, c_int64, POINTER(c_void_p), c_char_p]),
    'deva_b200_peer_open': (c_int, [c_int, c_char_p, POINTER(c_void_p)]),
    'deva_b200_peer_close': (c_int, [c_int, c_void_p]),
    'deva_b200_peer_free': (c_int, [c_int, c_void_p]),
    'deva_b200_gather_rows': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    'deva_b200_gather_f32': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    'deva_b200_gather_cols_f16': (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int, c_int, c_void_p]),
    'deva_b200_usage': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    'deva_b200_conv2d': (c_int, [POINTER(ConvDesc), c_void_p]),
    'deva_b200_stem_im2col': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    'deva_b200_nchw_to_nhwc': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    'deva_b200_nhwc_to_nchw': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    'deva_b200_maxpool': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    'deva_b200_up2_add': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    'deva_b200_area_down': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    'deva_b200_area_down_plane': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    'deva_b200_cbam': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    'deva_b200_up2_add_split': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    'deva_b200_cbam_split': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                     c_int, c_void_p]),
    'deva_b200_gru': (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    'deva_b200_sum_parts': (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_int64, c_void_p]),
    'deva_b200_key_tail': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    'deva_b200_output_tail': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    'deva_b200_head_gather3x3': (c_int, [c_void_p, c_void_p, ctypes.c_float, c_int, c_int, c_int, c_void_p]),
    'deva_b200_transpose_append': (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p]),
    'deva_b200_ingest_rgb8': (c_int, [c_void_p, c_void_p, c_int, c_int, ctypes.POINTER(ctypes.c_float),
                                      ctypes.POINTER(ctypes.c_float), c_void_p]),
    'deva_b200_prob_to_ids': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                      c_void_p]),
    'deva_b200_resize_rgb8_workspace_bytes': (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    'deva_b200_resize_rgb8': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                      ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float), c_void_p]),
    'deva_b200_resize_aa_weights': (c_int, [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    'deva_b200_resize_labels': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
}
EXPORTS = tuple(_SIGNATURES.keys())


def lib():
    """Load (once) and return the shared library; raises if it is missing or mismatched."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f'deva_b200: CUDA library not built: {LIB_PATH} (run __graft_entry__.build() or '
                               f'`make -C {os.path.dirname(LIB_PATH)}`); there is no CPU fallback')
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        if handle.deva_b200_abi_version() != ABI_VERSION:
            raise RuntimeError('deva_b200: ABI version mismatch between deva/_native.py and libdeva_b200.so')
        _lib = handle
    return _lib


def _check(rc: int, what: str):
    if rc != 0:
        msg = lib().deva_b200_last_error()
        raise RuntimeError(f'deva_b200.{what} failed ({rc}): {msg.decode() if msg else "?"}')


def _ptr(t):
    return None if t is None else c_void_p(t.data_ptr())


def _stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def launch_count() -> int:
    return int(lib().deva_b200_launch_count())


def require_device():
    if not torch.cuda.is_available():
        raise RuntimeError('deva_b200: no CUDA device; the sm_100a kernels have no CPU fallback')
    _check(lib().deva_b200_device_check(), 'device_check')


def _f32(t):
    assert t.dtype == torch.float32 and t.is_cuda, (t.dtype, t.device)
    return t


# ------------------------------------------------------------------------------------------ wrappers
def pack_query(qk, qe, stride_c, stride_q, ck, q, q_hi, q_lo, bsq):
    _check(lib().deva_b200_pack_query(_ptr(_f32(qk)), _ptr(_f32(qe)), stride_c, stride_q, ck, q, _ptr(q_hi),
                                      _ptr(q_lo), _ptr(bsq), _stream()), 'pack_query')


def pack_keys(key, selection, stride_c, stride_t, shrinkage, ck, n, k_hi, k_lo, neg_s, raw_key, raw_sel, raw_shr):
    _check(lib().deva_b200_pack_keys(_ptr(_f32(key)), _ptr(selection), stride_c, stride_t, _ptr(_f32(shrinkage)), ck,
                                     n, _ptr(k_hi), _ptr(k_lo), _ptr(neg_s), _ptr(raw_key), _ptr(raw_sel),
                                     _ptr(raw_shr), _stream()), 'pack_keys')


def append_values(src, ld_src, dst, ld_dst, rows, n):
    _check(lib().deva_b200_append_values(_ptr(_f32(src)), ld_src, _ptr(dst), ld_dst, rows, n, _stream()),
           'append_values')


def simtopk_workspace_bytes(q):
    return int(lib().deva_b200_simtopk_workspace_bytes(q))


def sim_topk(k_hi, k_lo, neg_s, n_window, n_lead, q_hi, q_lo, bsq, q, ck, top_k, workspace, out_idx, out_w,
             affinity, ld_affinity, use_cnt, life_cnt, n_long, count_long, count_work, out_sim=None, prev_idx=None,
             thr_ws=None):
    _check(lib().deva_b200_sim_topk(_ptr(k_hi), _ptr(k_lo), _ptr(neg_s), n_window, n_lead, _ptr(q_hi), _ptr(q_lo),
                                    _ptr(bsq), q, ck, top_k, _ptr(workspace), _ptr(out_idx), _ptr(out_w),
                                    _ptr(affinity), ld_affinity, _ptr(use_cnt), _ptr(life_cnt), n_long,
                                    int(count_long), int(count_work), _ptr(out_sim), _ptr(prev_idx), _ptr(thr_ws),
                                    _stream()), 'sim_topk')


def merge_lists(part_val, part_idx, n_lists, top_k, q, q_pitch, out_idx, out_w, out_sim=None):
    _check(lib().deva_b200_merge_lists(_ptr(part_val), _ptr(part_idx), n_lists, top_k, q, q_pitch, _ptr(out_idx),
                                       _ptr(out_w), _ptr(out_sim), _stream()), 'merge_lists')


def sim_dense_softmax(k_hi, k_lo, neg_s, shrinkage, n_window, n_lead, q_hi, q_lo, bsq, q, ck, sim_ws, ld_sim,
                      affinity, ld_affinity, shr_out):
    _check(lib().deva_b200_sim_dense_softmax(_ptr(k_hi), _ptr(k_lo), _ptr(neg_s), _ptr(shrinkage), n_window, n_lead,
                                             _ptr(q_hi), _ptr(q_lo), _ptr(bsq), q, ck, _ptr(sim_ws), ld_sim,
                                             _ptr(affinity), ld_affinity, _ptr(shr_out), _stream()),
           'sim_dense_softmax')


def readout(values, values_ld, values_rows, val_row, out_row, rows_per_group, affinity, ld_affinity, n_window, q,
            out, ld_out, out_tok=None):
    n = len(val_row)
    assert n == len(out_row)
    arr_v = (c_int32 * n)(*val_row)
    arr_o = (c_int32 * n)(*out_row)
    _check(lib().deva_b200_readout(_ptr(values), values_ld, values_rows, arr_v, arr_o, n, rows_per_group,
                                   _ptr(affinity), ld_affinity, n_window, q, _ptr(out), ld_out, _ptr(out_tok),
                                   _stream()), 'readout')


def readout_sparse_workspace_bytes(q, n_window):
    return int(lib().deva_b200_readout_sparse_workspace_bytes(q, n_window))


def readout_sparse(values, values_ld, values_rows, val_row, out_row, rows_per_group, idx, w, top_k, n_window, q,
                   workspace, out, ld_out, out_tok=None):
    n = len(val_row)
    arr_v = (c_int32 * n)(*val_row)
    arr_o = (c_int32 * n)(*out_row)
    _check(lib().deva_b200_readout_sparse(_ptr(values), values_ld, values_rows, arr_v, arr_o, n, rows_per_group,
                                          _ptr(idx), _ptr(w), top_k, n_window, q, _ptr(workspace), _ptr(out), ld_out,
                                          _ptr(out_tok), _stream()), 'readout_sparse')


def readout_sparse_scatter(values, values_ld, values_rows, val_row, out_row, owner, rows_per_group, idx, w, top_k,
                           n_window, q, workspace, rank_dst_ptrs, ld_out):
    """rank_dst_ptrs: device addresses (ints) of every rank's fp32 [objects_owned * rows_per_group, q] buffer."""
    n = len(val_row)
    arr_v, arr_o, arr_w = (c_int32 * n)(*val_row), (c_int32 * n)(*out_row), (c_int32 * n)(*owner)
    ptrs = (c_void_p * len(rank_dst_ptrs))(*rank_dst_ptrs)
    _check(lib().deva_b200_readout_sparse_scatter(_ptr(values), values_ld, values_rows, arr_v, arr_o, arr_w, n,
                                                  rows_per_group, _ptr(idx), _ptr(w), top_k, n_window, q,
                                                  _ptr(workspace), ptrs, len(rank_dst_ptrs), ld_out, _stream()),
           'readout_sparse_scatter')


def peer_alloc(device: int, nbytes: int):
    """-> (device address, 64-byte CUDA IPC handle) of a zeroed cudaMalloc'ed buffer on ``device``."""
    ptr, handle = c_void_p(), ctypes.create_string_buffer(64)
    _check(lib().deva_b200_peer_alloc(device, nbytes, ctypes.byref(ptr), handle), 'peer_alloc')
    return int(ptr.value), handle.raw


def peer_open(device: int, handle: bytes) -> int:
    ptr = c_void_p()
    _check(lib().deva_b200_peer_open(device, handle, ctypes.byref(ptr)), 'peer_open')
    return int(ptr.value)


def peer_close(device: int, ptr: int):
    _check(lib().deva_b200_peer_close(device, c_void_p(ptr)), 'peer_close')


def peer_free(device: int, ptr: int):
    _check(lib().deva_b200_peer_free(device, c_void_p(ptr)), 'peer_free')


def enable_peer_access(device: int, peer_device: int):
    _check(lib().deva_b200_enable_peer_access(device, peer_device), 'enable_peer_access')


def gather_rows(dst, src, idx, n, row_bytes):
    _check(lib().deva_b200_gather_rows(_ptr(dst), _ptr(src), _ptr(idx), n, row_bytes, _stream()), 'gather_rows')


def gather_f32(dst, src, idx, n):
    _check(lib().deva_b200_gather_f32(_ptr(dst), _ptr(src), _ptr(idx), n, _stream()), 'gather_f32')


def gather_cols_f16(dst, ld_dst, src, ld_src, idx, rows, n):
    _check(lib().deva_b200_gather_cols_f16(_ptr(dst), ld_dst, _ptr(src), ld_src, _ptr(idx), rows, n, _stream()),
           'gather_cols_f16')


def usage(out, use_cnt, life_cnt, n):
    _check(lib().deva_b200_usage(_ptr(out), _ptr(use_cnt), _ptr(life_cnt), n, _stream()), 'usage')


# ------------------------------------------------------------------------------------------ network path
def _p(t):
    return None if t is None else t.data_ptr()


def conv2d(x, batch, h, w, cin_pad, w_packed, kh, stride, cout, cout_pad, nt, th, tw, bias, x2=None, x_lo=None, res=None,
           res_lo=None, res_broadcast=False, rank1_w=None, rank1_x=None, out_raw=None, out_relu=None, out_f32=None,
           out_raw_lo=None, out_relu_lo=None, head_w=None, head_out=None, head_n=0, gate_h=None, gate_out=None,
           split_mode=0, ksplit=0, x_lo8=None, w8_packed=None, acc_scale=0.0, out_relu_lo8=None):
    d = ConvDesc(_p(x), _p(x2), _p(x_lo), split_mode, batch, h, w, cin_pad, _p(w_packed), kh, kh, stride, cout, cout_pad, nt, th, tw,
                 _p(bias), _p(res), _p(res_lo), int(res_broadcast), _p(rank1_w), _p(rank1_x), _p(out_raw), _p(out_relu),
                 _p(out_f32), _p(out_raw_lo), _p(out_relu_lo), _p(head_w), _p(head_out), head_n, _p(gate_h), _p(gate_out), _p(x_lo8), _p(w8_packed), acc_scale,
                 _p(out_relu_lo8), ksplit)
    _check(lib().deva_b200_conv2d(ctypes.byref(d), _stream()), 'conv2d')


def stem_im2col(src, dst, b, c, h, w, k_pad, dst_lo=None):
    _check(lib().deva_b200_stem_im2col(_ptr(_f32(src)), _ptr(dst), _ptr(dst_lo), b, c, h, w, k_pad, _stream()),
           'stem_im2col')


def nchw_to_nhwc(src, dst, b, c, h, w, c_pad):
    _check(lib().deva_b200_nchw_to_nhwc(_ptr(src), _ptr(dst), b, c, h, w, c_pad, _stream()), 'nchw_to_nhwc')


def nhwc_to_nchw(src, dst, b, c, h, w):
    _check(lib().deva_b200_nhwc_to_nchw(_ptr(src), _ptr(dst), b, c, h, w, _stream()), 'nhwc_to_nchw')


def maxpool(x, y, b, h, w, c, x_lo=None, y_lo=None):
    _check(lib().deva_b200_maxpool(_ptr(x), _ptr(x_lo), _ptr(y), _ptr(y_lo), b, h, w, c, _stream()), 'maxpool')


def up2_add(g, skip, raw, relu, b, h, w, c):
    _check(lib().deva_b200_up2_add(_ptr(g), _ptr(skip), _ptr(raw), _ptr(relu), b, h, w, c, _stream()), 'up2_add')


def area_down(x, y, b, h, w, c, r):
    _check(lib().deva_b200_area_down(_ptr(x), _ptr(y), b, h, w, c, r, _stream()), 'area_down')


def area_down_plane(x, y, b, h, w, r):
    _check(lib().deva_b200_area_down_plane(_ptr(x), _ptr(y), b, h, w, r, _stream()), 'area_down_plane')


def cbam(x, w1, b1, w2, b2, ws, bs, scratch, raw, relu, b, h, w, c, r):
    _check(lib().deva_b200_cbam(_ptr(x), _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2), _ptr(ws), _ptr(bs), _ptr(scratch),
                                _ptr(raw), _ptr(relu), b, h, w, c, r, _stream()), 'cbam')


def up2_add_split(g, g_lo, skip, raw, raw_lo, relu, b, h, w, c, skip_lo=None, relu_lo=None, relu_lo8=None):
    _check(lib().deva_b200_up2_add_split(_ptr(g), _ptr(g_lo), _ptr(skip), _ptr(skip_lo), _ptr(raw), _ptr(raw_lo),
                                         _ptr(relu), _ptr(relu_lo), _ptr(relu_lo8), b, h, w, c, _stream()), 'up2_add_split')


def cbam_split(x, x_lo, w1, b1, w2, b2, ws, bs, scratch, raw, raw_lo, relu, b, h, w, c, r, relu_lo=None, pool_lo=True):
    _check(lib().deva_b200_cbam_split(_ptr(x), _ptr(x_lo), _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2), _ptr(ws), _ptr(bs),
                                      _ptr(scratch), _ptr(raw), _ptr(raw_lo), _ptr(relu), _ptr(relu_lo), int(pool_lo), b, h,
                                      w, c, r, _stream()), 'cbam_split')


def gru(values, h, out, pixels, c):
    _check(lib().deva_b200_gru(_ptr(values), _ptr(h), _ptr(out), pixels, c, _stream()), 'gru')


def sum_parts(parts, n_parts, part_stride, n, res=None, res_lo=None, raw=None, raw_lo=None, relu=None, relu_lo=None):
    _check(lib().deva_b200_sum_parts(_ptr(parts), n_parts, part_stride, _ptr(res), _ptr(res_lo), _ptr(raw), _ptr(raw_lo),
                                     _ptr(relu), _ptr(relu_lo), n, _stream()), 'sum_parts')


def key_tail(y, ld, q, ck, key, shrinkage, selection, n_parts=1, part_stride=0):
    _check(lib().deva_b200_key_tail(_ptr(y), ld, q, ck, n_parts, part_stride, _ptr(key), _ptr(shrinkage), _ptr(selection),
                                    _stream()), 'key_tail')


def output_tail(logits, agg, prob, logits_out, k, h, w):
    _check(lib().deva_b200_output_tail(_ptr(logits), _ptr(agg), _ptr(prob), _ptr(logits_out), k, h, w, _stream()),
           'output_tail')


def ingest_rgb8(src, dst, h, w, mean, std):
    m = (ctypes.c_float * 3)(*[float(v) for v in mean])
    s = (ctypes.c_float * 3)(*[float(v) for v in std])
    _check(lib().deva_b200_ingest_rgb8(_ptr(src), _ptr(dst), h, w, m, s, _stream()), 'ingest_rgb8')


def prob_to_ids(prob, c, h, w, out_h, out_w, flip, lut, out_u8, out_i64):
    _check(lib().deva_b200_prob_to_ids(_ptr(prob), c, h, w, out_h, out_w, int(flip), _p(lut), _p(out_u8), _p(out_i64),
                                       _stream()), 'prob_to_ids')


RESIZE_MODES = {'reader': 0, 'demo': 1}  # DEVA_B200_RESIZE_READER / _DEMO


def resize_rgb8_workspace_bytes(h, w, out_h, out_w, mode):
    return lib().deva_b200_resize_rgb8_workspace_bytes(h, w, out_h, out_w, RESIZE_MODES[mode])


def resize_rgb8(src, dst, ws, h, w, out_h, out_w, mode, mean, std):
    m = (ctypes.c_float * 3)(*[float(v) for v in mean])
    s = (ctypes.c_float * 3)(*[float(v) for v in std])
    _check(lib().deva_b200_resize_rgb8(_ptr(src), _ptr(dst), _p(ws), h, w, out_h, out_w, RESIZE_MODES[mode], m, s,
                                       _stream()), 'resize_rgb8')


def resize_aa_weights(n_in, n_out):
    """Host tap tables of the antialiased resize n_in -> n_out: (x0 int32 [n_out], n int32 [n_out], w fp32 [n_out, T])."""
    taps = 2 * (n_in // n_out + 2) + 1  # >= 2 * ceil(max(n_in / n_out, 1)) + 1
    x0 = torch.empty(n_out, dtype=torch.int32)
    n = torch.empty(n_out, dtype=torch.int32)
    w = torch.empty(n_out, taps, dtype=torch.float32)
    _check(lib().deva_b200_resize_aa_weights(n_in, n_out, taps, _ptr(x0), _ptr(n), _ptr(w)), 'resize_aa_weights')
    return x0, n, w


def resize_labels(src, dst, h, w, out_h, out_w, src_y, src_x):
    _check(lib().deva_b200_resize_labels(_ptr(src), _ptr(dst), h, w, out_h, out_w, _ptr(src_y), _ptr(src_x), _stream()),
           'resize_labels')


def transpose_append(src, dst, ld_dst, n, c):
    _check(lib().deva_b200_transpose_append(_ptr(src), _ptr(dst), ld_dst, n, c, _stream()), 'transpose_append')


def head_gather3x3(z, out, bias, b, h, w):
    _check(lib().deva_b200_head_gather3x3(_ptr(z), _ptr(out), float(bias), b, h, w, _stream()), 'head_gather3x3')
