"""ctypes binding of libpnp_ovss_b200.so (the C ABI declared in include/pnp_ovss_b200.h).

There is no CPU fallback: if the library has not been built (`python __graft_entry__.py` or
`make -C pnp_ovss_b200/csrc`) importing an op raises, and every op refuses non-CUDA tensors."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpnp_ovss_b200.so")

c_int, c_float, c_double, c_void_p, c_size_t = ctypes.c_int, ctypes.c_float, ctypes.c_double, ctypes.c_void_p, ctypes.c_size_t


class PnpError(RuntimeError):
    pass


class Lattice(ctypes.Structure):
    """struct pnp_lattice (include/pnp_ovss_b200.h)."""
    _fields_ = [("d", c_int), ("n_images", c_int), ("n_pixels", c_int), ("shared", c_int), ("n_vertices", c_int),
                ("max_row", c_int), ("vertex_stride", c_int), ("width", c_int),
                ("offset", c_void_p), ("bary", c_void_p), ("nbr", c_void_p), ("row_ptr", c_void_p), ("csr_pix", c_void_p),
                ("csr_w", c_void_p), ("csr_norm", c_void_p), ("norm", c_void_p), ("counters", c_void_p)]


_LP = ctypes.POINTER(Lattice)

# name -> (restype, argtypes); must list every symbol the header declares (tests/test_boundary.py checks)
SIGNATURES = {
    "pnp_abi_version": (c_int, []),
    "pnp_error_string": (ctypes.c_char_p, [c_int]),
    "pnp_compiled_sm": (c_int, []),
    "pnp_xattn_softmax_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "pnp_xattn_softmax_bwd_gradcam": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int,
                                              c_int, c_float, c_int, c_void_p]),
    "pnp_token_merge": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "pnp_salience_dropout_round": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int,
                                           c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "pnp_threshold_upsample_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "pnp_threshold_upsample": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_int, c_int, c_float,
                                       c_int, c_int, c_void_p]),
    "pnp_gaussian_blur_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_double]),
    "pnp_gaussian_blur": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_double, c_int,
                                  c_void_p]),
    "pnp_lowrank_blur_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_double, c_int]),
    "pnp_lowrank_blur_unary": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_int,
                                       c_int, c_float, c_int, c_int, c_double, c_void_p]),
    "pnp_lowrank_blur_unary_padded": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int,
                                              c_int, c_int, c_float, c_int, c_int, c_double, c_void_p]),
    "pnp_lattice_storage_bytes": (c_size_t, [c_int, c_int, c_int]),
    "pnp_lattice_build_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "pnp_lattice_init": (c_int, [_LP, c_void_p, c_size_t, c_int, c_int, c_int, c_int]),
    "pnp_lattice_build": (c_int, [_LP, c_void_p, c_int, c_int, c_float, c_float, c_float, c_float, c_float, c_void_p,
                                  c_size_t, c_void_p]),
    "pnp_lattice_finish": (c_int, [_LP, c_void_p]),
    "pnp_crf_unary_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "pnp_crf_unary_from_maps": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_void_p]),
    "pnp_crf_pack_cn_to_nc": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "pnp_crf_unpack_nc_to_cn": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "pnp_crf_scratch_bytes": (c_size_t, [ctypes.POINTER(_LP), c_int, c_int, c_int]),
    "pnp_crf_filter": (c_int, [_LP, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_void_p]),
    "pnp_crf_inference": (c_int, [ctypes.POINTER(_LP), ctypes.POINTER(c_float), c_int, c_void_p, c_void_p, c_void_p,
                                  c_size_t, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "pnp_tf32_split3": (c_int, [c_void_p, c_void_p, ctypes.c_longlong, c_int, c_void_p]),
    "pnp_gelu_tf32_split3": (c_int, [c_void_p, c_void_p, c_void_p, ctypes.c_longlong, c_int, c_void_p]),
    "pnp_layernorm_tf32_split3": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p,
                                          ctypes.c_longlong, c_int, c_void_p]),
    "pnp_fp16_split3": (c_int, [c_void_p, c_float, c_float, c_void_p, c_void_p, ctypes.c_longlong, c_int, c_void_p]),
    "pnp_gelu_fp16_split3": (c_int, [c_void_p, c_float, c_void_p, c_float, c_void_p, c_void_p, ctypes.c_longlong, c_int, c_void_p]),
    "pnp_layernorm_fp16_split3": (c_int, [c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_float, c_void_p,
                                          c_int, c_float, c_void_p, c_void_p, ctypes.c_longlong, c_int, c_void_p]),
    "pnp_attention_fp16x3_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "pnp_attention_fp16x3": (c_int, [c_void_p, c_float, c_float, c_void_p, c_void_p, c_float, c_void_p, c_size_t, c_void_p, c_int, c_int,
                                     c_int, c_int, c_void_p]),
    "pnp_profile_num_kernels": (c_int, []),
    "pnp_profile_start": (c_int, [ctypes.c_uint]),
    "pnp_profile_stop": (c_int, [ctypes.POINTER(c_float), ctypes.POINTER(c_int), c_int]),
    "pnp_profile_kernel_name": (ctypes.c_char_p, [c_int]),
    "pnp_profile_filter_stream": (c_int, [c_void_p, c_int]),
    "pnp_argmax_channels": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "pnp_confusion_accumulate": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                         c_int, c_void_p]),
    "pnp_label_map": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p]),
}

_lib = None


def load():
    """Load the shared library (once) and attach signatures.  Raises PnpError if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PnpError(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C pnp_ovss_b200/csrc`).  pnp_ovss_b200 has no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:
            raise PnpError("libpnp_ovss_b200.so does not export %s (stale build?)" % name) from exc
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.pnp_abi_version() != 1:
        raise PnpError("ABI version mismatch: header 1, library %d" % lib.pnp_abi_version())
    _lib = lib
    return lib


def check(code, what):
    if code != 0:
        msg = load().pnp_error_string(code).decode()
        raise PnpError("%s failed: %s (code %d)" % (what, msg, code))
