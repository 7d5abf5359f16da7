"""pnp_ovss_b200 -- the PnP-OVSS mask-extraction hot path as hand-written sm_100a CUDA behind a C ABI.

  include/pnp_ovss_b200.h   the C ABI (libpnp_ovss_b200.so, built from pnp_ovss_b200/csrc/*.cu)
  _lib / ops                ctypes binding and tensor-level wrappers (pointers + stream only)
  host                      string/table logic of the path (token segments, relabel LUT, sharding)
  reference_api             drop-in replacements with the reference's function names and signatures
  pipeline                  batched on-device composition + the int64 confusion-matrix all-reduce
  blip_itm                  BLIP ITM-large whose block-8 cross-attention uses kernel (a) (random init offline)
  lavis_compat              LAVIS checkpoint -> that model; GradCAM from a live LAVIS BlipITM with kernel (a) patched in
  data, driver              the reference's dataset layouts / transform / tokenizer; driver with the reference's CLI
  segment                   segment_images: label maps of caller-supplied images and class names, without ground truth

There is no CPU fallback anywhere in this package (oracle/ is test infrastructure and is never imported here)."""
from ._lib import PnpError, LIB_PATH  # noqa: F401
from .segment import segment_images  # noqa: F401

__all__ = ["PnpError", "LIB_PATH", "segment_images"]
