"""decaf377_b200 -- B200-native batch engine for the decaf377 group.

Host-side mirror of the reference crate's public surface (src/lib.rs:7-29):
``Fq``, ``Fr``, ``Element``, ``Encoding``, ``EncodingError``, ``ZETA`` plus the
batch entry points that are the point of this package.  All group/field batch
work runs in hand-written CUDA (sm_100a) behind the C ABI declared in
``include/decaf377_b200.h``.
"""
from .api import (  # noqa: F401
    Element, AffinePoint, Encoding, EncodingError, Fq, Fr, ZETA,
    init, init_multi, set_device, get_device, device_list, shutdown, sync, join, launch_count,
    imad_peak, msm_set_window, msm_set_host_chunks, msm_set_tail_overlap, debug_build, debug_counts,
    batch_sub, batch_neg, batch_double, batch_on_curve, fq_batch_from_le_bytes_mod_order, msm_multi, batch_msm,
    msm_segmented, msm_segmented_last,
    msm_set_normalize, msm_set_groups,
    msm_stage_info, msm_timeline, pinned_empty, pinned_copy,
    batch_decompress, batch_compress, batch_compress_fmt, batch_affine_serialize, batch_affine_deserialize,
    batch_encode_to_curve, batch_hash_to_curve,
    batch_scalar_mul, fixed_base_mul, batch_add, batch_element_eq, element_sum,
    vartime_multiscalar_mul, msm_submit, msm_wait, MsmBases, FixedBases, fq_batch_op, fq_batch_isqrt,
    fq_batch_sqrt_ratio_zeta, field_batch_deserialize, batch_normalize, FIELD_FQ, FIELD_FR,
    PT_ELEMENT, PT_ENCODING, PT_AFFINE, PT_XYZ, PT_BASES, OUT_ELEMENT, OUT_ENCODING, SCALARS_MONTGOMERY,
)
from . import device  # noqa: F401
