/* decaf377_b200 -- C ABI of the B200-native decaf377 batch engine.
 *
 * The reference crate (penumbra-zone/decaf377 v0.10.1) has no FFI; its "plugin
 * API" is the public Rust surface of src/lib.rs:7-29.  This header is the seam
 * a Rust shim (see INTEGRATION.md) binds with `extern "C"`; every entry point
 * names the reference item it replaces.  All paths are relative to the
 * reference tree.
 *
 * Conventions
 *  - Buffers are caller-owned, contiguous, little-endian.  Functions without a
 *    `_dev` suffix take HOST pointers (pinned memory gives full PCIe speed),
 *    copy in, run on the GPU and copy out before returning.  `_dev` functions
 *    take DEVICE pointers on the current device and run asynchronously on the
 *    engine's stream (d377_stream()); call d377_sync() before reading results.
 *  - Fq on the wire:
 *      "canonical" = 32-byte LE integer < q        (Fq::to_bytes, fields/fq.rs:117)
 *      "montgomery"= 32-byte LE of x*2^256 mod q   (the in-memory form of both
 *                    reference backends, fields/fq/u32/wrapper.rs:93-104)
 *  - Element on the wire: X||Y||Z||T, 4 x 32-byte montgomery Fq = 128 bytes
 *    (ark_curve/element/projective.rs:13-16; min_curve/element.rs:31-38).
 *    The projective representative is NOT unique; compare via encodings or
 *    d377_batch_element_eq.
 *  - Encoding: 32 bytes (ark_curve/encoding.rs:14-15).
 *  - Fr scalars: canonical 32-byte LE integers < r (fields/fr.rs:117).
 *  - Return value: 0 on success, a negative D377_ERR_* otherwise.  Per-element
 *    decode failures (EncodingError::InvalidEncoding, src/error.rs:2-5) never
 *    abort a batch: they are reported in the `ok` byte array (1 = Ok, 0 = Err)
 *    and the corresponding output element is the identity.
 *  - There is NO CPU fallback: every function fails with D377_ERR_CUDA /
 *    D377_ERR_NOT_INITIALISED when no usable GPU is present.
 *  - Devices and threads: the library keeps one engine (streams, workspaces, tables) per
 *    CUDA device it has been initialised for.  Every entry point may be called from any
 *    host thread: it locks the engine it acts on and makes that engine's device current
 *    for the duration of the call (the caller's current device is restored on return).
 *    The engine a call acts on is the one the calling thread selected with
 *    d377_set_device, else the one the most recent d377_init / d377_init_multi chose.
 *    Calls on one engine are serialised; calls on different engines run concurrently.
 *  - Untrusted limbs: montgomery inputs are expected canonical (< q), which is all the
 *    reference can produce, but any 256-bit string is accepted and read as an integer
 *    mod q (it is brought below 2q on load); nothing overflows or hangs on bad bytes.
 */
#ifndef DECAF377_B200_H
#define DECAF377_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define D377_OK 0
#define D377_ERR_INVALID_ARG (-1)
#define D377_ERR_CUDA (-2)
#define D377_ERR_NOT_INITIALISED (-3)
#define D377_ERR_SCALAR_RANGE (-4) /* a scalar was not < r (Fr::from_bytes_checked, fr.rs:108) */
#define D377_ERR_INVALID_ENCODING (-5) /* MSM over encodings met an invalid encoding */

/* point input formats for d377_msm* and d377_batch_scalar_mul */
#define D377_PT_ELEMENT 0  /* 128 B  X||Y||Z||T montgomery */
#define D377_PT_ENCODING 1 /* 32 B   decaf377 Encoding */
#define D377_PT_AFFINE 2   /* 64 B   x||y montgomery, Z = 1 (AffinePoint, ark_curve/element/affine.rs) */
#define D377_PT_XYZ 3      /* 96 B   X||Y||Z montgomery: an Element without its redundant T = XY/Z.
                            * d377_msm* only.  The Rust shim copies the coordinates of an
                            * Element one by one anyway (Projective is not repr(C)); leaving T
                            * out moves 128 instead of 160 bytes per (scalar, point) pair over
                            * PCIe, which is the bound of a host-buffer MSM. */
#define D377_PT_BASES 4    /* prepared bases: `points` is the DEVICE pointer d377_msm_bases_create
                            * (128 B per base) or d377_msm_bases_create_windowed returned.  d377_msm* only, host-buffer entry points
                            * included: only the scalars cross the link. */

/* Scalars as the reference keeps them in memory.  `Fr` is stored in Montgomery form
 * (fields/fr/u64/wrapper.rs, fr/u32/wrapper.rs: x * 2^256 mod r), and Fr::to_bytes /
 * into_bigint costs a Montgomery reduction per scalar on the host -- more host time for
 * 2^24 scalars than the whole MSM takes on the GPU.  OR this flag into `point_format`
 * (d377_msm*, d377_batch_scalar_mul*) or into `out_format` (d377_fixed_base_mul*,
 * d377_fixed_bases_mul*) and pass the 32 bytes of the in-memory limbs instead: the
 * conversion (Fr::into_bigint, fields/fr/arkworks.rs:36-57) then runs on the GPU.  Every 256-bit string is a valid
 * Montgomery representative, so D377_ERR_SCALAR_RANGE cannot occur with it. */
#define D377_SCALARS_MONTGOMERY 0x100

/* output formats */
#define D377_OUT_ELEMENT 0  /* 128 B */
#define D377_OUT_ENCODING 1 /* 32 B, i.e. fused vartime_compress */

/* ---- life cycle -------------------------------------------------------- */

/* Create the engine of CUDA device `device` (streams, small buffers; the constant tables
 * -- the reference's lazily built SquareRootTables, ark_curve/invsqrt.rs:66 -- are part of
 * the module image) and make it the process default.  Idempotent; engines of other devices
 * stay alive. */
int d377_init(int device);
/* The same for `ndev` (1..8) distinct devices at once; devices[0] becomes the default and
 * the gathering device of d377_msm_multi*.  Enables peer access between them where the
 * hardware allows (NVLink / NVSwitch on a B200 box). */
int d377_init_multi(const int* devices, int ndev);
/* Select, for the CALLING THREAD, the initialised device later calls act on
 * (device < 0: back to the process default). */
int d377_set_device(int device);
/* Device the calling thread's calls act on, -1 if none is initialised. */
int d377_get_device(void);
/* Initialised devices in initialisation order; returns their number (devices may be NULL). */
int d377_device_list(int* devices, int cap);
/* Release every engine. */
int d377_shutdown(void);
/* Engine stream as a cudaStream_t, for callers that enqueue their own work. */
void* d377_stream(void);
/* Stream on which the results of asynchronous MSMs (d377_msm_dev_async, d377_msm_submit)
 * become complete: the tail of a Pippenger (stitching, bucket reduction, Horner, compress)
 * runs on a stream of its own so that the next MSM's head can start under it.  Work a
 * caller enqueues there (e.g. an all-gather of partial sums) is ordered after those
 * results without stalling the engine stream; every other entry point, d377_join and
 * d377_sync order the engine stream behind it again. */
void* d377_result_stream(void);
/* Order the engine stream behind everything enqueued so far (no host synchronisation). */
int d377_join(void);
/* Wait for the engine stream (after a join).  Reports the status of the asynchronous MSMs
 * enqueued since the last d377_sync (D377_ERR_SCALAR_RANGE / D377_ERR_INVALID_ENCODING). */
int d377_sync(void);
/* Human-readable description of the last error on this thread's last call. */
const char* d377_last_error(void);
/* Page-locked host memory for the host-pointer entry points: with pinned input and
 * output buffers the chunks of a batch overlap upload, kernel and download, and
 * PCIe runs at full speed; pageable buffers work but are staged by the driver.
 * d377_host_alloc returns NULL on failure (see d377_last_error). */
void* d377_host_alloc(size_t bytes);
int d377_host_free(void* p);
/* Number of kernels this library has launched since d377_init (for bench.py's
 * gpu_launches accounting). */
uint64_t d377_launch_count(void);

/* ---- Encoding::vartime_decompress (ark_curve/encoding.rs:32-83) -------- */
int d377_batch_decompress(const uint8_t* enc, size_t n, uint8_t* elements, uint8_t* ok);
int d377_batch_decompress_dev(const uint8_t* enc, size_t n, uint8_t* elements, uint8_t* ok);

/* ---- Element::vartime_compress (ark_curve/encoding.rs:116-128) --------- */
int d377_batch_compress(const uint8_t* elements, size_t n, uint8_t* enc);
int d377_batch_compress_dev(const uint8_t* elements, size_t n, uint8_t* enc);

/* ---- The same two calls over the other point layouts --------------------
 * CanonicalSerialize / CanonicalDeserialize for AffinePoint (ark_curve/serialize.rs:8-46:
 * serialize = AffinePoint -> Element -> vartime_compress; deserialize = Encoding ->
 * vartime_decompress -> Element -> AffinePoint), without the 128-byte detour:
 *   d377_batch_decompress_fmt: out_format D377_PT_ELEMENT (128 B, == d377_batch_decompress)
 *     or D377_PT_AFFINE (64 B x||y montgomery; decompression yields Z = 1, so these are the
 *     first two coordinates of the Element form; rejected encodings give the identity (0, 1)
 *     and ok[i] = 0).
 *   d377_batch_compress_fmt: point_format D377_PT_ELEMENT, D377_PT_AFFINE (Z = 1, T = xy) or
 *     D377_PT_XYZ (96 B, T implied: the representative (XZ : YZ : Z^2 : XY) is compressed,
 *     same encoding since the encoding depends on the point only). */
int d377_batch_decompress_fmt(const uint8_t* enc, size_t n, int out_format, uint8_t* out,
                              uint8_t* ok);
int d377_batch_decompress_fmt_dev(const uint8_t* enc, size_t n, int out_format, uint8_t* out,
                                  uint8_t* ok);
int d377_batch_compress_fmt(const uint8_t* points, int point_format, size_t n, uint8_t* enc);
int d377_batch_compress_fmt_dev(const uint8_t* points, int point_format, size_t n, uint8_t* enc);

/* ---- Element::encode_to_curve (ark_curve/elligator.rs:74-76) ------------
 * r: n x 32 bytes, each reduced mod q exactly like
 * Fq::from_le_bytes_mod_order(&bytes[..32]) (fields/fq.rs:90-102), as the
 * reference's own tests feed it (tests/operations.rs:6-11).
 * With D377_OUT_ENCODING the 32 bytes are those of
 * encode_to_curve(r).vartime_compress(), computed without the second inverse
 * square root (the encoding is read off the Jacobi-quartic pair of the map). */
int d377_batch_encode_to_curve(const uint8_t* r, size_t n, uint8_t* out, int out_format);
int d377_batch_encode_to_curve_dev(const uint8_t* r, size_t n, uint8_t* out, int out_format);
/* Same with `in_width` (1..256) bytes per input, reduced exactly like
 * Fq::from_le_bytes_mod_order(&bytes[..in_width]) for ANY length (fields/fq.rs:90-102:
 * 32-byte little-endian chunks, the last one zero-padded, folded from the most significant
 * chunk down with 2^256 mod q; the reference's own property test feeds 80 bytes,
 * fields/fq/arkworks.rs:586-593).  64 bytes is the usual hash-output input. */
int d377_batch_encode_to_curve_wide(const uint8_t* r, size_t in_width, size_t n, uint8_t* out,
                                    int out_format);
int d377_batch_encode_to_curve_wide_dev(const uint8_t* r, size_t in_width, size_t n, uint8_t* out,
                                        int out_format);

/* ---- Element::hash_to_curve (ark_curve/elligator.rs:67-71) ------------- */
int d377_batch_hash_to_curve(const uint8_t* r1, const uint8_t* r2, size_t n, uint8_t* out,
                             int out_format);
int d377_batch_hash_to_curve_dev(const uint8_t* r1, const uint8_t* r2, size_t n, uint8_t* out,
                                 int out_format);
int d377_batch_hash_to_curve_wide(const uint8_t* r1, const uint8_t* r2, size_t in_width, size_t n,
                                  uint8_t* out, int out_format);
int d377_batch_hash_to_curve_wide_dev(const uint8_t* r1, const uint8_t* r2, size_t in_width, size_t n,
                                      uint8_t* out, int out_format);

/* ---- &Element * &Fr (ark_curve/ops/projective.rs:106-191) --------------
 * out[i] = scalars[i] * points[i].  With D377_PT_ENCODING inputs, `ok` (may be
 * NULL) receives the decode status; an invalid encoding yields the identity. */
int d377_batch_scalar_mul(const uint8_t* points, int point_format, const uint8_t* scalars,
                          size_t n, uint8_t* out, int out_format, uint8_t* ok);
int d377_batch_scalar_mul_dev(const uint8_t* points, int point_format, const uint8_t* scalars,
                              size_t n, uint8_t* out, int out_format, uint8_t* ok);

/* ---- Element::GENERATOR * s (ark_curve/element/projective.rs:20-22) ----
 * Fixed-base multiplication with precomputed window tables (built on the GPU
 * on first use; the reference has none).  scalars: n x 32 bytes, ANY 256-bit
 * little-endian integer (a canonical Fr in the reference).  D377_OUT_ELEMENT uses
 * a 48 MiB table of Edwards multiples (built on first use, ~5 ms; that call blocks);
 * D377_OUT_ENCODING = the bytes of (GENERATOR * s).vartime_compress(): batches of at least
 * 2^18 scalars compute them on the Jacobi quartic over a second table (1.6 GB of device
 * memory, built in ~0.15 s by the first such call and used by every call after it);
 * smaller batches take the Edwards table + compress.  Both paths give the same bytes. */
int d377_fixed_base_mul(const uint8_t* scalars, size_t n, uint8_t* out, int out_format);
int d377_fixed_base_mul_dev(const uint8_t* scalars, size_t n, uint8_t* out, int out_format);

/* ---- fixed-base multiplication over caller-chosen bases --------------------
 * Prepared fixed bases: window tables of k caller-chosen points B_0..B_{k-1}, the geometry
 * of the generator table (16 signed 16-bit windows, 2^15 cached affine multiples each, plus
 * the 2^256 * B_j carry entry): (16 * 2^15 + 1) * 96 B = 48 MiB per base.  points: k inputs in
 * point_format 0..3 (host memory; device memory for _dev).  An invalid encoding fails with
 * D377_ERR_INVALID_ENCODING.  A table that cannot be allocated fails with D377_ERR_CUDA and
 * d377_last_error names the byte count before any input is read; k = 0, a null pointer, a
 * bad format and a k whose byte count overflows give D377_ERR_INVALID_ARG.  No failure leaves
 * anything registered.  The handle is a device pointer owned by the library until
 * d377_fixed_bases_destroy or d377_shutdown, and it is valid on the device it was created on
 * (it is NOT a D377_PT_BASES handle of d377_msm*).  The creating call blocks. */
int d377_fixed_bases_create(const uint8_t* points, int point_format, size_t k, uint8_t** tables);
int d377_fixed_bases_create_dev(const uint8_t* points, int point_format, size_t k, uint8_t** tables);
/* k and device bytes of a live handle */
int d377_fixed_bases_info(const uint8_t* tables, size_t* k, size_t* bytes);
/* a handle that is not live (destroyed, never created, of another device) is refused;
 * NULL is a no-op */
int d377_fixed_bases_destroy(uint8_t* tables);
/* out[i] = sum_j scalars[i*k + j] * B_j for i < n: n rows of k 32-byte scalars, each ANY
 * 256-bit LE integer (as d377_fixed_base_mul); OR D377_SCALARS_MONTGOMERY into out_format
 * for in-memory Fr limbs.  out: n x 128 B (D377_OUT_ELEMENT) or n x 32 B (D377_OUT_ENCODING).
 * Every call uses all k bases (a zero scalar adds the identity).  k = 1 is fixed-base
 * multiplication by an arbitrary point.  One accumulator walks the 16 windows of every base
 * in turn: 16 k mixed additions per row, plus one compress for encodings.  n = 0 is a no-op;
 * a handle that is not a live fixed-bases handle of the calling thread's engine is refused
 * with D377_ERR_INVALID_ARG. */
int d377_fixed_bases_mul(const uint8_t* tables, const uint8_t* scalars, size_t n, uint8_t* out, int out_format);
int d377_fixed_bases_mul_dev(const uint8_t* tables, const uint8_t* scalars, size_t n, uint8_t* out, int out_format);

/* ---- Element + Element, PartialEq (ark_curve/ops/projective.rs:5-104,
 *      element/projective.rs:65-70) ------------------------------------- */
int d377_batch_add(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out);
int d377_batch_add_dev(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out);
/* Sub (ops/projective.rs:50-87), Neg (:90-96: (X, Y, Z, T) -> (-X, Y, Z, -T)) and
 * doubling (the group law behind `+=` with itself, min_curve/element.rs:119-136). */
int d377_batch_sub(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out);
int d377_batch_sub_dev(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out);
int d377_batch_neg(const uint8_t* a, size_t n, uint8_t* out);
int d377_batch_neg_dev(const uint8_t* a, size_t n, uint8_t* out);
int d377_batch_double(const uint8_t* a, size_t n, uint8_t* out);
int d377_batch_double_dev(const uint8_t* a, size_t n, uint8_t* out);
int d377_batch_element_eq(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* eq);
int d377_batch_element_eq_dev(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* eq);
/* out = sum of n elements (Sum<Element>, element/projective.rs:131-140). */
int d377_element_sum(const uint8_t* elements, size_t n, uint8_t out_element[128],
                     uint8_t out_encoding[32]);
int d377_element_sum_dev(const uint8_t* elements, size_t n, uint8_t* out_element,
                         uint8_t* out_encoding);
/* Same, enqueued on the result stream (d377_result_stream): combines the partial sums of
 * asynchronous MSMs while the engine stream already runs the next MSM's head. */
int d377_element_sum_result_dev(const uint8_t* elements, size_t n, uint8_t* out_element,
                                uint8_t* out_encoding);
/* OnCurve::is_on_curve (ark_curve/on_curve.rs:17-38): ok[i] = 1 iff element i satisfies the
 * curve equation, T Z = X Y and Z != 0 and -- when check_order != 0 -- [2r]P is the
 * identity (one scalar multiplication per element). */
int d377_batch_on_curve(const uint8_t* elements, size_t n, int check_order, uint8_t* ok);
int d377_batch_on_curve_dev(const uint8_t* elements, size_t n, int check_order, uint8_t* ok);

/* ---- many independent small MSMs in one call ------------------------------------
 * Element::vartime_multiscalar_mul (element/projective.rs:99-117) called in a loop, e.g. a
 * batch of verification equations: MSM j is the sum over i in [offsets[j], offsets[j+1])
 * of scalars[i] * points[i]; offsets has nmsm + 1 non-decreasing entries starting at 0
 * (empty segments give the identity).  Every pair goes through the signed-window ladder of
 * d377_batch_scalar_mul and the products of a segment are added by one warp -- no Pippenger,
 * so the cost is per pair (~18 M pairs/s on a B200) whatever the grouping; a single MSM
 * above a few thousand pairs is better served by d377_msm.  point_format 0..2 (optionally
 * | D377_SCALARS_MONTGOMERY); scalars are read as 256-bit integers (k and k mod r give the
 * same element).  out: nmsm x 128 B or 32 B.  ok (may be NULL): ok[j] = 0 iff segment j
 * contains an invalid encoding (that pair then counts as the identity).  The _dev twin takes
 * device pointers (offsets included) and the total number of pairs n = offsets[nmsm]. */
int d377_batch_msm(const uint8_t* scalars, const uint8_t* points, int point_format,
                   const uint32_t* offsets, size_t nmsm, uint8_t* out, int out_format, uint8_t* ok);
int d377_batch_msm_dev(const uint8_t* scalars, const uint8_t* points, int point_format,
                       const uint32_t* offsets, size_t nmsm, size_t n, uint8_t* out, int out_format,
                       uint8_t* ok);

/* ---- many independent MSMs in one segmented Pippenger ----------------------------------
 * The results and contract of d377_batch_msm (MSM j = sum over i in [offsets[j], offsets[j+1])
 * of scalars[i] * points[i]; an empty segment gives the identity; scalars are any 256-bit LE
 * integers, optionally | D377_SCALARS_MONTGOMERY on point_format; out: nmsm x 128 B canonical
 * Elements or nmsm x 32 B encodings; ok (may be NULL): ok[j] = 0 iff segment j holds an
 * invalid encoding, which counts as the identity), computed by one Pippenger over all
 * segments: segment j's window w is bucket set j*W + w of one flat bucket space, so sort,
 * accumulation and bucket reduction are shared, and each segment ends in its own Horner.
 * point_format 0..3 (D377_PT_BASES is refused).  The cost is per pair and window plus per
 * bucket (2^(c-1) per segment and window), not a ladder per pair.
 * Measured on one B200 (1000 W power limit), device resident, back to back, 2^22 pairs: faster
 * than d377_batch_msm at every segment length measured, from 64 pairs (3.1x) to 65 536 (11x),
 * and faster than one d377_msm_dev_async per segment at every length up to 65 536 pairs (4.2x
 * there, 62x at 1 024); DESIGN.md 3.4.1 has the table.
 * `offsets` is HOST memory for BOTH forms: the library validates it (offsets[0] = 0,
 * non-decreasing, offsets[nmsm] <= 0xfffffff0), chooses the window width c (4..16;
 * d377_msm_set_window applies) and cuts the segments into chunks whose bucket sums stay under
 * 1 GiB before anything is launched, and copies it up itself (the array may be reused when
 * the call returns).  A segment too long for one chunk at the width is refused with
 * D377_ERR_INVALID_ARG.  _dev takes device scalars, points, out and ok and only enqueues on
 * the engine stream (d377_stream()), behind every earlier call; the outputs are complete there.
 * Refusals leave out / ok untouched; nmsm = 0 is a no-op. */
int d377_msm_segmented(const uint8_t* scalars, const uint8_t* points, int point_format,
                       const uint32_t* offsets, size_t nmsm, uint8_t* out, int out_format, uint8_t* ok);
int d377_msm_segmented_dev(const uint8_t* scalars, const uint8_t* points, int point_format,
                           const uint32_t* offsets /* HOST */, size_t nmsm, uint8_t* out, int out_format,
                           uint8_t* ok);
/* c, W = ceil(257 / c) and the number of segment chunks of the most recent d377_msm_segmented*
 * call of this engine (any pointer may be NULL); D377_ERR_INVALID_ARG before the first. */
int d377_msm_segmented_last(int* c, int* windows, size_t* chunks);

/* ---- CurveGroup::normalize_batch / ScalarMul::batch_convert_to_mul_base
 *      (ark_curve/element.rs:27-34,74-81) ----------------------------------
 * Element (128 B) -> AffinePoint x||y (64 B montgomery, x = X/Z, y = Y/Z), one field
 * inversion per up to 64 elements (Montgomery's trick).  The output is the
 * D377_PT_AFFINE input format of d377_msm / d377_batch_scalar_mul. */
int d377_batch_normalize(const uint8_t* elements, size_t n, uint8_t* affine);
int d377_batch_normalize_dev(const uint8_t* elements, size_t n, uint8_t* affine);

/* ---- Element::vartime_multiscalar_mul (element/projective.rs:99-117) and
 *      <Element as VariableBaseMSM>::msm (ark_curve/element.rs:37) --------
 * Q = sum_i scalars[i] * points[i] by a signed-digit Pippenger.  n = 0 yields
 * the identity (Element::default()).  Either output pointer may be NULL.
 * For a multi-GPU MSM each rank calls this on its slice with
 * out_encoding = NULL and the 128-byte partial sums are combined with
 * d377_element_sum after an all-gather (see decaf377_b200/dist.py). */
int d377_msm(const uint8_t* scalars, const uint8_t* points, int point_format, size_t n,
             uint8_t out_element[128], uint8_t out_encoding[32]);
int d377_msm_dev(const uint8_t* scalars, const uint8_t* points, int point_format, size_t n,
                 uint8_t* out_element, uint8_t* out_encoding);
/* d377_msm_dev without the host synchronisation: the MSM is only enqueued, its outputs are
 * complete on d377_result_stream() (and on the engine stream after d377_join / any later
 * call), and a non-canonical scalar or invalid encoding is reported by the next d377_sync.
 * Back-to-back calls overlap the latency-bound tail of one MSM with the head of the next. */
#define D377_MSM_INPUTS_READY 1 /* the scalar and point buffers are complete when the call is
                                 * made (not still being produced by work queued on
                                 * d377_stream()): the scalar side of this MSM -- digit
                                 * recoding and counting sort -- may then start under the
                                 * previous MSM's bucket accumulation */
int d377_msm_dev_async(const uint8_t* scalars, const uint8_t* points, int point_format, size_t n,
                       uint8_t* out_element, uint8_t* out_encoding, int flags);
/* ---- one MSM over several GPUs of this process (SURVEY 8e) ------------------
 * The first `ngpu` devices of d377_init_multi each run a complete Pippenger over a
 * contiguous slice of the pairs (sizes differ by at most one); the last kernel of each
 * stores its 128-byte partial sum straight into the first device's memory (a peer store
 * over NVLink; cudaMemcpyPeerAsync without peer access), where the partial sums are
 * added and compressed.  One persistent host thread per device enqueues its slice, so the
 * GPUs start together.  d377_msm_multi takes HOST buffers (pinned memory from
 * d377_host_alloc is usable by every device); d377_msm_multi_dev takes, per device, DEVICE
 * pointers to that device's slice and its length.  point_format 0..3; results in host
 * memory; blocks until done.  The multi-process form (one process per GPU, NCCL
 * all-gather of the partial sums) is decaf377_b200/dist.py. */
int d377_msm_multi(const uint8_t* scalars, const uint8_t* points, int point_format, size_t n,
                   int ngpu, uint8_t out_element[128], uint8_t out_encoding[32]);
int d377_msm_multi_dev(const uint8_t* const* scalars, const uint8_t* const* points,
                       int point_format, const size_t* n, int ngpu, uint8_t out_element[128],
                       uint8_t out_encoding[32]);
/* Asynchronous form of d377_msm_multi_dev: only enqueues (up to four calls may be in flight
 * without any waiting on the device side), so consecutive MSMs overlap on every GPU the way
 * d377_msm_dev_async calls do on one.  out_element / out_encoding are DEVICE pointers on the
 * first device (either may be NULL), complete on that device's result stream
 * (d377_result_stream with the first device selected) and after d377_multi_sync, which waits
 * for every initialised device and reports the sticky status of every leg. */
int d377_msm_multi_dev_async(const uint8_t* const* scalars, const uint8_t* const* points,
                             int point_format, const size_t* n, int ngpu,
                             uint8_t* out_element_dev, uint8_t* out_encoding_dev);
int d377_multi_sync(void);
/* Pipelined form of d377_msm for back-to-back MSMs over host buffers: submit copies the
 * inputs up on a copy stream and enqueues the MSM behind them without blocking, so the
 * transfer of one MSM overlaps the computation of the previous ones.  Four slots (0..3)
 * may be in flight (two keep a link-bound stream of large MSMs busy; small MSMs, whose
 * result arrives a tail after their bucket accumulation, need three); the host buffers
 * (pinned memory for full PCIe speed) must stay valid until d377_msm_wait(slot, ...)
 * returns the result (and the error status). */
int d377_msm_submit(const uint8_t* scalars, const uint8_t* points, int point_format, size_t n,
                    int slot);
int d377_msm_wait(int slot, uint8_t out_element[128], uint8_t out_encoding[32]);
/* Override the Pippenger window width c (0 = choose from n; otherwise 4..22).  MSMs over
 * windowed bases (d377_msm_bases_create_windowed) always use the width of the set. */
int d377_msm_set_window(int c);
/* 1 (default): run MSM tails on the result stream, overlapped with the next MSM's head;
 * 0: everything on the engine stream (A/B measurements). */
int d377_msm_set_tail_overlap(int on);
/* Host-buffer MSMs (d377_msm, d377_msm_submit) are cut into k sub-MSMs so that the
 * upload of one overlaps the Pippenger of the previous one; 0 = choose from n
 * (1 below 2^22 pairs, up to 4 above), k <= 8. */
int d377_msm_set_host_chunks(int k);
/* Device time (ms, CUDA events) of the stages of the most recent single-chunk MSM:
 * points, count, scan, scatter, accumulate, stitch, bucket_reduce, tail; plus the
 * geometry it ran with.  The scalar side runs on its own stream, overlapped with
 * `points` and `accumulate`: its whole span is reported as `count` (scan = scatter = 0),
 * and `accumulate` is the engine-stream span from the first to the last accumulation
 * launch (it includes any wait for a sorted list). */
/* ---- long-lived MSM bases ------------------------------------------------
 * ScalarMul::batch_convert_to_mul_base once (ark_curve/element.rs:27-34), then
 * VariableBaseMSM::msm(&bases, &scalars) many times (element.rs:37): the bases are uploaded
 * and converted to the 128-byte bucket operands of the Pippenger kernels ONCE; every later
 * d377_msm / d377_msm_submit / d377_msm_dev call with D377_PT_BASES moves only the 32-byte
 * scalars and skips the normalisation.  `points`: n inputs in `point_format` (any of 0..3),
 * host memory for d377_msm_bases_create, device memory for the _dev twin.  *bases receives
 * a device pointer owned by the library until d377_msm_bases_destroy (or d377_shutdown,
 * which releases every set still alive); the library keeps a registry of live sets and an
 * MSM with D377_PT_BASES is refused unless `points` is such a pointer of the same device
 * and n' <= n (any prefix may be used).  Invalid encodings among the bases make the call
 * fail with D377_ERR_INVALID_ENCODING. */
int d377_msm_bases_create(const uint8_t* points, int point_format, size_t n, uint8_t** bases);
int d377_msm_bases_create_dev(const uint8_t* points, int point_format, size_t n, uint8_t** bases);
/* Prepared bases with precomputed window multiples: the table holds 2^(c*j) * P_i for
 * j = 0 .. W-1, W = ceil(252 / c), 128 B per entry (n * W * 128 B of device memory), laid out
 * window-major (entry (i, j) is record j*n + i).  Every MSM over such a set adds all its
 * windows into ONE set of 2^(c-1) buckets per window group and has no Horner tail.
 * c = 0: chosen from n; otherwise 4 <= c <= 22.  The handle is used exactly like the one
 * d377_msm_bases_create returns: d377_msm* with D377_PT_BASES, any prefix n' <= n,
 * d377_msm_bases_destroy, released by d377_shutdown.  The MSM always uses the set's c
 * (d377_msm_set_window does not apply), so a small prefix of a large set still pays for
 * the reduction of the large set's 2^(c-1) buckets.
 * Refused with D377_ERR_INVALID_ARG before anything is allocated or read: c outside [4, 22]
 * (other than 0) and n * W >= 2^31.  If the table cannot be allocated the call returns
 * D377_ERR_CUDA and d377_last_error names the byte count.  Invalid encodings among the
 * bases give D377_ERR_INVALID_ENCODING.
 * Measured on one B200 (1000 W; DESIGN.md 3.5): creation ~0.45 s for 2^24 bases at c = 21
 * (27 ms for 2^20), 1536 B of device memory per base at c = 21 (W = 12); per MSM against a
 * plain set, back to back 23.6 against 25.2 ms at 2^24, blocking 0.72 against 1.12 ms at 2^16. */
int d377_msm_bases_create_windowed(const uint8_t* points, int point_format, size_t n, int c, uint8_t** bases);
int d377_msm_bases_create_windowed_dev(const uint8_t* points, int point_format, size_t n, int c, uint8_t** bases);
/* n, c, W and device bytes of a live handle (W = 1 and c = 0 for a plain prepared set) */
int d377_msm_bases_info(const uint8_t* bases, size_t* n, int* c, int* windows, size_t* bytes);
/* *windowed = 1 if the most recent single-chunk MSM ran over a windowed set of bases */
int d377_msm_last_windowed(int* windowed);
int d377_msm_bases_destroy(uint8_t* bases);
int d377_msm_stage_info(float ms[8], int* c, int* W, uint64_t* n);
/* Timeline of the most recent single-chunk MSM, four floats per window group in the order
 * the groups were processed (highest windows first), in ms after the MSM's start: sorted
 * list ready (sort stream), accumulation start, accumulation end (engine stream), tail end
 * (tail stream: stitch, bucket reduction, Horner step).  cap = floats available in ms. */
int d377_msm_timeline(float* ms, int cap, int* ngroups);
/* *mixed = 1 if the bucket additions of the most recent MSM were mixed additions against
 * affine points (7 multiplications: affine / encoding inputs, or Element inputs that were
 * batch-normalised first), 0 if they were projective cached additions (8). */
int d377_msm_last_mode(int* mixed);
/* Element inputs of an MSM are batch-normalised to affine first (so that the bucket
 * additions are mixed) when the batch is large enough for that to pay: 0 = decide from n
 * (default), 1 = always, -1 = never.  Affine / encoding inputs are always mixed. */
int d377_msm_set_normalize(int mode);
/* The windows of an MSM are processed in groups: the scalar side (digit recoding,
 * histogram, counting sort) of group k+1 runs on a second stream while the bucket
 * additions of group k run on the engine stream.  0 = choose from n (1 group for small
 * MSMs, up to 4), otherwise the number of groups (<= 8, clamped to the window count). */
int d377_msm_set_groups(int groups);

/* ---- field-layer entry points (parity tests of rows a2-a5) -------------
 * op: 0 mul, 1 square(a), 2 add, 3 sub, 4 neg(a), 5 to_montgomery(a),
 *     6 from_montgomery(a), 7 from_le_bytes_mod_order(a) -> montgomery,
 *     8 inverse(a) by the binary extended Euclid, 9 inverse(a) by Fermat (0 -> 0),
 *     10 a * 6042, 11 a * 12086 (the small-constant product of the curve formulas).
 * a, b, out: n x 32-byte montgomery Fq (ops 5/7 take raw bytes, 6 returns
 * canonical bytes).  Replaces fields/fq/u32/fiat.rs:162,1360,2555,2646,2725,
 * 2800,3584 and fields/fq.rs:90-102. */
int d377_fq_batch_op(int op, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out);
/* Fq::from_le_bytes_mod_order for inputs of any length (fields/fq.rs:90-102; property
 * fields/fq/arkworks.rs:586-593): n x in_width bytes (1..256) -> n x 32 montgomery. */
int d377_fq_batch_from_le_bytes_mod_order(const uint8_t* bytes, size_t in_width, size_t n,
                                          uint8_t* out);
int d377_fq_batch_from_le_bytes_mod_order_dev(const uint8_t* bytes, size_t in_width, size_t n,
                                              uint8_t* out);
/* Fq::sqrt_ratio_zeta(&ONE, &x) (ark_curve/invsqrt.rs:75-166): x, out montgomery;
 * was_square[i] in {0,1}.  Returns the same root as the reference. */
int d377_fq_batch_isqrt(const uint8_t* x, size_t n, uint8_t* out, uint8_t* was_square);
int d377_fq_batch_isqrt_dev(const uint8_t* x, size_t n, uint8_t* out, uint8_t* was_square);
/* Fq::sqrt_ratio_zeta(&num, &den) for a general ratio (ark_curve/invsqrt.rs:69-166;
 * benches/sqrt.rs:41-52; the R1CS witness of r1cs/fqvar_ext.rs:29-36): num, den, out
 * montgomery.  (1, sqrt(num/den)) | (1, 0) if num = 0 | (0, 0) if den = 0 |
 * (0, sqrt(zeta*num/den)); computed step by step as the reference does, so the root
 * returned is the reference's. */
int d377_fq_batch_sqrt_ratio_zeta(const uint8_t* num, const uint8_t* den, size_t n, uint8_t* out,
                                  uint8_t* was_square);
int d377_fq_batch_sqrt_ratio_zeta_dev(const uint8_t* num, const uint8_t* den, size_t n,
                                      uint8_t* out, uint8_t* was_square);
/* CanonicalDeserialize for field elements (fields/fq/arkworks.rs:189-229,
 * fields/fr/arkworks.rs, Fq::from_bytes_checked fields/fq.rs:108): n x 32 canonical LE
 * bytes; ok[i] = 0 when the value is >= the modulus (SerializationError::InvalidData).
 * field 0 = Fq: out (may be NULL) receives the montgomery form; field 1 = Fr: out (may be
 * NULL) receives the canonical bytes unchanged (scalars stay canonical on this ABI).
 * Rejected entries are written as zero.  CanonicalSerialize for Fq is
 * d377_fq_batch_op(6, ...); for Element / Encoding it is d377_batch_compress and
 * CanonicalDeserialize is d377_batch_decompress (ark_curve/encoding.rs:143-176,253-292);
 * for AffinePoint they are d377_batch_compress_fmt / d377_batch_decompress_fmt with
 * D377_PT_AFFINE (ark_curve/serialize.rs:8-46). */
int d377_field_batch_deserialize(int field, const uint8_t* bytes, size_t n, uint8_t* out,
                                 uint8_t* ok);
int d377_field_batch_deserialize_dev(int field, const uint8_t* bytes, size_t n, uint8_t* out,
                                     uint8_t* ok);
/* Sustained IMAD.WIDE.U32 issue-rate microbenchmark used as the roofline
 * denominator: returns giga 32x32->64 multiply-adds per second. */
int d377_imad_peak(double* gimad_per_s);
/* Debug builds (libdecaf377_b200_dbg.so, compiled with -DD377_DEBUG_ON_CURVE
 * [-DD377_DEBUG_ORDER]) check every point the kernels produce -- decompress, Elligator,
 * scalar multiplication, fixed base, add / sub / neg / double, MSM result -- against
 * OnCurve::is_on_curve (ark_curve/on_curve.rs:17-38; the reference keeps that predicate
 * alive through debug assertions in CI).  d377_debug_build: 0 = release, 1 = curve
 * equation + Segre + Z != 0, 2 = also [2r]P = 0.  d377_debug_counts: points checked and
 * failures since the library was loaded (both 0 in a release build). */
int d377_debug_build(void);
int d377_debug_counts(uint64_t* failures, uint64_t* checked);

#ifdef __cplusplus
}
#endif
#endif
