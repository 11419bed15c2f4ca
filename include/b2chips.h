/*
 * b2chips.h — C ABI of libb2chips.so: the B200 (sm_100a) replacement for the native calls that
 * harry-gibson/dl_image_segmentation's hot path reaches through TensorFlow, rasterio/GDAL/libtiff,
 * libpng/zlib and numpy.ma.  The reference has no FFI of its own (it is pure Python,
 * dl_segmentation_utils/__init__.py:1-15); every entry point below therefore cites the reference
 * CALL SITE whose third-party native work it replaces.  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes.  Every function returns 0 on success, non-zero on misuse or
 *     CUDA failure; b2_last_error() then returns a thread-local message.
 *   - All *_dev pointers are device memory owned by the caller; the library allocates nothing but a
 *     per-context workspace.  Work is enqueued on `stream` (a cudaStream_t passed as void*); nothing
 *     synchronises the host unless stated.
 *   - Per-item failures (a corrupt chip, a bad CRC) are DATA: they come back in a status array, as the
 *     reference's skip-and-continue loop expects (_img_to_tf_mp.py:127-136).
 *   - One b2_ctx per (process, device), used by one host thread at a time (one writer per worker,
 *     _img_to_tf_mp.py:119).
 */
#ifndef B2CHIPS_H
#define B2CHIPS_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2_VERSION 100 /* 0.1.0 */

typedef struct b2_ctx b2_ctx;
typedef void* b2_stream; /* cudaStream_t */

/* element types (numpy names) */
enum { B2_U8 = 0, B2_U16 = 1, B2_I16 = 2, B2_U32 = 3, B2_I32 = 4, B2_F32 = 5, B2_F64 = 6, B2_I8 = 7 };

/* ------------------------------------------------------------------ context */
int b2_version(void);
const char* b2_last_error(void);
int b2_ctx_create(int device, b2_ctx** out);
int b2_ctx_destroy(b2_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
uint64_t b2_ctx_launch_count(const b2_ctx* ctx);
int b2_ctx_sm_count(const b2_ctx* ctx);

/* ------------------------------------------------------------------ K3: compositors
 * b2_median_composite_u16 replaces np.repeat + np.ma.masked_where + np.ma.median(axis=0)
 *   (_descartes_img_chips.py:562-567).  stack (T,H,W,B) u16 bands-innermost; valid (T,H,W) u8, 0 = masked;
 *   nodata (T,H,W,B) u8 or NULL, non-zero = masked (the pre-existing mask np.ma.masked_where ORs with).
 *   out (H,W,B) float64: middle value, or mean of the two middles; out_mask (H,W,B) u8 = 1 and out = 0.0
 *   where no scene is valid.
 */
int b2_median_composite_u16(b2_ctx* ctx, const uint16_t* stack_dev, const uint8_t* valid_dev,
                            const uint8_t* nodata_dev, int T, int H, int W, int B,
                            double* out_dev, uint8_t* out_mask_dev, b2_stream stream);

/* b2_nearest_date_mosaic replaces the filter + sort + SceneCollection.mosaic of create_img_array_for_tile
 *   (_descartes_img_chips.py:603-626, key function :461-469).  For each of n_chips chips:
 *   scene t is eligible iff min_day <= scene_day[t] < max_day and (max_cf is NaN or scene_cf[t] < max_cf);
 *   out pixel = stack[t*] with t* the eligible scene, valid at that pixel, of least |scene_day - ref_day|,
 *   ties to the HIGHER scene index (stable descending sort, painted last).  The distance is exact over the whole
 *   int32 range (up to 2^32 - 1).  min_day = INT32_MIN means no lower bound and max_day = INT32_MAX no upper bound:
 *   a scene dated INT32_MAX is then eligible.  stacks_dev / valids_dev: device arrays of n_chips device pointers to
 *   (T,H,W,B) and (T,H,W) u8; each stack aligned to its pixel size B * elem_bytes when that is 2, 4, 8 or 16.
 *   scene_day_dev / scene_cf_dev: (n_chips,T).  out (n_chips,H,W,B) same element type;
 *   out_mask (n_chips,H,W) u8 = 1 where no valid scene (out = 0); src_index (n_chips,H,W) int16 or NULL;
 *   n_eligible (n_chips) int32 or NULL — 0 means the reference returns None (:614-615).
 *   stats_acc (B,4) uint64 or NULL: the exact band statistics of b2_band_stats over the VALID output pixels are
 *   accumulated in the same pass (uint8 / uint16 chips of at most 4 bands), so configs[4]'s per-band mean / std cost
 *   no second read of the output.  The counters are those of b2_band_stats, split the same way.
 */
int b2_nearest_date_mosaic(b2_ctx* ctx, const void* const* stacks_dev, const uint8_t* const* valids_dev,
                           const int32_t* scene_day_dev, const float* scene_cf_dev,
                           int32_t ref_day, int32_t min_day, int32_t max_day, float max_cf,
                           int n_chips, int T, int H, int W, int B, int elem_bytes,
                           void* out_dev, uint8_t* out_mask_dev, int16_t* src_index_dev,
                           int32_t* n_eligible_dev, uint64_t* stats_acc_dev, b2_stream stream);

/* ------------------------------------------------------------------ K4: cast / normalise / one-hot / statistics
 * North-star row A17 (not in the reference; nearest analogue parse_tfrecords.ipynb cell 21).
 *   img (N,H,W,C) of img_dtype; label (N,H,W) of label_dtype (B2_U8 or B2_F32); mean/std (C) float32.
 *   img_out = (float(x) - mean[c]) / std[c]  (IEEE float32);  onehot_out (N,H,W,K) = label==k ? 1 : 0.
 *   Either output may be NULL.
 */
int b2_normalise_onehot(b2_ctx* ctx, const void* img_dev, int img_dtype, const void* label_dev, int label_dtype,
                        const float* mean_dev, const float* std_dev, uint64_t n_pixels, int C, int K,
                        float* img_out_dev, float* onehot_out_dev, b2_stream stream);

/* Exact integer per-band statistics over pixels with valid != 0 (valid NULL = all): acc (B,4) uint64 += { n, sum x,
 *   lo, hi } with sum x*x = lo + 2^16 * hi.  The kernels split partial sums of x*x (per CTA or per slot, not per pixel)
 *   into their low 16 bits and the rest, so lo and hi on their own depend on the launch: only lo + 2^16 * hi is
 *   defined.  dtype B2_U8 or B2_U16.  Accumulates (caller zeroes acc). */
int b2_band_stats(b2_ctx* ctx, const void* img_dev, int dtype, const uint8_t* valid_dev, uint64_t n_pixels, int B,
                  uint64_t* acc_dev, b2_stream stream);

/* ------------------------------------------------------------------ K2: TFRecord framing, CRC-32C, Example payloads
 * Replace tf.io.TFRecordWriter.write / TFRecordDataset (framing + masked CRC-32C), Example.SerializeToString,
 * tf.io.parse_single_example, tf.io.decode_raw and tf.reshape
 *   (_img_to_tf_mp.py:119,141; _tfrecord_image_translation.py:211,249,306-314,394-407; parse_tfrecords.ipynb cell 4).
 */

/* CRC-32C (unmasked) of n byte ranges of one device buffer. */
int b2_crc32c(b2_ctx* ctx, const uint8_t* data_dev, const uint64_t* offsets_dev, const uint64_t* lens_dev, int n,
              uint64_t max_len, uint32_t* crc_out_dev, b2_stream stream);

/* Walk the frames of one shard exactly as RecordReader does.  rec_offsets/rec_lens (capacity max_records) receive
 * the offset and length of each record's DATA.  result_dev[0] = number of records found, result_dev[1] = 0 ok,
 * 1 = corrupt/truncated frame or bad length-CRC at record result_dev[0], 2 = capacity exceeded.
 * shard_dev must be 16-byte aligned. */
int b2_tfrecord_scan(b2_ctx* ctx, const uint8_t* shard_dev, uint64_t nbytes, uint64_t max_records,
                     uint64_t* rec_offsets_dev, uint64_t* rec_lens_dev, int64_t* result_dev, b2_stream stream);

typedef struct {
    uint64_t img_off, img_len; /* payload of image/image_data, offset from shard start, length in bytes      */
    uint64_t tgt_off, tgt_len; /* payload of target/target_data                                              */
    uint64_t id_off, id_len;   /* identifier bytes                                                           */
    int32_t img_kind, tgt_kind; /* 1 = BytesList (one value), 2 = FloatList (packed float32), 0 = absent     */
    int32_t height, width, channels, tgt_height, tgt_width;
    int32_t status; /* 0 ok; 1 malformed protobuf; 2 required key missing / wrong type / not exactly one value */
} b2_example_index;

/* Locate the eight features of each Example (any key order, unknown fields skipped, last duplicate wins). */
int b2_tfrecord_index(b2_ctx* ctx, const uint8_t* shard_dev, const uint64_t* rec_offsets_dev,
                      const uint64_t* rec_lens_dev, int n, b2_example_index* index_out_dev, b2_stream stream);

/* ---- device-resident shard tables: open + parse with NO host round trip in between -------------------------------
 * b2_tfrecord_open = b2_tfrecord_scan + b2_tfrecord_index writing ONE caller-owned table (b2_tfrecord_table_bytes
 * bytes, 16-byte aligned) that b2_tfrecord_parse_table consumes directly, so a reader can enqueue
 * open -> parse for shard after shard (on alternating streams) and read the tables back once per batch.
 * Layout (b2_tfrecord_table_layout): offsets[0] hdr int64[8] = { records, scan status (as b2_tfrecord_scan),
 * tiles, longest record, records whose parse status != 0, .. }, [1] rec_offsets uint64[max_records],
 * [2] rec_lens uint64[max_records], [3] index b2_example_index[max_records], [4] tile_start uint32[max_records+1],
 * [5] tile2rec uint32[offsets[6]], offsets[7] = total bytes.  The rest of the table is scratch. */
uint64_t b2_tfrecord_table_bytes(uint64_t shard_nbytes, uint64_t max_records);
int b2_tfrecord_table_layout(uint64_t shard_nbytes, uint64_t max_records, uint64_t offsets[8]);
int b2_tfrecord_open(b2_ctx* ctx, const uint8_t* shard_dev, uint64_t shard_nbytes, uint64_t max_records,
                     uint8_t* table_dev, b2_stream stream);

enum { B2_SINK_NONE = 0, B2_SINK_RAW = 1, B2_SINK_NORM_ONEHOT = 2, B2_SINK_NORM_ONEHOT_F32 = 3, B2_SINK_STATS = 4,
       B2_SINK_STATS_F32 = 5 };
typedef struct {
    int32_t mode;        /* B2_SINK_NONE: CRC only.  RAW: payload bytes copied as stored (uint8 arrays; packed
                            little-endian float32 == float arrays).  NORM_ONEHOT: uint8 image -> normalised float32,
                            uint8 target -> one-hot float32 (K classes).  NORM_ONEHOT_F32: the same outputs from
                            packed float32 FloatList payloads (the higher-dtype array records): image ->
                            (x - mean[c]) / std[c] with IEEE float32 division, target -> one-hot where a label
                            equal to an integer k < K is class k (-0.0 is class 0; NaN, +-inf, negative,
                            non-integral and >= K labels give an all-zero row).
                            STATS (records as NORM_ONEHOT) and STATS_F32 (records as NORM_ONEHOT_F32): exact
                            per-band statistics of the images and a histogram of the labels, read in the same
                            pass as the CRC; nothing else is written.  channels = C (1..64); mean, std and
                            num_classes are not read.  img_out = uint64 acc[C][5] += { n, sum x (two's
                            complement int64), sum x^2 lo, sum x^2 hi, excluded } per band, with sum x^2 =
                            lo + 2^16 * hi: the kernel splits per-CTA partial sums, so only that sum is defined.
                            tgt_out = uint64 hist[257] += labels equal to v in bin v (0..255; -0.0 is 0), bin 256
                            for labels equal to no such integer (NaN, +-inf, negative, non-integral, > 255;
                            always 0 in STATS).  STATS_F32 counts an image value that is an integer in
                            [-2^16, 2^16) (u8, u16 and i16 sources); any other value goes to its band's
                            `excluded` and into no sum.  STATS excludes nothing.  Either output may be NULL
                            (skipped); both must be 8-byte aligned with img_stride = tgt_stride = 0.  The
                            counters ACCUMULATE (the caller zeroes them), also from several launches on
                            several streams.  A record with status 2 or 3 adds nothing, but a record's data
                            CRC is known only after its bytes were counted: the counters are defined only
                            when every record's status is 0 (check hdr[4] or the status array).             */
    int32_t verify_crc;  /* non-zero: compute each record's data CRC and compare with the stored masked CRC   */
    void* img_out;       /* record i lands at img_out + i*img_stride (bytes)                                  */
    uint64_t img_stride;
    void* tgt_out;
    uint64_t tgt_stride;
    const float* mean;   /* (channels) device, NORM_ONEHOT and NORM_ONEHOT_F32 only                           */
    const float* std;
    int32_t channels;
    int32_t num_classes;
} b2_parse_sink;

/* One fused pass over the records: CRC verify + payload scatter/cast.  status_dev[i]: 0 ok, 1 data-CRC mismatch
 * (TF: DataLossError), 2 index status != 0, 3 payload larger than its output stride (RAW).  The two normalise + one-hot
 * modes apply one rule with element width E (1 byte: NORM_ONEHOT, BytesList; 4 bytes: NORM_ONEHOT_F32, packed
 * FloatList, as parse_higher_dtype_array_proto followed by normalise and one-hot): 2 for a record that does not fit the
 * template (a payload that is not of the mode's kind, a BytesList record in NORM_ONEHOT_F32 included; image/channels != sink
 * channels; a negative dimension; image length != E*height*width*channels bytes or target length != E*target
 * height*width bytes), 3 for a payload whose floats do not fit its output row or of 2^31 elements or more (image
 * elements, or target elements * K).  Unpacked FloatList is status 2 from the index.  Uses the context workspace:
 * calls on one context must be stream-ordered (b2_tfrecord_parse_table has no such restriction). */
int b2_tfrecord_parse(b2_ctx* ctx, const uint8_t* shard_dev, uint64_t shard_nbytes, const uint64_t* rec_offsets_dev,
                      const uint64_t* rec_lens_dev, const b2_example_index* index_dev, int n,
                      uint64_t max_record_len, const b2_parse_sink* sink, int32_t* status_dev, b2_stream stream);

/* The same fused pass over every record of an opened shard; grid and record count come from the table on the
 * device.  status_dev needs max_records entries; entries >= hdr[0] are left untouched.  hdr[4] counts the records
 * whose status is non-zero.  A table may be parsed again (e.g. with another sink) without re-opening. */
int b2_tfrecord_parse_table(b2_ctx* ctx, const uint8_t* shard_dev, uint64_t shard_nbytes, uint64_t max_records,
                            uint8_t* table_dev, const b2_parse_sink* sink, int32_t* status_dev, b2_stream stream);

/* Host-side: the protobuf bytes around the two payloads for convert_to_example's eight keys in sorted
 * (deterministic) order (_tfrecord_image_translation.py:199-211).  kind 1 = BytesList, 2 = FloatList.
 * Writes three scaffold pieces (before image payload, between the payloads, after target payload) into
 * scaffold[cap]; returns total Example length in *example_len and piece lengths in piece_len[3]. */
int b2_example_layout(int kind, uint64_t img_payload_bytes, uint64_t tgt_payload_bytes,
                      int64_t img_h, int64_t img_w, int64_t img_c, int64_t tgt_h, int64_t tgt_w,
                      const uint8_t* identifier, uint64_t identifier_len,
                      uint8_t* scaffold, uint64_t cap, uint32_t piece_len[3], uint64_t* example_len);


typedef struct {
    uint64_t out_off;       /* where the framed record starts in out_dev                                      */
    uint64_t example_len;   /* length of the Example (frame adds 16)                                          */
    uint64_t scaffold_off;  /* offset of this record's three scaffold pieces (concatenated) in scaffold_dev  */
    uint32_t piece_len[3];
    int32_t src_dtype;      /* element type of img_src (B2_U8 .. B2_F32); B2_U8 also covers raw file bytes   */
    int32_t tgt_dtype;
    int32_t kind;           /* 1 BytesList (bytes copied), 2 FloatList (elements widened to float32)         */
    const void* img_src;    /* device */
    uint64_t img_count;     /* elements (bytes for kind 1)                                                    */
    const void* tgt_src;
    uint64_t tgt_count;
} b2_build_desc;

/* Serialise + frame n records: header (length + masked CRC), Example bytes, footer (masked data CRC). */
int b2_tfrecord_build(b2_ctx* ctx, const b2_build_desc* descs_dev, int n, uint64_t max_record_bytes,
                      const uint8_t* scaffold_dev, uint8_t* out_dev, b2_stream stream);

/* The same for n records in one call (the translators' worker loop, _img_to_tf_mp.py:123-141, per batch instead of per
 * chip): dims is n x {img_h, img_w, img_c, tgt_h, tgt_w}; identifiers are ids[id_off[i] .. id_off[i+1]).  Fills out_off
 * (records back to back from 0, 16 framing bytes each), example_len, scaffold_off, piece_len and kind of descs[i]; the
 * caller fills the payload sources.  scaffold needs 320 bytes + the identifier per record. */
int b2_example_layout_batch(int n, const int32_t* kind, const uint64_t* img_payload_bytes, const uint64_t* tgt_payload_bytes,
                            const int32_t* dims, const uint8_t* ids, const uint64_t* id_off, b2_build_desc* descs,
                            uint8_t* scaffold, uint64_t scaffold_cap, uint64_t* scaffold_len, uint64_t* total_bytes,
                            uint64_t* max_record);

/* ------------------------------------------------------------------ K1: chip decode (TIFF LZW / DEFLATE / none, PNG)
 * Replace rasterio MemoryFile(...).open().read() -> GDAL -> libtiff/libpng (_img_to_tf_mp.py:45-48,
 * _tfrecord_image_translation.py:320-326,369-381) and tf.image.decode_png / tf.io.decode_image
 * (_img_to_tf_threaded.py:59, _tfrecord_image_translation.py:283,289), including reshape_as_image
 * (_img_to_tf_mp.py:69): the output is written (H,W,bands) directly.
 */
typedef struct {
    int32_t format;      /* 1 TIFF, 2 PNG                                                                     */
    int32_t width, height, samples; /* what src.width / src.height / src.count return (_img_to_tf_mp.py:51-53) */
    int32_t dtype;       /* B2_U8 ...                                                                         */
    int32_t compression; /* TIFF tag 259 (1 none, 5 LZW, 8/32946 DEFLATE); 8 for PNG                          */
    int32_t predictor, planar, big_endian, tiled;
    int32_t block_w, block_h, blocks_across, blocks_down;
    int32_t n_blocks;    /* TIFF: tiles/strips (all planes); PNG: number of IDAT chunks                       */
    int32_t status;      /* 0 ok, 2 corrupt header, 3 flavour out of scope                                    */
    int32_t has_nodata, pad_;
    double nodata;       /* GDAL_NODATA tag 42113 (_descartes_img_chips.py:794-795)                           */
    uint64_t block_bytes; /* decoded bytes of one full block (PNG: h * (1 + row bytes) filtered bytes)          */
    /* what src.get_transform() / src.read_crs() return (_img_to_tf_mp.py:49-50), for identifiers built with
     * dltile_from_filename=False (:63-67): GDAL-order affine, default (0,1,0,0,0,1); EPSG code or 0               */
    double geotransform[6];
    int32_t has_geo, epsg;
    int32_t png_bit_depth, png_color_type; /* IHDR fields (0 for TIFF)                                          */
} b2_image_info;

/* How PNG flavours beyond 8-bit grey / RGB(A) are presented (flags of b2_image_probe / b2_decode_plan_batch).
 * The two reference paths disagree on them, so the caller says which one it replaces:
 *   B2_PNG_AS_TF   tf.image.decode_png(dtype=uint8) (_img_to_tf_threaded.py:59, _tfrecord_image_translation.py:283,289;
 *                  libpng transforms): palette -> RGB (RGBA with tRNS), 1/2/4-bit grey scaled to 0..255,
 *                  16-bit samples -> their high byte;
 *   0              rasterio / GDAL's PNG driver (_img_to_tf_mp.py:45-48): palette -> one band of indices,
 *                  1/2/4-bit grey unscaled, 16-bit samples -> uint16.
 * 8-bit grey, grey+alpha, RGB and RGBA are the same in both.  Adam7-interlaced files are decoded for bit depths 8 and
 * 16; interlaced 1/2/4-bit files are out of scope (status 3). */
#define B2_PNG_AS_TF 1u
/* b2_decode_plan_batch only: the blobs already lie inside the staging buffer (b2_read_files put them there 16-byte
 * aligned; the blobs of the records of a shard lie wherever the shard has them) — so nothing is gathered: the stream
 * table points at the files in place and the whole buffer is uploaded. */
#define B2_PLAN_INPLACE 0x1000u

/* Host-side header parse (TIFF IFD / PNG chunks); never touches the GPU. */
int b2_image_probe(const uint8_t* blob, uint64_t size, uint32_t flags, b2_image_info* info);
/* Host-side: offset / byte count / decoded length of each compressed block (TIFF) or IDAT payload (PNG). */
int b2_image_blocks(const uint8_t* blob, uint64_t size, const b2_image_info* info, uint64_t* offsets,
                    uint64_t* counts, uint64_t* decoded_len, int cap);

typedef struct {         /* one compressed stream = one warp of work                                          */
    uint64_t src_off;    /* offset in blob_dev                                                                */
    uint64_t dst_off;    /* offset in scratch_dev                                                             */
    uint32_t src_len;
    uint32_t dst_len;    /* bytes the stream must decode to                                                   */
    int32_t codec;       /* 1 stored, 5 LZW, 8 zlib                                                           */
    int32_t image;       /* owning image: failures are reported in status_dev[image]                          */
} b2_stream_desc;

typedef struct {         /* one image to assemble from its decoded blocks                                     */
    uint64_t scratch_off; /* first decoded block (blocks consecutive, block_bytes apart)                      */
    uint64_t out_off;    /* where the (H,W,samples) array starts in out_dev                                   */
    uint64_t block_bytes;
    int32_t format, width, height, samples, bytes_per_sample, predictor, planar, big_endian;
    int32_t block_w, block_h, blocks_across, blocks_down;
    int32_t png_bit_depth, png_color_type, png_flags, png_converted; /* PNG flavours that need the expand pass:   *
                           * scratch = filtered bytes | un-filtered bytes | 256-entry RGBA palette (16-byte aligned each) */
} b2_image_desc;

typedef struct {
    uint64_t stage_bytes;      /* host staging buffer needed for the compressed bytes                          */
    uint64_t scratch_bytes;    /* device scratch for the decoded blocks                                        */
    uint64_t out_bytes;        /* device buffer for the assembled (H,W,samples) arrays (256-byte aligned each) */
    uint64_t compressed_bytes;
    int32_t n_streams;
    uint32_t codec_mask;       /* for b2_decode_streams                                                        */
    uint32_t max_raw_len;
    int32_t filled;            /* 1: streams / images / stage were written; 0: sizes only (buffers too small)  */
} b2_decode_plan;

/* Host-side, multi-threaded: plan the decode of a whole batch of encoded chips in ONE call — b2_image_probe +
 * b2_image_blocks for every file, the stream and image descriptor tables, and the gather of all compressed bytes
 * into one (pinned) staging buffer.  Replaces the per-file open / header read inside the reference's worker loop
 * (_img_to_tf_mp.py:43-53, _img_to_tf_threaded.py:87-105).  Call with streams == NULL (or too small a capacity)
 * to learn the sizes.  status[i] != 0 marks a file the reference would skip (:133-136); its streams are inert. */
int b2_decode_plan_batch(const uint8_t* const* blobs, const uint64_t* sizes, int n, b2_image_info* infos_out,
                         int32_t* status_out, b2_image_desc* images_out, b2_stream_desc* streams_out, int streams_cap,
                         uint8_t* stage_host, uint64_t stage_cap, int n_threads, uint32_t flags, b2_decode_plan* plan);

/* Host-side, multi-threaded: read n files back to back into dst (every file starts 16-byte aligned).  Replaces the
 * per-file open(filename,'rb').read() of the reference's worker loops (_img_to_tf_mp.py:43-44,
 * _img_to_tf_threaded.py:87-88), which costs the Python shim ~30 us of interpreter time per file.
 * offsets / sizes: [n], filled in both modes.  status[i] = 0, or the errno of the failing call (that chip is then
 * skipped the way the reference's except branch does, :133-136).  *needed = bytes dst must hold.  With dst == NULL or
 * dst_cap < *needed only the sizes are gathered (call again with a buffer).  n_threads <= 0: one per host core (<= 32). */
int b2_read_files(const char* const* paths, int n, uint8_t* dst, uint64_t dst_cap, uint64_t* offsets, uint64_t* sizes,
                  int32_t* status, int n_threads, uint64_t* needed);

/* codec_mask: bit0 LZW, bit1 zlib, bit2 stored streams present.  status_dev (one int32 per image) must be
 * zeroed by the caller; non-zero afterwards = that image failed to decode (skip it, _img_to_tf_mp.py:133-136). */
int b2_decode_streams(b2_ctx* ctx, const uint8_t* blob_dev, const b2_stream_desc* streams_dev, int n_streams,
                      uint32_t codec_mask, uint32_t max_raw_len, uint8_t* scratch_dev, int32_t* status_dev,
                      b2_stream stream);
/* TIFF: predictor-2 undo, byte order, plane interleave, edge-tile crop -> (H,W,samples).  PNG: un-filter. */
int b2_assemble_images(b2_ctx* ctx, uint8_t* scratch_dev, const b2_image_desc* images_dev,
                       const b2_image_desc* images_host, int n_images, uint8_t* out_dev, int32_t* status_dev,
                       b2_stream stream);

/* ------------------------------------------------------------------ K1w: GeoTIFF writer (tile split + TIFF-LZW encode)
 * Replace GDAL's GTiff driver with COMPRESS=LZW, TILED=TRUE behind _gdal_dataset_from_geocontext + WriteArray
 * (_descartes_img_chips.py:781-797, 804-849): the chip pair a composite is saved as.  The IFD / GeoTIFF tags are
 * assembled on the host (dl_image_segmentation_b200/_geotiff.py). */
typedef struct {
    uint64_t src_off;    /* raw tile bytes in raw_dev                                                          */
    uint64_t dst_off;    /* where the code stream goes in out_dev (multiple of 4)                              */
    uint32_t src_len;
    uint32_t dst_cap;    /* 3/2 * src_len + 16 always suffices                                                 */
} b2_enc_desc;

/* TIFF-LZW encode n streams (MSB-first, leading Clear, early-change widths, Clear at 4094 entries, EOI).
 * out_len_dev[i] = bytes produced, 0xFFFFFFFF if dst_cap was too small. */
int b2_lzw_encode(b2_ctx* ctx, const uint8_t* raw_dev, const b2_enc_desc* descs_dev, int n, uint8_t* out_dev,
                  uint32_t* out_len_dev, b2_stream stream);

/* The same streams with an additional Clear code every restart_bytes input bytes (a multiple of 16, at most 1024).  A
 * Clear may appear anywhere in TIFF-LZW, every reader handles it; the pieces between two Clears are independent, so a
 * tile is encoded by hundreds of threads instead of one serial walk (one chip pair: 59 ms -> under 1 ms) and the
 * dictionaries are small enough for 28 of them per SM.  Codes stay 9-11 bits wide: noisy 16-bit imagery comes out a
 * few per cent smaller than with the full 4094-entry table, label rasters larger (0.14 -> 0.24 of raw).  descs are in
 * HOST memory here (the library plans the pieces); out_len as above.  Synchronises the stream once (upload of the plan). */
int b2_lzw_encode_restart(b2_ctx* ctx, const uint8_t* raw_dev, const b2_enc_desc* descs_host, int n, uint32_t restart_bytes,
                          uint8_t* out_dev, uint32_t* out_len_dev, b2_stream stream);

/* (H,W) raster of pixel_bytes-byte pixels (bands interleaved) -> zero-padded tile_w x tile_h tiles, tile-major. */
int b2_tile_split(b2_ctx* ctx, const uint8_t* img_dev, int H, int W, int pixel_bytes, int tile_w, int tile_h,
                  uint8_t* tiles_dev, b2_stream stream);

/* ------------------------------------------------------------------ K1j: baseline JPEG decode (SURVEY 8f row 4)
 * Replace tf.image.decode_jpeg(image_data, channels=0) behind ImageCoder.decode_jpeg
 * (_img_to_tf_threaded.py:36-38, 51-56), which _process_image runs on every .jpg chip (:97-103): libjpeg with its
 * default settings — accurate integer ("islow") inverse DCT, triangle-filter ("fancy") chroma upsampling, 16-bit
 * fixed-point YCbCr -> RGB.  In scope: 8-bit sequential Huffman files (SOF0 / SOF1) with one interleaved scan,
 * 1 component -> (H,W,1) or 3 components -> (H,W,3) RGB, any 1..4 sampling factors that divide the maximum, restart
 * intervals.  Progressive / arithmetic / lossless / 12-bit / 4-component / multi-scan files are reported as
 * unsupported (chip status 3) and skipped the way the reference skips a chip it cannot decode (:196-199). */
typedef struct {
    int32_t width, height, components;
    int32_t ycc;                    /* 1: components are Y,Cb,Cr -> RGB on output (libjpeg's JFIF / Adobe / id guess)  */
    int32_t h[3], v[3];             /* sampling factors (1,1 for a single component: never interleaved)               */
    int32_t tq[3], td[3], ta[3];    /* quantisation / DC / AC table selectors                                          */
    int32_t restart_interval;       /* MCUs between RSTn markers, 0 = none                                             */
    int32_t mcus_across, mcus_down;
    uint32_t scan_off;              /* first entropy-coded byte of the file                                            */
    uint32_t reserved;
    uint16_t qt[4][64];             /* natural (row-major) order                                                       */
    uint8_t huff_counts[2][4][16];  /* [0 DC | 1 AC][table][code length - 1]                                           */
    uint8_t huff_syms[2][4][256];
} b2_jpeg_info;

typedef struct {
    uint64_t src_off;    /* the file's bytes in blob_dev                                                             */
    uint64_t coef_off;   /* int16 index into coef_dev: 64 per block, component after component, blocks row-major     */
    uint64_t plane_off;  /* byte offset into planes_dev (multiple of 16): padded component planes one after another  */
    uint64_t out_off;    /* byte offset into out_dev: (H,W,components) uint8                                         */
    uint32_t src_len;
    int32_t image;       /* slot in status_dev                                                                       */
} b2_jpeg_job;

/* Host-side marker walk up to the first SOS.  Returns the chip status: 0 ok, 1 not a JPEG / corrupt header,
 * 3 a JPEG flavour out of scope (b2_last_error() says which). */
int b2_jpeg_probe(const uint8_t* blob, uint64_t size, b2_jpeg_info* info);
/* Host-side: int16 coefficients, bytes of padded component planes and bytes of the (H,W,components) result. */
int b2_jpeg_sizes(const b2_jpeg_info* info, uint64_t* coef_count, uint64_t* plane_bytes, uint64_t* out_bytes);
typedef struct {
    uint64_t stage_bytes;  /* host staging buffer needed for the files' bytes (each file 16-byte aligned)           */
    uint64_t coef_count;   /* int16 coefficients of all jobs                                                       */
    uint64_t plane_bytes;  /* padded component planes of all jobs                                                  */
    uint64_t out_bytes;    /* (H,W,components) results, each 256-byte aligned                                      */
    int32_t n_jobs;        /* files that passed b2_jpeg_probe                                                      */
    int32_t filled;        /* 1: stage_host was large enough and holds the bytes                                   */
} b2_jpeg_plan;

/* Host-side, multi-threaded: b2_jpeg_probe + b2_jpeg_sizes for a whole batch of files in ONE call, the job table and the
 * gather of the files' bytes into one (pinned) staging buffer — the per-file header read of the reference's worker
 * loop (_img_to_tf_threaded.py:87-105) without ~20 us of interpreter time per file.  status_out[i] (one per file) is
 * the probe's; infos_out / jobs_out are compact (n_jobs entries, input order), jobs_out[j].image = the file's index i.
 * With stage_host == NULL or stage_cap too small only sizes, infos and jobs are produced (filled = 0). */
int b2_jpeg_plan_batch(const uint8_t* const* blobs, const uint64_t* sizes, int n, b2_jpeg_info* infos_out,
                       int32_t* status_out, b2_jpeg_job* jobs_out, uint8_t* stage_host, uint64_t stage_cap,
                       int n_threads, b2_jpeg_plan* plan);

/* Entropy decode (one warp per file) -> inverse DCT (one thread per 8x8 block) -> upsample + colour conversion (one
 * thread per pixel).  coef_dev must hold coef_count int16 (zeroed here), infos / jobs are given both as device and as
 * host arrays (the host copy sizes the launches).  status_dev as for b2_decode_streams: 2 = corrupt entropy data. */
int b2_jpeg_decode(b2_ctx* ctx, const uint8_t* blob_dev, const b2_jpeg_info* infos_dev, const b2_jpeg_info* infos_host,
                   const b2_jpeg_job* jobs_dev, const b2_jpeg_job* jobs_host, int n, int16_t* coef_dev,
                   uint64_t coef_count, uint8_t* planes_dev, uint8_t* out_dev, int32_t* status_dev, b2_stream stream);

/* ------------------------------------------------------------------ K1je: baseline JPEG encode (SURVEY 8f row 4)
 * Replace tf.image.encode_jpeg(image, format='', quality=100) behind ImageCoder.png_to_jpeg
 * (_img_to_tf_threaded.py:36-38), the convert_png_to_jpg option of images_to_tfrecords_mt (:92-95): libjpeg's
 * compressor with default settings (4:2:0 for RGB, standard Huffman tables, JFIF header).  Scan bytes are identical to
 * libjpeg-turbo's; TensorFlow's header differs from a plain libjpeg one only in the JFIF density fields (unit 1,
 * 300 x 300), which b2_jpeg_header takes as arguments. */
typedef struct {
    uint64_t src_off;   /* (H,W,components) uint8 pixels in pixels_dev                                              */
    uint64_t coef_off;  /* int16 index into coef_dev: 64 per block, blocks in coding order                           */
    uint64_t out_off;   /* where the scan bytes go in out_dev                                                       */
    uint32_t out_cap;   /* b2_jpeg_encode_sizes' scan_cap always suffices                                           */
    int32_t width, height, components; /* 1 (grey) or 3 (RGB)                                                       */
} b2_jpeg_enc_job;

/* Host-side: SOI, JFIF APP0, DQT, SOF0, DHT, SOS — everything before the scan bytes (the file ends with FF D9). */
int b2_jpeg_header(int height, int width, int components, int quality, int density_unit, int x_density, int y_density,
                   uint8_t* out, uint64_t cap, uint64_t* len);
/* Host-side: int16 coefficients and an upper bound of the scan bytes of one image. */
int b2_jpeg_encode_sizes(int height, int width, int components, uint64_t* coef_count, uint64_t* scan_cap);
/* Colour conversion + down-sampling + forward DCT + quantisation (one thread per block), then block-parallel Huffman
 * coding (bit count per block, scan per image, every block writes its bits) and byte stuffing; out_off multiples of 16.  out_len_dev[j] = scan bytes of image j, 0xFFFFFFFF if out_cap was too small. */
int b2_jpeg_encode_scan(b2_ctx* ctx, const uint8_t* pixels_dev, const b2_jpeg_enc_job* jobs_dev,
                        const b2_jpeg_enc_job* jobs_host, int n, int quality, int16_t* coef_dev, uint64_t coef_count,
                        uint8_t* out_dev, uint32_t* out_len_dev, b2_stream stream);

/* n byte ranges src[src_off[i] .. +len[i]) -> dst[dst_off[i] ..): the GeoTIFF writer packs the code streams of a batch
 * (each in a capacity-sized slot) into one dense buffer on the device before the single copy to the host.  All device. */
int b2_gather_ranges(b2_ctx* ctx, const uint8_t* src, const uint64_t* src_off, const uint64_t* dst_off, const uint32_t* len,
                     int n, uint32_t max_len, uint8_t* dst, b2_stream stream);

/* ------------------------------------------------------------------ label rasterisation (SURVEY 8(f) row 4)
 * Replaces gdal.RasterizeLayer(mem_ds, [1], layer, options=['ALL_TOUCHED=TRUE'[, 'ATTRIBUTE=...']]) over a raster filled with
 * background_value, create_label_array_for_tile (_descartes_img_chips.py:633-689): polygons (any number of rings each:
 * holes, multi-polygons) burnt in feature order — the last feature touching a pixel wins — with GDAL's two passes per
 * feature: the pixel-centre scanline fill and, for ALL_TOUCHED, every pixel an edge passes through.
 * Everything is in PIXEL space (the host applies the inverse geotransform) and on the device:
 *   fill_segs      double[4] per edge of the fill pass (x1, y1, x2, y2; rings implicitly closed), grouped by feature
 *   fill_seg_off   uint32[n_features + 1]   feat_miny int32[n_features] (first scanline of the feature, clipped to the raster)
 *   job_off        uint32[n_features + 1]   prefix sum of the features' scanline counts; n_jobs = job_off[n_features]
 *   line_segs      double[4] per edge of the ALL_TOUCHED pass (n_line_segs = 0: centre-only burn), line_seg_feat its feature
 *   values         uint8[n_features] burn values
 *   job_ints_off   uint64[n_jobs + 1]   job j sorts its scanline's crossings in ints_ws[job_ints_off[j] .. job_ints_off[j + 1]):
 *                  at least the number of the feature's non-horizontal edges whose y-span holds that pixel-centre line
 *                  (a row with more crossings than its room burns only the spans of the first ones)
 *   owner_ws       int32[width * height] scratch; ints_ws int32[job_ints_off[n_jobs]] scratch; out uint8[height * width]
 * width * height must be below 2^31. */
int b2_rasterize_polygons(b2_ctx* ctx, const double* fill_segs, const uint32_t* fill_seg_off, const int32_t* feat_miny,
                          const uint32_t* job_off, uint32_t n_jobs, const double* line_segs, const uint32_t* line_seg_feat,
                          uint32_t n_line_segs, const uint8_t* values, int n_features, int width, int height, int background,
                          const uint64_t* job_ints_off, int32_t* owner_ws, int32_t* ints_ws, uint8_t* out, b2_stream stream);

/* Replaces the on-the-fly reprojection RasterizeLayer applies to every geometry, from the layer's SRS to the raster's, before
 * it burns (_descartes_img_chips.py:667-688; OGRGeometry::transform, PROJ's `utm`): n interleaved (x, y) double vertices,
 * in_dev -> out_dev (may be the same buffer).  src_epsg / dst_epsg: 4326 (x = longitude, y = latitude, degrees, GeoJSON axis
 * order; longitudes come out in [-180, 180)), 326zz (WGS84 UTM north, zone zz = 1..60) or 327zz (south, false northing
 * 10 000 000 m); k0 = 0.9996, false easting 500 000 m, central meridian -183 + 6 zz degrees.  Krueger series of order 6 in
 * the third flattening (Karney 2011), FP64; UTM -> UTM goes through latitude / longitude in the same thread; equal codes
 * copy.  A vertex that is not finite, lies beyond a pole or 90 degrees or more from the destination's central meridian
 * becomes (NaN, NaN).  An unsupported code is an error.  No datum shifts. */
int b2_project_points(b2_ctx* ctx, const double* in_dev, double* out_dev, uint64_t n, int src_epsg, int dst_epsg,
                      b2_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* B2CHIPS_H */
