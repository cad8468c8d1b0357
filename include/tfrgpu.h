/*
 * tfrgpu.h -- C ABI of libtfrgpu.so: the B200-native TFRecord decode/encode hot path
 * behind the spark-tfrecord DataSource API.
 *
 * Every entry point below is what a JNI (or ctypes) shim binds; there are no C++ or
 * torch types in any signature.  Each declaration cites the reference interface
 * (linkedin/spark-tfrecord @ 5bc46ee) it replaces.  Shorthand:
 *   M/ = src/main/scala/com/linkedin/spark/datasources/tfrecord/
 *
 * Conventions
 *   - every function returns int32_t: 0 (TFR_OK) or a negative TFR_E_* code;
 *     a human-readable message for the last failure on a handle is available through
 *     tfr_last_error().  No exception ever crosses this boundary.
 *   - handles are thread-confined, the library is re-entrant: one decoder/encoder per
 *     Spark task thread (M/TFRecordFileReader.scala:16-20 is called once per file per
 *     task; M/TFRecordOutputWriter.scala:12-24 is one instance per task).
 *   - the CUDA device is mandatory.  There is no CPU fallback anywhere behind this ABI:
 *     creating a decoder/encoder without a usable sm_100 device fails with TFR_E_CUDA.
 */
#ifndef TFRGPU_H_
#define TFRGPU_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TFR_ABI_VERSION 2

/* ---- status codes (SURVEY.md section 8b "error conventions") ------------------------- */
enum {
  TFR_OK = 0,
  TFR_E_INVALID_ARG      = -1,  /* bad handle / null pointer / bad enum              */
  TFR_E_UNSUPPORTED_TYPE = -2,  /* M/TFRecordDeserializer.scala:119,123 ; M/TFRecordSerializer.scala:147,151 -> RuntimeException at construction */
  TFR_E_BAD_RECORD_TYPE  = -3,  /* M/TFRecordFileReader.scala:78-79 -> IllegalArgumentException */
  TFR_E_CUDA             = -4,  /* no device / CUDA runtime error                     */
  TFR_E_OOM              = -5,
  TFR_E_BATCH_TOO_LARGE  = -6,  /* a batch must stay below 2 GiB of framed bytes and int32 Arrow offsets */
  /* per-record data errors; the JNI shim maps them to the Java exception the
   * reference would have thrown for the same record (see INTEGRATION.md)            */
  TFR_E_CRC_LENGTH       = -10, /* tensorflow-hadoop TFRecordReader: length CRC mismatch -> IOException      */
  TFR_E_CRC_DATA         = -11, /* payload CRC mismatch -> IOException                                        */
  TFR_E_TRUNCATED        = -12, /* EOF inside a record -> IOException                                         */
  TFR_E_RECORD_TOO_LARGE = -13, /* length > Integer.MAX_VALUE -> IOException                                  */
  TFR_E_MALFORMED_PROTO  = -14, /* Example.parseFrom / SequenceExample.parseFrom (M/TFRecordFileReader.scala:73,76) -> InvalidProtocolBufferException */
  TFR_E_KIND_MISMATCH    = -15, /* require(...) M/TFRecordDeserializer.scala:178,189,201,212 -> IllegalArgumentException */
  TFR_E_EMPTY_SCALAR     = -16, /* .head on empty list M/TFRecordDeserializer.scala:75-94 -> NoSuchElementException */
  TFR_E_NULL_IN_NONNULL  = -17, /* M/TFRecordDeserializer.scala:31,56 ; M/TFRecordSerializer.scala:29-31,53-55 -> NullPointerException */
  TFR_E_BAD_NESTING      = -18  /* 2-D column fed from context / scalar column fed from feature_lists:
                                   M/TFRecordDeserializer.scala:119,142 -> RuntimeException */
};

/* ---- schema -------------------------------------------------------------------------- */
/* element types: the Spark SQL types the reference accepts (M/TFRecordDeserializer.scala:70-124,
 * M/TFRecordSerializer.scala:68-152; README "supported data types")                       */
enum {
  TFR_T_NULL    = 0,  /* NullType: always null on read (:71-72), never written (:70)          */
  TFR_T_INT32   = 1,  /* IntegerType <- Int64List, low 32 bits (:74-75)                       */
  TFR_T_INT64   = 2,  /* LongType                                                             */
  TFR_T_FLOAT32 = 3,  /* FloatType                                                            */
  TFR_T_FLOAT64 = 4,  /* DoubleType <- FloatList widened (:83-84); written via toFloat        */
  TFR_T_DECIMAL = 5,  /* DecimalType: carried as float64 (f.toDouble, :86-87); the JVM shim wraps it in Decimal */
  TFR_T_STRING  = 6,  /* StringType <- BytesList, Java UTF-8 decode/re-encode semantics (:89-91) */
  TFR_T_BINARY  = 7   /* BinaryType <- BytesList raw (:93-95)                                 */
};

/* record types: the `recordType` DataSource option (M/TFRecordFileReader.scala:22,69-80) */
enum { TFR_RT_EXAMPLE = 0, TFR_RT_SEQUENCE_EXAMPLE = 1, TFR_RT_BYTE_ARRAY = 2 };

/* One StructField of the (required) schema.  depth 0 = scalar, 1 = ArrayType(elem),
 * 2 = ArrayType(ArrayType(elem)) (SequenceExample feature_lists only).                    */
typedef struct tfr_field {
  const char* name;      /* UTF-8 bytes, not necessarily NUL terminated */
  int32_t     name_len;
  int32_t     elem_type; /* TFR_T_*  */
  int32_t     depth;     /* 0, 1, 2  */
  int32_t     nullable;  /* StructField.nullable */
} tfr_field;

typedef struct tfr_schema  tfr_schema;
typedef struct tfr_decoder tfr_decoder;
typedef struct tfr_encoder tfr_encoder;
typedef struct tfr_batch   tfr_batch;

int32_t tfr_abi_version(void);
/* message text for a status code (static storage) */
const char* tfr_status_string(int32_t status);
/* last error text recorded on this thread by a failing call (create-time errors) */
const char* tfr_last_error(void);

/* Replaces `new TFRecordDeserializer(schema)` (M/TFRecordFileReader.scala:44) and
 * `new TFRecordSerializer(dataSchema)` (M/TFRecordOutputWriter.scala:24): validates the types
 * up front the way TFRecordSerializer's constructor does (M/TFRecordSerializer.scala:14).   */
int32_t tfr_schema_create(const tfr_field* fields, int32_t n_fields, int32_t record_type,
                          tfr_schema** out);
void    tfr_schema_destroy(tfr_schema*);
int32_t tfr_schema_num_fields(const tfr_schema*);

/* ---- decode: replaces the body of the buildReader closure ---------------------------- */
/* flags */
#define TFR_F_VERIFY_CRC   0x1u  /* tensorflow-hadoop's CRC check (on by default there)   */
#define TFR_F_DEFAULT      (TFR_F_VERIFY_CRC)

/* Replaces TFRecordFileReader.readFile's setup (M/TFRecordFileReader.scala:16-44):
 * binds a device, a CUDA stream and reusable device/pinned buffers.                        */
int32_t tfr_decoder_create(const tfr_schema*, int32_t device, uint32_t flags, tfr_decoder** out);
void    tfr_decoder_destroy(tfr_decoder*);

/* Pinned host staging the caller fills with framed file bytes (the JVM sees it as a direct
 * ByteBuffer).  Grows on demand; the pointer stays valid until the next call that needs
 * more capacity or destroy.  A decoder has tfr_decoder_num_staging_slots() such buffers so
 * that block t+1 can be read from the file while block t is in flight (tfr_decode_submit);
 * a slot may be refilled once the batch decoded from it has been waited on.
 * tfr_decoder_staging is slot 0.                                                           */
int32_t tfr_decoder_staging(tfr_decoder*, size_t min_bytes, void** host_ptr, size_t* capacity);
int32_t tfr_decoder_staging_slot(tfr_decoder*, int32_t slot, size_t min_bytes, void** host_ptr, size_t* capacity);
int32_t tfr_decoder_num_staging_slots(void);

/* The hot path.  Replaces the per-record loop recordReader.nextKeyValue -> parseFrom ->
 * deserializeExample (M/TFRecordFileReader.scala:49-81, M/TFRecordDeserializer.scala:21-61).
 *   data/nbytes : framed TFRecord bytes (u64 len | u32 maskedcrc(len) | payload | u32 maskedcrc)
 *                 starting at a record boundary; in host memory (pageable or the pinned
 *                 staging above) or in device memory (data_on_device != 0).  Device input: any
 *                 alignment gets the single-pass tile kernels, and NO padding around the buffer is
 *                 required: 16-byte groups that cross data or data + nbytes are never bulk-copied,
 *                 and no 4-byte aligned word that holds no byte of the buffer is ever touched.
 *                 The buffer must stay valid and unchanged until the batch has been waited on.
 *   is_final    : nonzero -> a trailing partial record is TFR_E_TRUNCATED (EOF inside a
 *                 record); zero -> it is left unconsumed (see *consumed).
 * tfr_decode returns when the batch is complete and verified (*consumed is final): no kernel
 * reads `data` any more, so a device buffer may be overwritten or freed right away.
 * A data error does not fail the call: rows before the first bad record are delivered and
 * the error is reported by tfr_batch_status, like the reference's iterator which yields
 * rows until the throwing record.
 *
 * tfr_decode_submit is the pipelined form: it enqueues the copy, the frame index and the decode
 * and returns without waiting.  Once a decoder has seen its first batches (record size and
 * column shapes learned) this involves no host/device synchronisation at all; the batch's
 * result, including consumed_bytes, is available after tfr_batch_wait / tfr_batch_status /
 * tfr_batch_columns / tfr_batch_to_host, which also redo -- transparently, with identical
 * results -- any batch the single-pass kernels could not vouch for.  At most
 * tfr_decoder_num_staging_slots() submitted batches are in flight per decoder; a further
 * submit first waits for the oldest one.                                                   */
int32_t tfr_decode(tfr_decoder*, const void* data, size_t nbytes, int32_t data_on_device,
                   int32_t is_final, tfr_batch** out, size_t* consumed);
int32_t tfr_decode_submit(tfr_decoder*, const void* data, size_t nbytes, int32_t data_on_device,
                          int32_t is_final, tfr_batch** out);

int32_t tfr_decoder_stream(tfr_decoder*, void** cuda_stream /* cudaStream_t */);

/* Measurement hooks (bench.py): with profiling enabled the decoder brackets every stage with CUDA
 * events on its own stream.  tfr_decoder_get_profile synchronises the stream and returns cumulative
 * device milliseconds per stage since profiling was enabled:
 *   ms[0] frame index (scan+check+repair+finish+emit)   ms[1] decode pass 1 (CRC + parse)
 *   ms[2] scans + summary                               ms[3] decode pass 2 (variable-width emit)
 *   ms[4] validity pack                                 ms[5] H2D of the input (host input only)
 *   ms[6] D2H of the Arrow buffers (tfr_batch_to_host[_async])
 * plus the number of kernel launches and of pass-1 launches.                                  */
#define TFR_PROFILE_STAGES 8
int32_t tfr_decoder_set_profiling(tfr_decoder*, int32_t enable);
int32_t tfr_decoder_get_profile(tfr_decoder*, double* ms /* [TFR_PROFILE_STAGES] */, int64_t* kernel_launches,
                                int64_t* pass1_launches);
/* counters since creation: [0] batches decoded, [1] submitted speculatively (no host sync), [2] of those redone after
 * the device raised a flag, [3] batches through count mode (ragged / learning), [4] through the general kernels,
 * [5] column shapes (re)learned, [6] batches re-run by the single-pass kernel's transcoding instantiation (malformed
 * UTF-8 in a string column)                                                                                       */
int32_t tfr_decoder_get_stats(tfr_decoder*, int64_t* out, int32_t n /* <= 8 */);

int32_t tfr_batch_wait(tfr_batch*);
typedef struct tfr_batch_info {
  int64_t n_rows;          /* rows delivered (records before the first error)              */
  int64_t n_records;       /* record frames found in the consumed bytes                    */
  int64_t consumed_bytes;
  int32_t error_code;      /* TFR_OK or the TFR_E_* of the first failing record            */
  int64_t error_row;       /* its 0-based record index, -1 if none                         */
  int32_t error_field;     /* schema field index for semantic errors, -1 otherwise         */
  int64_t out_bytes;       /* Arrow bytes produced (validity+offsets+values, all columns)  */
  int32_t frame_repairs;   /* chunks whose speculative boundary had to be re-chained       */
} tfr_batch_info;
int32_t tfr_batch_status(tfr_batch*, tfr_batch_info* out);
/* Bytes of the submitted block this batch consumes, available as soon as the batch's frame index has run -- before its
 * rows are decoded.  The block loop of a streaming reader (TFRecordFileReader.scala:49-61: records are read one after
 * the other, so block t+1 starts where block t's last complete record ended) calls this right after tfr_decode_submit,
 * cuts and submits the next block, and only then waits for this one's rows: the decode of block t runs under the frame
 * index of block t+1.  For a batch that later reports an error, tfr_batch_info.consumed_bytes (the bytes in front of the
 * failing record) is what counts; the reader stops there anyway.                                                     */
int32_t tfr_batch_consumed(tfr_batch*, size_t* consumed);

/* One output column in Arrow layout.  n_levels offset arrays (int32, Arrow list/binary
 * offsets) from the outermost (one entry per row + 1) to the innermost, then the leaf
 * values.  Scalar fixed width: n_levels = 0.  Pointers are device pointers
 * (tfr_batch_columns) or host pointers (tfr_batch_to_host).                                */
typedef struct tfr_column {
  int32_t  elem_type;      /* TFR_T_*                                                      */
  int32_t  depth;
  int32_t  n_levels;       /* depth + (elem is STRING/BINARY ? 1 : 0)                      */
  int32_t  value_width;    /* bytes per leaf value (1 for STRING/BINARY data)              */
  int64_t  n_rows;
  int64_t  null_count;
  uint8_t* validity;       /* Arrow bitmap, LSB first, bit=1 -> valid; (n_rows+7)/8 bytes  */
  int32_t* offsets[3];
  int64_t  n_offsets[3];   /* entries in offsets[i] (= parent count + 1)                   */
  void*    values;
  int64_t  n_values;       /* leaf elements (bytes for STRING/BINARY)                      */
} tfr_column;

int32_t tfr_batch_num_columns(tfr_batch*);
/* device-resident view (zero copy; valid until tfr_batch_release) */
int32_t tfr_batch_columns(tfr_batch*, tfr_column* out, int32_t n);
/* copies every buffer to pinned host memory owned by the batch (D2H on the decoder's
 * copy-out stream) -- the path a row-based InternalRow consumer uses.  tfr_batch_to_host_async
 * only enqueues the copy behind the batch's kernels (so that it overlaps the next batch's
 * H2D and decode); tfr_batch_to_host waits for it and returns the host view.               */
int32_t tfr_batch_to_host_async(tfr_batch*);
int32_t tfr_batch_to_host(tfr_batch*, tfr_column* out, int32_t n);
/* Arrow C Data Interface export of one column from the host copy (struct ArrowArray /
 * struct ArrowSchema from arrow/c/abi.h, passed as void* to keep this header standalone);
 * the consumer calls ->release.  Device variant fills struct ArrowDeviceArray.             */
int32_t tfr_batch_export_arrow_host(tfr_batch*, int32_t column, void* arrow_array, void* arrow_schema);
int32_t tfr_batch_export_arrow_device(tfr_batch*, int32_t column, void* arrow_device_array, void* arrow_schema);
void    tfr_batch_release(tfr_batch*);

/* ---- encode: replaces TFRecordOutputWriter.write/close -------------------------------- */
/* Replaces the constructor M/TFRecordOutputWriter.scala:12-24.                             */
int32_t tfr_encoder_create(const tfr_schema*, int32_t device, uint32_t flags, tfr_encoder** out);
void    tfr_encoder_destroy(tfr_encoder*);

/* Replaces write(row) for a batch of rows (M/TFRecordOutputWriter.scala:26-38 ->
 * serializeExample M/TFRecordSerializer.scala:20-35 -> toByteArray -> TFRecordWriter.write):
 * columns in the tfr_column layout above (host or device pointers), n = number of schema
 * fields.  Produces the framed bytes of all rows, in row order, byte-identical to what the
 * reference writer appends to its output stream.  *out_dev is device memory owned by the
 * encoder, valid until the next tfr_encode/destroy.  A null in a non-nullable column is
 * TFR_E_NULL_IN_NONNULL with *error_row set.
 * tfr_encode may return with the last kernel still queued on tfr_encoder_stream:
 *   - host columns (columns_on_device == 0) have been copied when the call returns and may
 *     be reused or freed at once;
 *   - device columns are read by that kernel: keep them valid and unchanged until the
 *     encoder's stream has drained (tfr_encoder_result_host returns, the stream is
 *     synchronised, or the caller's own work is ordered behind it with an event);
 *   - *out_dev holds the bytes once the same point is reached: device consumers order their
 *     reads behind tfr_encoder_stream; tfr_encoder_result_host waits itself.               */
int32_t tfr_encode(tfr_encoder*, const tfr_column* columns, int32_t n, int32_t columns_on_device,
                   void** out_dev, size_t* out_bytes, int64_t* error_row);
/* copy the last encode result to host memory (pinned staging owned by the encoder) */
int32_t tfr_encoder_result_host(tfr_encoder*, void** host_ptr, size_t* nbytes);
int32_t tfr_encoder_stream(tfr_encoder*, void** cuda_stream);

/* ---- schema inference (SURVEY.md 8f.1; M/TensorFlowInferSchema.scala:35-58) ------------ */
/* lattice codes of M/TensorFlowInferSchema.scala:194-207; merge = max, 0 = identity     */
enum { TFR_INF_NULL = 0, TFR_INF_LONG = 1, TFR_INF_FLOAT = 2, TFR_INF_STRING = 3,
       TFR_INF_ARR_LONG = 4, TFR_INF_ARR_FLOAT = 5, TFR_INF_ARR_STRING = 6,
       TFR_INF_ARR2_LONG = 7, TFR_INF_ARR2_FLOAT = 8, TFR_INF_ARR2_STRING = 9,
       TFR_INF_ARR2_NULL = 10 /* ArrayType(ArrayType(null)): a FeatureList whose steps are all empty (:102-107) */ };
typedef struct tfr_infer tfr_infer;
int32_t tfr_infer_create(int32_t record_type, int32_t device, tfr_infer** out);
/* accumulate one block of framed bytes (seqOp of rdd.aggregate, :40,43).  tfr_infer_update takes a whole
 * file (a trailing partial record is TFR_E_TRUNCATED); tfr_infer_update_block streams a file of any size in
 * blocks below 2 GiB with the tfr_decode contract (is_final / *consumed).                                  */
int32_t tfr_infer_update(tfr_infer*, const void* data, size_t nbytes, int32_t data_on_device);
int32_t tfr_infer_update_block(tfr_infer*, const void* data, size_t nbytes, int32_t data_on_device,
                               int32_t is_final, size_t* consumed);
/* number of distinct feature names seen so far, then the (name, code) pairs; names are
 * returned sorted bytewise so that ranks can merge them deterministically               */
int32_t tfr_infer_result(tfr_infer*, int32_t* n_names);
int32_t tfr_infer_name(tfr_infer*, int32_t i, const char** name, int32_t* name_len, int32_t* code);
void    tfr_infer_destroy(tfr_infer*);

#ifdef __cplusplus
}
#endif
#endif /* TFRGPU_H_ */
