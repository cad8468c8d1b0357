// api.cu -- the C ABI of libtfrgpu.so (include/tfrgpu.h) and the host-side runtime above the kernels:
// schema lowering, per-task decoder/encoder handles (device + stream + reusable buffers), batch
// ownership, host copies and Arrow C Data Interface export.  No torch types, no CPU fallback: every
// compute path below launches the sm_100a kernels of frame.cuh / decode.cuh / scan.cuh / encode.cuh.
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>      // header-only NVTX 3: ranges show up in Nsight Systems / ncu --nvtx, cost nothing when no tool is attached
#include <algorithm>
#include <cmath>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"
#include "decode.cuh"
#include "encode.cuh"
#include "encode_tile.cuh"
#include "bytes_tile.cuh"
#include "frame.cuh"
#include "host_util.h"
#include "infer.cuh"
#include "scan.cuh"
#include "tile.cuh"

// ---------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
static int32_t fail(int32_t code, const std::string& msg) { g_last_error = msg; return code; }
#define CUDA_TRY(expr)                                                                             \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess) return fail(TFR_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
  } while (0)

int32_t DevBuf::ensure(size_t bytes) {
  cudaError_t e = ensure_raw(bytes);
  if (e != cudaSuccess) return fail(e == cudaErrorMemoryAllocation ? TFR_E_OOM : TFR_E_CUDA, std::string("device allocation failed: ") + cudaGetErrorString(e));
  return TFR_OK;
}
#define TRY(expr) do { int32_t _rc = (expr); if (_rc) return _rc; } while (0)

// NVTX range over one C-ABI call (SURVEY.md section 5: the tracing hook of this path)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

extern "C" int32_t tfr_abi_version(void) { return TFR_ABI_VERSION; }
extern "C" const char* tfr_last_error(void) { return g_last_error.c_str(); }
extern "C" const char* tfr_status_string(int32_t s) {
  switch (s) {
    case TFR_OK: return "ok";
    case TFR_E_INVALID_ARG: return "invalid argument";
    case TFR_E_UNSUPPORTED_TYPE: return "unsupported data type";
    case TFR_E_BAD_RECORD_TYPE: return "unsupported recordType: recordType can be ByteArray, Example or SequenceExample";
    case TFR_E_CUDA: return "CUDA error / no usable device";
    case TFR_E_OOM: return "out of memory";
    case TFR_E_BATCH_TOO_LARGE: return "batch too large (2 GiB of framed bytes / int32 Arrow offsets)";
    case TFR_E_CRC_LENGTH: return "Length header crc32 checking failed";
    case TFR_E_CRC_DATA: return "Data crc32 checking failed";
    case TFR_E_TRUNCATED: return "End of file reached before reading fully";
    case TFR_E_RECORD_TOO_LARGE: return "Record size exceeds max value of int32";
    case TFR_E_MALFORMED_PROTO: return "Protocol message was malformed";
    case TFR_E_KIND_MISMATCH: return "Feature must be of the list kind the column type requires";
    case TFR_E_EMPTY_SCALAR: return "head of empty list";
    case TFR_E_NULL_IN_NONNULL: return "field does not allow null values";
    case TFR_E_BAD_NESTING: return "Cannot convert Feature/FeatureList to this array nesting";
    default: return "unknown status";
  }
}

// ---------------------------------------------------------------------------------------------
// per-device context: CRC tables
// ---------------------------------------------------------------------------------------------
struct DeviceCtx {
  std::once_flag once;
  CrcTables* d_tabs = nullptr;
  cudaError_t err = cudaSuccess;
  int sm_count = 148;
  int max_smem_optin = 48 * 1024;
  std::mutex smem_mu;                                  // guards smem_set
  std::map<const void*, size_t> smem_set;              // kernel -> the opt-in dynamic shared memory set on this device
};
static DeviceCtx g_ctx[64];

// The opt-in limit of dynamic shared memory is an attribute of the kernel on the device, shared by every handle and thread,
// and cudaFuncSetAttribute SETS it.  This is its one owner: the value only ever grows, and it is read, compared and set under
// the device's lock, so a launch with at most `bytes` is valid afterwards whatever other handles launch meanwhile.  The
// caller has made ctx's device current.
static cudaError_t ensure_dyn_smem(DeviceCtx* ctx, const void* kernel, size_t bytes) {
  std::lock_guard<std::mutex> lk(ctx->smem_mu);
  size_t& cur = ctx->smem_set[kernel];
  if (cur >= bytes) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) cur = bytes;
  return e;
}

static void build_crc_tables(CrcTables& t) {
  const uint32_t POLY = 0x82F63B78u;
  for (uint32_t i = 0; i < 256; ++i) {
    uint32_t c = i;
    for (int k = 0; k < 8; ++k) c = (c >> 1) ^ (POLY & (0u - (c & 1u)));
    t.t0[i] = c;
  }
  auto mulmod = [&](uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (int i = 31; i >= 0; --i) {
      if ((a >> i) & 1u) p ^= b;
      b = (b >> 1) ^ (POLY & (0u - (b & 1u)));
    }
    return p;
  };
  auto xpow_bytes = [&](uint32_t nbytes) {     // x^(8*nbytes) mod P
    uint32_t x8 = 0x80000000u;
    for (int i = 0; i < 8; ++i) x8 = (x8 >> 1) ^ (POLY & (0u - (x8 & 1u)));
    uint32_t r = 0x80000000u, base = x8;
    while (nbytes) { if (nbytes & 1) r = mulmod(r, base); base = mulmod(base, base); nbytes >>= 1; }
    return r;
  };
  uint32_t x128 = xpow_bytes(128);
  for (int s = 0; s < 4; ++s)
    for (uint32_t b = 0; b < 256; ++b) t.k128[s][b] = mulmod(x128, b << (8 * s));
  for (uint32_t k = 0; k < 40; ++k) t.xw[k] = xpow_bytes(4 * k);
  for (uint32_t i = 0; i < 256; ++i) {
    t.s8[0][i] = t.t0[i];
    for (int k = 1; k < 8; ++k) t.s8[k][i] = (t.s8[k - 1][i] >> 8) ^ t.t0[t.s8[k - 1][i] & 0xff];
  }
  for (uint32_t m = 0; m < 512; ++m) t.xp16[m] = xpow_bytes(16 * m);
  memset(t.g5, 0, sizeof t.g5);
  for (uint32_t k = 0; k < 13; ++k)
    for (uint32_t v = 0; v < 32; ++v) {
      uint32_t r = 0;
      for (uint32_t j = 0; j < 5; ++j) {
        const uint32_t bit = 5 * k + j;
        if (((v >> j) & 1u) && bit < 64) r ^= t.s8[7 - bit / 8][1u << (bit % 8)];
      }
      t.g5[k * 32 + v] = r;
    }
  for (uint32_t v = 0; v < 32; ++v) t.g5[416 + v] = t.t0[v];
  for (uint32_t w = 0; w < 8; ++w) t.g5[448 + w] = t.t0[w << 5];
}

static int32_t get_ctx(int device, DeviceCtx** out) {
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return fail(TFR_E_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e));
  if (device < 0 || device >= ndev || device >= 64) return fail(TFR_E_INVALID_ARG, "bad device index");
  DeviceCtx& c = g_ctx[device];
  std::call_once(c.once, [&] {
    c.err = cudaSetDevice(device);
    if (c.err != cudaSuccess) return;
    cudaDeviceProp prop;
    c.err = cudaGetDeviceProperties(&prop, device);
    if (c.err != cudaSuccess) return;
    c.sm_count = prop.multiProcessorCount;
    c.max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    {   // keep stream-ordered allocations cached in the pool instead of returning them to the OS at every sync
      cudaMemPool_t pool;
      if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        unsigned long long thr = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
      }
    }
    CrcTables* h = new CrcTables;
    build_crc_tables(*h);
    c.err = cudaMalloc(&c.d_tabs, sizeof(CrcTables));
    if (c.err == cudaSuccess) c.err = cudaMemcpy(c.d_tabs, h, sizeof(CrcTables), cudaMemcpyHostToDevice);
    delete h;
  });
  if (c.err != cudaSuccess) return fail(TFR_E_CUDA, std::string("device init: ") + cudaGetErrorString(c.err));
  *out = &c;
  return TFR_OK;
}

// ---------------------------------------------------------------------------------------------
// schema
// ---------------------------------------------------------------------------------------------
struct tfr_schema {
  int32_t record_type = 0;
  std::vector<DevField> fields;      // device layout, filled on the host
  std::vector<uint8_t> names;
  std::vector<int32_t> ht;
  std::vector<int32_t> var_field;    // var slot -> field
  std::vector<int32_t> fix_field;    // fix slot -> field
  int32_t n_fix = 0, n_var = 0, n_cnt = 0;
};

static uint32_t fnv1a(const uint8_t* p, uint32_t n) { uint32_t h = 2166136261u; for (uint32_t i = 0; i < n; ++i) h = (h ^ p[i]) * 16777619u; return h; }

extern "C" int32_t tfr_schema_create(const tfr_field* fields, int32_t n_fields, int32_t record_type, tfr_schema** out) {
  if (!out || n_fields < 0 || (n_fields > 0 && !fields)) return fail(TFR_E_INVALID_ARG, "null argument");
  if (record_type < TFR_RT_EXAMPLE || record_type > TFR_RT_BYTE_ARRAY)
    return fail(TFR_E_BAD_RECORD_TYPE, "Unsupported recordType: recordType can be ByteArray, Example or SequenceExample");
  if (n_fields > 4096) return fail(TFR_E_INVALID_ARG, "more than 4096 fields");
  auto* s = new tfr_schema;
  s->record_type = record_type;
  if (record_type == TFR_RT_BYTE_ARRAY) {
    // the single binary column of TensorFlowInferSchema.getSchemaForByteArray (M/TensorFlowInferSchema.scala:60-64);
    // the caller's field list is ignored like deserializeByteArray ignores the schema (:17-19)
    DevField d{};
    d.name_off = 0; d.name_len = 9; s->names.assign((const uint8_t*)"byteArray", (const uint8_t*)"byteArray" + 9);
    d.hash = fnv1a(s->names.data(), 9);
    d.elem_type = TFR_T_BINARY; d.depth = 0; d.nullable = 1; d.kind = K_BYTES; d.n_levels = 1; d.dup_next = -1;
    d.fix_slot = -1; d.var_slot = 0; d.cnt_slot = 0; d.width = 1;
    s->fields.push_back(d);
    s->var_field.push_back(0);
    s->n_var = 1; s->n_cnt = 1;
    s->ht.assign(2, -1);
    s->ht[d.hash & 1] = 0;
    *out = s;
    return TFR_OK;
  }
  for (int32_t i = 0; i < n_fields; ++i) {
    const tfr_field& f = fields[i];
    if (f.name_len < 0 || (f.name_len > 0 && !f.name)) { delete s; return fail(TFR_E_INVALID_ARG, "bad field name"); }
    std::string nm(f.name ? f.name : "", (size_t)f.name_len);
    // newFeatureWriter / newFeatureConverter: anything but these types throws (M/TFRecordDeserializer.scala:119-123,
    // M/TFRecordSerializer.scala:147,151); ArrayType(NullType) falls into the same default branch
    bool ok_type = f.elem_type >= TFR_T_NULL && f.elem_type <= TFR_T_BINARY && f.depth >= 0 && f.depth <= 2 &&
                   !(f.elem_type == TFR_T_NULL && f.depth > 0);
    if (!ok_type) { delete s; return fail(TFR_E_UNSUPPORTED_TYPE, "field '" + nm + "': data type is not supported"); }
    DevField d{};
    d.name_off = (uint32_t)s->names.size();
    d.name_len = (uint32_t)f.name_len;
    s->names.insert(s->names.end(), (const uint8_t*)f.name, (const uint8_t*)f.name + f.name_len);
    d.hash = fnv1a((const uint8_t*)f.name, d.name_len);
    d.elem_type = (int8_t)f.elem_type; d.depth = (int8_t)f.depth; d.nullable = f.nullable ? 1 : 0;
    d.kind = (int8_t)required_kind(f.elem_type);
    bool varlen = f.elem_type == TFR_T_STRING || f.elem_type == TFR_T_BINARY;
    d.n_levels = (int16_t)(f.depth + (varlen ? 1 : 0));
    d.dup_next = -1;
    d.width = type_width(f.elem_type);
    d.fix_slot = -1; d.var_slot = -1; d.cnt_slot = -1;
    if (f.elem_type == TFR_T_NULL) { /* no storage beyond validity */ }
    else if (d.n_levels == 0) { d.fix_slot = s->n_fix++; s->fix_field.push_back(i); }
    else { d.var_slot = s->n_var++; d.cnt_slot = s->n_cnt; s->n_cnt += d.n_levels; s->var_field.push_back(i); }
    s->fields.push_back(d);
  }
  // Spark refuses duplicate column names for file sources before the reader is built
  // (SchemaUtils.checkColumnNameDuplication), so they never reach TFRecordDeserializer
  size_t hsz = 2; while (hsz < 2 * (size_t)n_fields + 2) hsz <<= 1;
  s->ht.assign(hsz, -1);
  for (int32_t i = 0; i < n_fields; ++i) {
    const DevField& d = s->fields[i];
    size_t slot = d.hash & (hsz - 1);
    while (s->ht[slot] >= 0) {
      const DevField& o = s->fields[s->ht[slot]];
      if (o.hash == d.hash && o.name_len == d.name_len && memcmp(&s->names[o.name_off], &s->names[d.name_off], d.name_len) == 0) {
        delete s; return fail(TFR_E_INVALID_ARG, "Found duplicate column(s) in the data schema");
      }
      slot = (slot + 1) & (hsz - 1);
    }
    s->ht[slot] = i;
  }
  *out = s;
  return TFR_OK;
}
extern "C" void tfr_schema_destroy(tfr_schema* s) { delete s; }
extern "C" int32_t tfr_schema_num_fields(const tfr_schema* s) { return s ? (int32_t)s->fields.size() : 0; }

// device copy of a schema
struct DevSchemaBuf {
  DevField* d_fields = nullptr; uint8_t* d_names = nullptr; int32_t* d_ht = nullptr; int32_t* d_var_field = nullptr;
  FieldTemplate* d_templates = nullptr;
  uint8_t* d_tile_consts = nullptr; uint32_t tile_consts_bytes = 0;     // tile.cuh: per-schema constants in the shared-memory layout
  DevSchema view{};
  int32_t upload(const tfr_schema& s) {
    size_t nf = s.fields.size();
    CUDA_TRY(cudaMalloc(&d_fields, std::max<size_t>(1, nf) * sizeof(DevField)));
    CUDA_TRY(cudaMalloc(&d_names, std::max<size_t>(1, s.names.size())));
    CUDA_TRY(cudaMalloc(&d_ht, s.ht.size() * sizeof(int32_t)));
    CUDA_TRY(cudaMalloc(&d_var_field, std::max<size_t>(1, s.var_field.size()) * sizeof(int32_t)));
    if (nf) CUDA_TRY(cudaMemcpy(d_fields, s.fields.data(), nf * sizeof(DevField), cudaMemcpyHostToDevice));
    if (!s.names.empty()) CUDA_TRY(cudaMemcpy(d_names, s.names.data(), s.names.size(), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_ht, s.ht.data(), s.ht.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    if (!s.var_field.empty()) CUDA_TRY(cudaMemcpy(d_var_field, s.var_field.data(), s.var_field.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    {
      // canonical entry prefix of every field: 0A ? 0A klen key 12 ? kindtag ?   (? = length bytes, masked out)
      std::vector<FieldTemplate> tp(std::max<size_t>(1, nf));
      for (size_t f = 0; f < nf; ++f) {
        FieldTemplate& t = tp[f];
        memset(&t, 0, sizeof t);
        const DevField& fd = s.fields[f];
        t.kind = (uint32_t)fd.kind;
        const uint32_t klen = fd.name_len, total = klen + 8;
        if (fd.kind == K_NONE || klen >= 0x80 || total > TILE_TPL_WORDS * 4) continue;      // no template: generic parse
        uint8_t bytes[TILE_TPL_WORDS * 4] = {0}, mask[TILE_TPL_WORDS * 4] = {0};
        auto put = [&](uint32_t i, uint8_t b, bool fixed) { bytes[i] = b; mask[i] = fixed ? 0xFF : 0x00; };
        put(0, 0x0A, true); put(1, 0, false); put(2, 0x0A, true); put(3, (uint8_t)klen, true);
        for (uint32_t i = 0; i < klen; ++i) put(4 + i, s.names[fd.name_off + i], true);
        put(4 + klen, 0x12, true); put(5 + klen, 0, false);
        put(6 + klen, fd.kind == K_BYTES ? 0x0A : fd.kind == K_FLOAT ? 0x12 : 0x1A, true); put(7 + klen, 0, false);
        t.n_words = (uint16_t)((total + 3) / 4); t.klen = (uint16_t)klen;
        memcpy(t.words, bytes, sizeof bytes); memcpy(t.mask, mask, sizeof mask);
      }
      CUDA_TRY(cudaMalloc(&d_templates, tp.size() * sizeof(FieldTemplate)));
      CUDA_TRY(cudaMemcpy(d_templates, tp.data(), tp.size() * sizeof(FieldTemplate), cudaMemcpyHostToDevice));
    }
    view.n_fields = (int32_t)nf; view.record_type = s.record_type; view.ht_mask = (int32_t)s.ht.size() - 1;
    view.n_fix = s.n_fix; view.n_var = s.n_var; view.n_cnt = s.n_cnt;
    view.fields = d_fields; view.names = d_names; view.ht = d_ht;
    return TFR_OK;
  }
  // CRC tables | zeroed seen words | DevField[nf] | FieldTemplate[nf] | names, each section 16-byte aligned (tile_const_bytes)
  int32_t build_tile_consts(const tfr_schema& s, const CrcTables* d_tabs) {
    const uint32_t nf = (uint32_t)s.fields.size(), nb = (uint32_t)s.names.size();
    tile_consts_bytes = tile_const_bytes(nf, nb);
    CUDA_TRY(cudaMalloc(&d_tile_consts, tile_consts_bytes));
    CUDA_TRY(cudaMemset(d_tile_consts, 0, tile_consts_bytes));
    uint8_t* q = d_tile_consts;
    CUDA_TRY(cudaMemcpy(q, d_tabs->g5, TILE_CRC_BYTES, cudaMemcpyDeviceToDevice));   // g5 then xp16, contiguous in CrcTables
    q += TILE_CRC_BYTES + TILE_SEEN_BYTES;
    if (nf) CUDA_TRY(cudaMemcpy(q, d_fields, nf * sizeof(DevField), cudaMemcpyDeviceToDevice));
    q += (nf * sizeof(DevField) + 15) & ~(size_t)15;
    if (nf) CUDA_TRY(cudaMemcpy(q, d_templates, nf * sizeof(FieldTemplate), cudaMemcpyDeviceToDevice));
    q += (nf * sizeof(FieldTemplate) + 15) & ~(size_t)15;
    if (nb) CUDA_TRY(cudaMemcpy(q, d_names, nb, cudaMemcpyDeviceToDevice));
    return TFR_OK;
  }
  void free_all() { cudaFree(d_fields); cudaFree(d_names); cudaFree(d_ht); cudaFree(d_var_field); cudaFree(d_templates); cudaFree(d_tile_consts); }
};

#include "api_decode.inc"

// ---------------------------------------------------------------------------------------------
// Arrow C Data Interface export (arrow/c/abi.h structs restated in host_util.h)
// ---------------------------------------------------------------------------------------------
struct ExportPriv { tfr_batch* batch; std::vector<const void*> buffers; std::vector<ArrowArray*> children; ArrowArray* child_storage = nullptr; };

static void release_array(ArrowArray* a) {
  if (!a || !a->release) return;
  auto* p = (ExportPriv*)a->private_data;
  for (int64_t i = 0; i < a->n_children; ++i) {
    if (a->children[i]->release) a->children[i]->release(a->children[i]);
    delete a->children[i];
  }
  if (p) { if (p->batch) tfr_batch_release(p->batch); delete p; }
  a->release = nullptr;
}
static void release_schema(ArrowSchema* s) {
  if (!s || !s->release) return;
  for (int64_t i = 0; i < s->n_children; ++i) {
    if (s->children[i]->release) s->children[i]->release(s->children[i]);
    delete s->children[i];
  }
  delete[] s->children;
  free((void*)s->name);
  s->release = nullptr;
}
static const char* leaf_format(int t) {
  switch (t) {
    case TFR_T_INT32: return "i"; case TFR_T_INT64: return "l"; case TFR_T_FLOAT32: return "f";
    case TFR_T_FLOAT64: case TFR_T_DECIMAL: return "g"; case TFR_T_STRING: return "u"; case TFR_T_BINARY: return "z";
    default: return "n";
  }
}
static void build_schema(ArrowSchema* s, const char* name, int elem_type, int depth) {
  memset(s, 0, sizeof *s);
  s->name = strdup(name); s->flags = 2 /*ARROW_FLAG_NULLABLE*/; s->release = release_schema;
  if (depth == 0) { s->format = leaf_format(elem_type); return; }
  s->format = "+l";
  s->n_children = 1; s->children = new ArrowSchema*[1];
  s->children[0] = new ArrowSchema;
  build_schema(s->children[0], "item", elem_type, depth - 1);
}
// level: which offsets level this list node uses; leaves use the last level for utf8/binary
static void build_array(ArrowArray* a, const tfr_column& c, int level, int64_t length, tfr_batch* owner) {
  memset(a, 0, sizeof *a);
  auto* p = new ExportPriv;
  p->batch = owner;
  if (owner) owner->refs.fetch_add(1);
  a->private_data = p; a->release = release_array; a->length = length; a->offset = 0;
  const bool varlen = c.elem_type == TFR_T_STRING || c.elem_type == TFR_T_BINARY;
  const void* validity = level == 0 ? c.validity : nullptr;
  a->null_count = level == 0 ? c.null_count : 0;
  if (level < c.depth) {                 // list node
    p->buffers = {validity, c.offsets[level]};
    a->n_buffers = 2;
    a->n_children = 1;
    p->children.resize(1); p->children[0] = new ArrowArray;
    a->children = p->children.data();
    int64_t child_len = level + 1 < c.n_levels ? c.n_offsets[level + 1] - 1 : c.n_values;
    build_array(a->children[0], c, level + 1, child_len, nullptr);
  } else if (c.elem_type == TFR_T_NULL) {
    a->n_buffers = 0; a->null_count = length;
  } else if (varlen) {
    p->buffers = {validity, c.offsets[c.n_levels - 1], c.values};
    a->n_buffers = 3;
  } else {
    p->buffers = {validity, c.values};
    a->n_buffers = 2;
  }
  a->buffers = p->buffers.data();
}

extern "C" int32_t tfr_batch_export_arrow_host(tfr_batch* b, int32_t column, void* arrow_array, void* arrow_schema) {
  if (!b || !arrow_array || !arrow_schema || column < 0 || column >= (int32_t)b->cols.size()) return fail(TFR_E_INVALID_ARG, "bad argument");
  int32_t rc = tfr_batch_to_host(b, nullptr, (int32_t)b->cols.size());
  if (rc) return rc;
  const tfr_column& c = b->host_cols[column];
  const tfr_schema& S = b->dec->schema;
  std::string nm((const char*)&S.names[S.fields[column].name_off], S.fields[column].name_len);
  build_schema((ArrowSchema*)arrow_schema, nm.c_str(), c.elem_type, c.depth);
  build_array((ArrowArray*)arrow_array, c, 0, c.n_rows, b);
  return TFR_OK;
}
extern "C" int32_t tfr_batch_export_arrow_device(tfr_batch* b, int32_t column, void* arrow_device_array, void* arrow_schema) {
  if (!b || !arrow_device_array || !arrow_schema || column < 0 || column >= (int32_t)b->cols.size()) return fail(TFR_E_INVALID_ARG, "bad argument");
  int32_t rc = tfr_batch_wait(b);
  if (rc) return rc;
  const tfr_column& c = b->cols[column];
  const tfr_schema& S = b->dec->schema;
  std::string nm((const char*)&S.names[S.fields[column].name_off], S.fields[column].name_len);
  build_schema((ArrowSchema*)arrow_schema, nm.c_str(), c.elem_type, c.depth);
  auto* da = (ArrowDeviceArray*)arrow_device_array;
  memset(da, 0, sizeof *da);
  build_array(&da->array, c, 0, c.n_rows, b);
  da->device_id = b->dec->device; da->device_type = 2 /*ARROW_DEVICE_CUDA*/; da->sync_event = nullptr;   // batch already waited
  return TFR_OK;
}

#include "api_encode.inc"
