// datavalues.cc — host mirror of src/datavalues: DataValue, coercion, scalar merges, device arrays.
#include <algorithm>
#include <cinttypes>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <sstream>

#include "fq_host.h"

namespace fuse {

const char *data_type_name(DataType t) {
  static const char *n[] = {"Null", "Boolean", "Int8", "Int16", "Int32", "Int64", "UInt8",
                            "UInt16", "UInt32", "UInt64", "Float32", "Float64", "Utf8", "Struct"};
  return (t >= 0 && t <= FQ_STRUCT) ? n[t] : "?";
}
static bool is_numeric(DataType t) { return t >= FQ_I8 && t <= FQ_F64; }
static bool is_float(DataType t) { return t == FQ_F32 || t == FQ_F64; }
static bool is_signed(DataType t) { return t >= FQ_I8 && t <= FQ_I64; }
static bool is_unsigned(DataType t) { return t >= FQ_U8 && t <= FQ_U64; }
static size_t type_size(DataType t) {
  switch (t) {
    case FQ_BOOL: case FQ_I8: case FQ_U8: return 1;
    case FQ_I16: case FQ_U16: return 2;
    case FQ_I32: case FQ_U32: case FQ_F32: return 4;
    case FQ_I64: case FQ_U64: case FQ_F64: return 8;
    default: return 0;
  }
}

// data_type.rs:27-87
DataType numerical_coercion(const std::string &op, DataType l, DataType r) {
  auto unsupported = [&]() {
    return FuseQueryError::internal(std::string("Unsupported (") + data_type_name(l) + ") " + op + " (" + data_type_name(r) + ")");
  };
  if (!is_numeric(l) || !is_numeric(r)) throw unsupported();
  if (l == r) return l;
  static const DataType order[] = {FQ_F64, FQ_F32, FQ_I64, FQ_I32, FQ_I16, FQ_I8, FQ_U64, FQ_U32, FQ_U16, FQ_U8};
  for (DataType t : order)
    if (l == t || r == t) return t;
  throw unsupported();
}
DataType equal_coercion(const std::string &op, DataType l, DataType r) {
  if (l == r) return l;
  return numerical_coercion(op, l, r);
}

// ---------------------------------------------------------------------------------------------
// DataValue
// ---------------------------------------------------------------------------------------------
DataValue DataValue::of(DataType t, int64_t i, uint64_t u, double f) {
  DataValue v;
  v.tag = t;
  v.some = true;
  if (is_float(t)) v.f = t == FQ_F32 ? (double)(float)f : f;
  else if (is_unsigned(t)) v.u = u;
  else v.i = i;
  return v;
}
DataValue DataValue::from_abi(const fq_value &a) {
  DataValue v;
  v.tag = a.dtype;
  if (a.dtype == FQ_NULL) return v;
  v.some = a.some != 0;
  if (!v.some) return v;
  if (is_float(a.dtype)) v.f = a.v.f;
  else if (is_unsigned(a.dtype)) v.u = a.v.u;
  else v.i = a.v.i;
  return v;
}
bool DataValue::operator==(const DataValue &o) const {
  if (tag != o.tag) return false;
  if (tag == FQ_NULL) return true;
  if (tag == FQ_STRUCT) return items == o.items;
  if (some != o.some) return false;
  if (!some) return true;
  if (tag == FQ_UTF8) return s == o.s;
  if (is_float(tag)) return f == o.f;
  if (is_unsigned(tag)) return u == o.u;
  return i == o.i;
}
static std::string shortest(double f, bool f32) {
  char tmp[64];
  for (int prec = 1; prec <= 17; prec++) {
    snprintf(tmp, sizeof tmp, "%.*g", prec, f);
    double back = f32 ? (double)strtof(tmp, nullptr) : strtod(tmp, nullptr);
    if (back == f) break;
  }
  return tmp;
}
// Display / Debug: Some(x) -> "{}", None -> "NULL", Null -> "Null" (data_value.rs:200-239, macros.rs:201-208)
std::string DataValue::to_string() const {
  if (tag == FQ_NULL) return "Null";
  if (tag == FQ_STRUCT) {
    std::string o = "[";
    for (size_t k = 0; k < items.size(); k++) o += (k ? ", " : "") + items[k].to_string();
    return o + "]";
  }
  if (!some) return "NULL";
  char buf[64];
  switch (tag) {
    case FQ_BOOL: return i ? "true" : "false";
    case FQ_UTF8: return s;
    case FQ_F32: case FQ_F64: {
      if (std::isnan(f)) return "NaN";
      if (std::isinf(f)) return f < 0 ? "-inf" : "inf";
      std::string t = shortest(f, tag == FQ_F32);
      if (t.find('e') != std::string::npos) { snprintf(buf, sizeof buf, "%.0f", f); return buf; }
      return t;  // Rust Display prints 1.0 as "1"
    }
    default:
      if (is_unsigned(tag)) snprintf(buf, sizeof buf, "%" PRIu64, u);
      else snprintf(buf, sizeof buf, "%" PRId64, i);
      return buf;
  }
}
static const char *json_tag(DataType t) {
  static const char *n[] = {"Null", "Boolean", "Int8", "Int16", "Int32", "Int64", "UInt8", "UInt16",
                            "UInt32", "UInt64", "Float32", "Float64", "String", "Struct"};
  return n[t];
}
// serde_json of the externally tagged enum — the partial-state wire format
// (transform_aggregate_partial.rs:61-66): {"Struct":[{"UInt64":123},{"UInt64":456}]}, "Null", {"UInt64":null}
std::string DataValue::to_json() const {
  if (tag == FQ_NULL) return "\"Null\"";
  std::string o = std::string("{\"") + json_tag(tag) + "\":";
  if (tag == FQ_STRUCT) {
    o += "[";
    for (size_t k = 0; k < items.size(); k++) o += (k ? "," : "") + items[k].to_json();
    o += "]";
  } else if (!some) {
    o += "null";
  } else if (tag == FQ_BOOL) {
    o += i ? "true" : "false";
  } else if (tag == FQ_UTF8) {
    o += "\"";
    for (char c : s) {
      if (c == '"' || c == '\\') { o += '\\'; o += c; }
      else if ((unsigned char)c < 0x20) { char b[8]; snprintf(b, sizeof b, "\\u%04x", c); o += b; }
      else o += c;
    }
    o += "\"";
  } else if (is_float(tag)) {
    if (std::isnan(f) || std::isinf(f)) o += "null";
    else {
      std::string t = shortest(f, tag == FQ_F32);
      if (t.find_first_of(".en") == std::string::npos) t += ".0";
      o += t;
    }
  } else {
    char buf[32];
    if (is_unsigned(tag)) snprintf(buf, sizeof buf, "%" PRIu64, u);
    else snprintf(buf, sizeof buf, "%" PRId64, i);
    o += buf;
  }
  return o + "}";
}
namespace {
struct JsonIn {
  const std::string &s;
  size_t p = 0;
  void ws() { while (p < s.size() && isspace((unsigned char)s[p])) p++; }
  [[noreturn]] void bad(const std::string &what) { throw FuseQueryError::internal(what + " at column " + std::to_string(p + 1)); }
  std::string str() {
    if (p >= s.size() || s[p] != '"') bad("expected string");
    p++;
    std::string o;
    while (p < s.size() && s[p] != '"') {
      char c = s[p];
      if (c == '\\' && p + 1 < s.size()) {
        c = s[++p];
        if (c == 'n') c = '\n';
        else if (c == 't') c = '\t';
        else if (c == 'u' && p + 4 < s.size()) { c = (char)strtol(s.substr(p + 1, 4).c_str(), nullptr, 16); p += 4; }
      }
      o += c;
      p++;
    }
    if (p >= s.size()) bad("EOF while parsing a string");
    p++;
    return o;
  }
  DataValue value() {
    ws();
    if (p < s.size() && s[p] == '"') {
      std::string v = str();
      if (v != "Null") bad("unknown variant `" + v + "`");
      return DataValue::Null();
    }
    if (p >= s.size() || s[p] != '{') bad("expected value");
    p++;
    ws();
    std::string tag = str();
    DataType t = -1;
    for (int k = 1; k <= FQ_STRUCT; k++)
      if (tag == json_tag(k)) t = k;
    if (t < 0) bad("unknown variant `" + tag + "`");
    ws();
    if (p >= s.size() || s[p] != ':') bad("expected `:`");
    p++;
    ws();
    DataValue v;
    v.tag = t;
    if (t == FQ_STRUCT) {
      if (p >= s.size() || s[p] != '[') bad("expected `[`");
      p++;
      ws();
      while (p < s.size() && s[p] != ']') {
        v.items.push_back(value());
        ws();
        if (p < s.size() && s[p] == ',') { p++; ws(); }
      }
      if (p >= s.size()) bad("EOF while parsing a list");
      p++;
    } else if (s.compare(p, 4, "null") == 0) {
      p += 4;
    } else {
      v.some = true;
      if (t == FQ_BOOL) {
        if (s.compare(p, 4, "true") == 0) { v.i = 1; p += 4; }
        else if (s.compare(p, 5, "false") == 0) { v.i = 0; p += 5; }
        else bad("expected a boolean");
      } else if (t == FQ_UTF8) {
        v.s = str();
      } else {
        const char *b = s.c_str() + p;
        char *e = nullptr;
        if (is_float(t)) v.f = strtod(b, &e);
        else if (is_signed(t)) v.i = strtoll(b, &e, 10);
        else v.u = strtoull(b, &e, 10);
        if (e == b) bad("expected a number");
        p += (size_t)(e - b);
      }
    }
    ws();
    if (p >= s.size() || s[p] != '}') bad("expected `}`");
    p++;
    return v;
  }
};
}  // namespace
DataValue DataValue::from_json(const std::string &s) {
  JsonIn in{s};
  return in.value();
}

// ---------------------------------------------------------------------------------------------
// scalar (+) scalar.  The reference routes these through 1-element Arrow arrays
// (data_value_arithmetic.rs:19-24); 16 bytes do not go to the device: same coercion, same wrapping,
// same truncating divide, same errors, evaluated inline.
// ---------------------------------------------------------------------------------------------
namespace {
struct Wide { int kind; int64_t i; uint64_t u; double f; };   // 0 signed, 1 unsigned, 2 float
Wide wide_of(const DataValue &v) {
  if (is_float(v.tag)) return {2, 0, 0, v.f};
  if (is_unsigned(v.tag)) return {1, 0, v.u, 0};
  return {0, v.i, 0, 0};
}
// arrow cast of one value: false when it would become null
bool cast_scalar(const DataValue &v, DataType to, DataValue *out) {
  *out = DataValue::None(to);
  out->some = true;
  Wide w = wide_of(v);
  if (is_float(to)) {
    double d = w.kind == 2 ? w.f : (w.kind == 1 ? (double)w.u : (double)w.i);
    out->f = to == FQ_F32 ? (double)(w.kind == 2 ? (float)w.f : (w.kind == 1 ? (float)w.u : (float)w.i)) : d;
    return true;
  }
  static const int64_t smin[] = {INT8_MIN, INT16_MIN, INT32_MIN, INT64_MIN};
  static const int64_t smax[] = {INT8_MAX, INT16_MAX, INT32_MAX, INT64_MAX};
  static const uint64_t umax[] = {UINT8_MAX, UINT16_MAX, UINT32_MAX, UINT64_MAX};
  if (is_signed(to)) {
    int k = to - FQ_I8;
    if (w.kind == 0) { if (w.i < smin[k] || w.i > smax[k]) return false; out->i = w.i; }
    else if (w.kind == 1) { if (w.u > (uint64_t)smax[k]) return false; out->i = (int64_t)w.u; }
    else {
      if (std::isnan(w.f)) return false;
      double tr = std::trunc(w.f);
      if (k == 3 ? !(tr >= -9223372036854775808.0 && tr < 9223372036854775808.0) : (tr < (double)smin[k] || tr > (double)smax[k])) return false;
      out->i = (int64_t)tr;
    }
    return true;
  }
  int k = to - FQ_U8;
  if (w.kind == 0) { if (w.i < 0 || (uint64_t)w.i > umax[k]) return false; out->u = (uint64_t)w.i; }
  else if (w.kind == 1) { if (w.u > umax[k]) return false; out->u = w.u; }
  else {
    if (std::isnan(w.f)) return false;
    double tr = std::trunc(w.f);
    if (k == 3 ? !(tr > -1.0 && tr < 18446744073709551616.0) : (tr < 0 || tr > (double)umax[k])) return false;
    out->u = (uint64_t)tr;
  }
  return true;
}
int64_t wrap_signed(uint64_t x, DataType t) {
  switch (t) { case FQ_I8: return (int8_t)x; case FQ_I16: return (int16_t)x; case FQ_I32: return (int32_t)x; default: return (int64_t)x; }
}
uint64_t wrap_unsigned(uint64_t x, DataType t) {
  switch (t) { case FQ_U8: return (uint8_t)x; case FQ_U16: return (uint16_t)x; case FQ_U32: return (uint32_t)x; default: return x; }
}
const char *arith_sym(int op) { static const char *s[] = {"+", "-", "*", "/"}; return s[op & 3]; }
const char *agg_name(int op) { static const char *s[] = {"min", "max", "sum", "count"}; return s[op & 3]; }
// DataValue::to_array's refusal of Type(None) (data_value.rs:104-109)
void require_some(const DataValue &v) {
  if (v.tag == FQ_UTF8) return;
  if (v.tag == FQ_STRUCT || !v.some) throw FuseQueryError::internal("DataValue to array cannot be NONE " + v.to_string());
}
}  // namespace

DataValue data_value_arithmetic_op(int op, const DataValue &l, const DataValue &r) {
  if (l.tag == FQ_NULL) return r;
  if (r.tag == FQ_NULL) return l;
  require_some(l);
  require_some(r);
  DataType t = numerical_coercion(arith_sym(op), l.tag, r.tag);
  DataValue a, b;
  bool va = cast_scalar(l, t, &a), vb = cast_scalar(r, t, &b);
  DataValue out = DataValue::None(t);
  if (!va || !vb) return out;  // a null operand yields a null slot
  out.some = true;
  if (is_float(t)) {
    if (op == FQ_AR_DIV && b.f == 0.0) throw FuseQueryError::internal("Divide by zero error");
    double x = op == FQ_AR_ADD ? a.f + b.f : op == FQ_AR_SUB ? a.f - b.f : op == FQ_AR_MUL ? a.f * b.f : a.f / b.f;
    if (t == FQ_F32) {
      float fa = (float)a.f, fb = (float)b.f;
      x = op == FQ_AR_ADD ? fa + fb : op == FQ_AR_SUB ? fa - fb : op == FQ_AR_MUL ? fa * fb : fa / fb;
    }
    out.f = x;
  } else if (is_signed(t)) {
    if (op == FQ_AR_DIV) {
      if (b.i == 0) throw FuseQueryError::internal("Divide by zero error");
      out.i = b.i == -1 ? wrap_signed(0ull - (uint64_t)a.i, t) : a.i / b.i;
    } else {
      uint64_t x = op == FQ_AR_ADD ? (uint64_t)a.i + (uint64_t)b.i : op == FQ_AR_SUB ? (uint64_t)a.i - (uint64_t)b.i : (uint64_t)a.i * (uint64_t)b.i;
      out.i = wrap_signed(x, t);
    }
  } else {
    if (op == FQ_AR_DIV) {
      if (b.u == 0) throw FuseQueryError::internal("Divide by zero error");
      out.u = a.u / b.u;
    } else {
      uint64_t x = op == FQ_AR_ADD ? a.u + b.u : op == FQ_AR_SUB ? a.u - b.u : a.u * b.u;
      out.u = wrap_unsigned(x, t);
    }
  }
  return out;
}

DataValue data_value_aggregate_op(int op, const DataValue &l, const DataValue &r) {
  if (l.tag == FQ_NULL) return r;
  if (r.tag == FQ_NULL) return l;
  bool ok = l.tag == r.tag && (is_numeric(l.tag) || l.tag == FQ_UTF8);
  if (ok && l.tag == FQ_UTF8 && (op == FQ_AGG_SUM || op == FQ_AGG_COUNT)) ok = false;
  if (!ok)
    throw FuseQueryError::internal(std::string("Unsupported data_value_") + agg_name(op) + " for data type: left:" +
                                   data_type_name(l.tag) + ", right:" + data_type_name(r.tag));
  if (op == FQ_AGG_COUNT) return DataValue::UInt64(1);  // sic, data_value_aggregate.rs:20
  if (!l.some && !r.some) return DataValue::None(l.tag);
  if (!r.some) return l;
  if (!l.some) return r;
  DataValue out = DataValue::None(l.tag);
  out.some = true;
  DataType t = l.tag;
  if (t == FQ_UTF8) {
    int c = l.s.compare(r.s);
    out.s = (op == FQ_AGG_MIN ? c <= 0 : c >= 0) ? l.s : r.s;
  } else if (is_float(t)) {
    if (op == FQ_AGG_SUM) out.f = t == FQ_F32 ? (double)((float)l.f + (float)r.f) : l.f + r.f;
    else out.f = op == FQ_AGG_MIN ? std::fmin(l.f, r.f) : std::fmax(l.f, r.f);
  } else if (is_signed(t)) {
    if (op == FQ_AGG_SUM) out.i = wrap_signed((uint64_t)l.i + (uint64_t)r.i, t);
    else out.i = op == FQ_AGG_MIN ? std::min(l.i, r.i) : std::max(l.i, r.i);
  } else {
    if (op == FQ_AGG_SUM) out.u = wrap_unsigned(l.u + r.u, t);
    else out.u = op == FQ_AGG_MIN ? std::min(l.u, r.u) : std::max(l.u, r.u);
  }
  return out;
}

// ---------------------------------------------------------------------------------------------
// schema
// ---------------------------------------------------------------------------------------------
int DataSchema::index_of(const std::string &name) const {
  for (size_t i = 0; i < fields.size(); i++)
    if (fields[i].name == name) return (int)i;
  std::string valid;
  for (size_t i = 0; i < fields.size(); i++) valid += (i ? ", \"" : "\"") + fields[i].name + "\"";
  throw FuseQueryError::internal("Invalid argument error: Unable to get field named \"" + name + "\". Valid fields: [" + valid + "]");
}

// ---------------------------------------------------------------------------------------------
// GPU context + device arrays
// ---------------------------------------------------------------------------------------------
GpuContextRef GpuContext::create(int device) {
  fq_ctx *c = nullptr;
  fq_status st = fq_ctx_create(device, &c);
  if (st) throw FuseQueryError::from_abi(st, fq_last_error(nullptr));
  auto g = std::shared_ptr<GpuContext>(new GpuContext());
  g->ctx_ = c;
  g->device_ = device;
  return g;
}
GpuContext::~GpuContext() { fq_ctx_destroy(ctx_); }
void GpuContext::check(fq_status st) const {
  if (st) throw FuseQueryError::from_abi(st, fq_last_error(ctx_));
}
PipeHandle::~PipeHandle() {
  if (pipe) fq_pipe_destroy(ctx ? ctx->raw() : nullptr, pipe);
}

Utf8Dict::~Utf8Dict() {
  if (raw) fq_utf8_free(ctx ? ctx->raw() : nullptr, raw);
}
// strings rows[0 .. n) of `src` (NULL slots, per `valid`, as "") copied to the host
static std::vector<std::string> decode_rows(const GpuContextRef &ctx, const fq_utf8 *src, const fq_column *rows, uint64_t n, const fq_column *valid) {
  fq_utf8 *t = nullptr;
  ctx->check(fq_utf8_take(ctx->raw(), src, rows, n, valid, &t, ctx->stream));
  std::vector<int32_t> off(n + 1, 0);
  std::string bytes(fq_utf8_bytes(t), '\0');
  fq_status st = fq_utf8_download(ctx->raw(), t, off.data(), bytes.data(), ctx->stream);
  if (st == FQ_OK) st = fq_stream_synchronize(ctx->raw(), ctx->stream);
  fq_utf8_free(ctx->raw(), t);
  ctx->check(st);
  std::vector<std::string> out(n);
  for (uint64_t i = 0; i < n; i++) out[i] = bytes.substr((size_t)off[i], (size_t)(off[i + 1] - off[i]));
  return out;
}
std::string Utf8Dict::at(uint32_t code) const {
  if (code >= size) throw FuseQueryError::internal("dictionary code " + std::to_string(code) + " out of range");
  DataArrayRef rows = DataArray::from_host(ctx, FQ_U32, &code, 1);
  return decode_rows(ctx, raw, rows->column(), 1, nullptr)[0];
}

std::pair<uint64_t, uint64_t> Utf8Dict::bounds(const std::string &literal) const {
  std::lock_guard<std::mutex> lock(mu_);
  auto it = bounds_.find(literal);
  if (it != bounds_.end()) return it->second;
  std::pair<uint64_t, uint64_t> b;
  ctx->check(fq_utf8_bounds(ctx->raw(), raw, literal.data(), literal.size(), &b.first, &b.second, ctx->stream));
  if (bounds_.size() >= 4096) bounds_.clear();   // many distinct literals: keep the memory bounded
  bounds_[literal] = b;
  return b;
}
DataArrayRef Utf8Dict::like(const std::string &pattern, bool negate) const {
  std::lock_guard<std::mutex> lock(mu_);
  const auto key = std::make_pair(pattern, negate);
  auto it = like_.find(key);
  if (it != like_.end()) return it->second;
  const uint64_t bytes = std::max<uint64_t>(1, (size + 7) / 8);
  // fq_utf8_like writes ceil(size / 8) bytes: the table of an empty dictionary is one zero byte, so that no byte of it is left unset
  static const unsigned char zero = 0;
  DataArrayRef bits = size ? DataArray::alloc(ctx, FQ_U8, bytes) : DataArray::from_host(ctx, FQ_U8, &zero, 1);
  ctx->check(fq_utf8_like(ctx->raw(), raw, pattern.data(), pattern.size(), negate ? 1 : 0, bits->column(), ctx->stream));
  // many distinct patterns: keep the memory bounded (pipes that still read a table share its ownership)
  if (like_.size() >= 4096 || like_bytes_ + bytes > (256ull << 20)) {
    like_.clear();
    like_bytes_ = 0;
  }
  like_[key] = bits;
  like_bytes_ += bytes;
  return bits;
}

DataArray::~DataArray() {
  if (col_) fq_column_free(ctx_ ? ctx_->raw() : nullptr, col_);
}
DataArrayRef DataArray::device(GpuContextRef ctx, fq_column *col, DataArrayRef parent) {
  auto a = std::shared_ptr<DataArray>(new DataArray());
  a->ctx_ = std::move(ctx);
  a->col_ = col;
  a->dtype_ = fq_column_dtype(col);
  a->len_ = fq_column_len(col);
  a->parent_ = std::move(parent);
  return a;
}
DataArrayRef DataArray::alloc(GpuContextRef ctx, DataType t, uint64_t len) {
  fq_column *c = nullptr;
  ctx->check(fq_column_alloc(ctx->raw(), t, len, &c));
  return device(std::move(ctx), c);
}
DataArrayRef DataArray::from_host(GpuContextRef ctx, DataType t, const void *data, uint64_t len) {
  auto a = alloc(ctx, t, len);
  if (len) {
    ctx->check(fq_column_upload(ctx->raw(), a->col_, 0, data, len, ctx->stream));
    ctx->check(fq_stream_synchronize(ctx->raw(), ctx->stream));
  }
  return a;
}
DataArrayRef DataArray::from_arrow_bitmap(GpuContextRef ctx, const void *bits, uint64_t bit_offset, uint64_t len) {
  auto a = alloc(ctx, FQ_BOOL, len);
  if (len) {
    ctx->check(fq_column_upload_bits(ctx->raw(), a->col_, 0, bits, bit_offset, len, ctx->stream));
    ctx->check(fq_stream_synchronize(ctx->raw(), ctx->stream));
  }
  return a;
}
std::vector<unsigned char> DataArray::to_arrow_bitmap() const {
  if (dtype_ != FQ_BOOL) throw FuseQueryError::internal("to_arrow_bitmap on a non-Boolean array");
  std::vector<unsigned char> out((len_ + 7) / 8);
  if (len_) {
    ctx_->check(fq_column_download_bits(ctx_->raw(), col_, 0, out.data(), len_, ctx_->stream));
    ctx_->check(fq_stream_synchronize(ctx_->raw(), ctx_->stream));
  }
  return out;
}
void DataArray::set_validity(DataArrayRef validity) {
  if (is_host_utf8()) throw FuseQueryError::internal("validity on a Utf8 array is not supported");
  if (validity && (validity->data_type() != FQ_BOOL || validity->len() < len_)) throw FuseQueryError::internal("validity must be a Boolean array of the same length");
  ctx_->check(fq_column_set_validity(ctx_->raw(), col_, validity ? validity->column() : nullptr));
  validity_ = std::move(validity);
}
uint64_t DataArray::null_count() const {
  if (!validity_ || !len_) return 0;
  std::vector<unsigned char> v(len_);
  validity_->to_host(v.data());
  uint64_t n = 0;
  for (unsigned char b : v) n += b == 0;
  return n;
}
DataArrayRef DataArray::utf8(std::vector<std::string> values) {
  auto a = std::shared_ptr<DataArray>(new DataArray());
  a->dtype_ = FQ_UTF8;
  a->len_ = values.size();
  a->strings_ = std::move(values);
  return a;
}
DataArrayRef DataArray::utf8_dict(GpuContextRef ctx, const int32_t *offsets, const void *data, uint64_t len, const unsigned char *valid) {
  DataArrayRef v = valid ? from_host(ctx, FQ_BOOL, valid, len) : nullptr;
  fq_utf8 *src = nullptr;
  ctx->check(fq_utf8_create(ctx->raw(), offsets, data, len, v ? v->column() : nullptr, ctx->stream, &src));
  DataArrayRef codes = alloc(ctx, FQ_U32, len);
  auto d = std::make_shared<Utf8Dict>();
  d->ctx = ctx;
  const fq_status st = fq_utf8_dict_encode(ctx->raw(), src, codes->column(), &d->raw, ctx->stream);
  fq_utf8_free(ctx->raw(), src);
  ctx->check(st);
  d->size = fq_utf8_len(d->raw);
  if (v) codes->set_validity(v);
  return with_dict(codes, d);
}
DataArrayRef DataArray::with_dict(const DataArrayRef &codes, Utf8DictRef dict) {
  if (codes->data_type() != FQ_U32 || codes->dict_) throw FuseQueryError::internal("dictionary codes must be a UInt32 array");
  fq_column *c = nullptr;
  codes->ctx_->check(fq_column_slice(codes->ctx_->raw(), codes->col_, 0, codes->len_, &c));
  DataArrayRef a = device(codes->ctx_, c, codes->parent_ ? codes->parent_ : codes);   // a view: the codes stay alive
  a->validity_ = codes->validity_;
  a->dtype_ = FQ_UTF8;
  a->dict_ = std::move(dict);
  return a;
}
const std::vector<std::string> &DataArray::strings() const {
  if (dict_ && !decoded_) {
    strings_ = len_ ? decode_rows(ctx_, dict_->raw, col_, len_, validity_ ? validity_->column() : nullptr) : std::vector<std::string>{};
    decoded_ = true;
  }
  return strings_;
}
DataArrayRef DataArray::slice(uint64_t offset, uint64_t len) {
  if (is_host_utf8()) {
    std::vector<std::string> v(strings_.begin() + (long)std::min<uint64_t>(offset, len_), strings_.begin() + (long)std::min<uint64_t>(offset + len, len_));
    return utf8(std::move(v));
  }
  fq_column *c = nullptr;
  ctx_->check(fq_column_slice(ctx_->raw(), col_, offset, len, &c));
  DataArrayRef out = device(ctx_, c, parent_ ? parent_ : shared_from_this());  // the owner of the buffer stays alive
  if (validity_) out->validity_ = validity_->slice(offset, len);   // the C ABI sliced the device validity alongside
  out->dtype_ = dtype_;   // a dictionary array's slice shares its dictionary
  out->dict_ = dict_;
  return out;
}
void DataArray::to_host(void *out) const {
  if (is_utf8()) throw FuseQueryError::internal("to_host on a Utf8 array");
  if (!len_) return;
  ctx_->check(fq_column_download(ctx_->raw(), col_, 0, out, len_, ctx_->stream));
  ctx_->check(fq_stream_synchronize(ctx_->raw(), ctx_->stream));
}
// DataValue::try_from_array (data_value.rs:115-161)
DataValue DataArray::value(uint64_t index) const {
  if (index >= len_) throw FuseQueryError::internal("index out of bounds: the len is " + std::to_string(len_) + " but the index is " + std::to_string(index));
  if (is_host_utf8()) return DataValue::String(strings_[index]);
  if (dict_) {
    unsigned char ok = 1;
    if (validity_) {
      ctx_->check(fq_column_download(ctx_->raw(), validity_->column(), index, &ok, 1, ctx_->stream));
      ctx_->check(fq_stream_synchronize(ctx_->raw(), ctx_->stream));
    }
    return ok ? DataValue::String(strings()[index]) : DataValue::None(FQ_UTF8);
  }
  unsigned char buf[8] = {0};
  ctx_->check(fq_column_download(ctx_->raw(), col_, index, buf, 1, ctx_->stream));
  ctx_->check(fq_stream_synchronize(ctx_->raw(), ctx_->stream));
  DataValue v = DataValue::None(dtype_);
  if (validity_) {
    unsigned char ok = 1;
    ctx_->check(fq_column_download(ctx_->raw(), validity_->column(), index, &ok, 1, ctx_->stream));
    ctx_->check(fq_stream_synchronize(ctx_->raw(), ctx_->stream));
    if (!ok) return v;   // Type(None)
  }
  v.some = true;
  switch (dtype_) {
    case FQ_BOOL: v.i = buf[0] != 0; break;
    case FQ_I8: v.i = *(int8_t *)buf; break;
    case FQ_I16: v.i = *(int16_t *)buf; break;
    case FQ_I32: v.i = *(int32_t *)buf; break;
    case FQ_I64: v.i = *(int64_t *)buf; break;
    case FQ_U8: v.u = *(uint8_t *)buf; break;
    case FQ_U16: v.u = *(uint16_t *)buf; break;
    case FQ_U32: v.u = *(uint32_t *)buf; break;
    case FQ_U64: v.u = *(uint64_t *)buf; break;
    case FQ_F32: v.f = *(float *)buf; break;
    case FQ_F64: v.f = *(double *)buf; break;
    default: throw FuseQueryError::internal(std::string("Can't create a scalar of array of type \"") + data_type_name(dtype_) + "\"");
  }
  return v;
}

// DataValue::to_array (data_value.rs:76-112): broadcast a scalar to `size` rows on the device
DataArrayRef DataColumnarValue::to_array(GpuContextRef ctx, uint64_t size) const {
  if (!is_scalar) return array;
  if (scalar.tag == FQ_UTF8) {
    if (scalar.some) return DataArray::utf8(std::vector<std::string>(size, scalar.s));
    // Utf8(None) (min / max of strings that are all NULL) broadcasts to NULL rows, not to empty strings.  A host Utf8
    // array carries no validity, so the rows are an all-NULL column encoded like a table's: an empty dictionary
    std::vector<int32_t> offsets(size + 1, 0);
    std::vector<unsigned char> valid(size, 0);
    return DataArray::utf8_dict(std::move(ctx), offsets.data(), "", size, valid.data());
  }
  require_some(scalar);
  if (scalar.tag == FQ_NULL) throw FuseQueryError::internal("Unsupported on the device path: NullArray");
  // fill through the host: broadcasts only materialise for tiny arrays on this path (merge_result().to_array(1),
  // transform_aggregate_final.rs:68-72); per-row literals are immediates inside the fused kernels
  size_t w = type_size(scalar.tag);
  std::vector<unsigned char> host(w * size);
  unsigned char one[8] = {0};
  switch (scalar.tag) {
    case FQ_BOOL: one[0] = scalar.i ? 1 : 0; break;
    case FQ_I8: *(int8_t *)one = (int8_t)scalar.i; break;
    case FQ_I16: *(int16_t *)one = (int16_t)scalar.i; break;
    case FQ_I32: *(int32_t *)one = (int32_t)scalar.i; break;
    case FQ_I64: *(int64_t *)one = scalar.i; break;
    case FQ_U8: *(uint8_t *)one = (uint8_t)scalar.u; break;
    case FQ_U16: *(uint16_t *)one = (uint16_t)scalar.u; break;
    case FQ_U32: *(uint32_t *)one = (uint32_t)scalar.u; break;
    case FQ_U64: *(uint64_t *)one = scalar.u; break;
    case FQ_F32: *(float *)one = (float)scalar.f; break;
    default: *(double *)one = scalar.f; break;
  }
  for (uint64_t k = 0; k < size; k++) memcpy(host.data() + k * w, one, w);
  return DataArray::from_host(std::move(ctx), scalar.tag, host.data(), size);
}

// ---------------------------------------------------------------------------------------------
// GpuGroup
// ---------------------------------------------------------------------------------------------
GpuGroup::GpuGroup(GpuContextRef gpu, int rank, int world, uint64_t row_bytes) : gpu_(std::move(gpu)), rank_(rank), world_(world) {
  gpu_->check(fq_group_create(gpu_->raw(), rank, world, row_bytes, &raw_));
}
GpuGroup::~GpuGroup() { fq_group_destroy(gpu_->raw(), raw_); }
std::string GpuGroup::handle() const {
  std::string h(64, '\0');
  gpu_->check(fq_group_handle(gpu_->raw(), raw_, &h[0]));
  return h;
}
void GpuGroup::connect(const std::vector<std::string> &handles) {
  if ((int)handles.size() != world_) throw FuseQueryError::internal("group of " + std::to_string(world_) + " ranks got " + std::to_string(handles.size()) + " handles");
  std::string blob;
  for (const auto &h : handles) {
    std::string x = h;
    x.resize(64, '\0');
    blob += x;
  }
  gpu_->check(fq_group_connect(gpu_->raw(), raw_, blob.data()));
}
std::pair<std::vector<DataArrayRef>, uint64_t> GpuGroup::gather(const std::vector<DataArrayRef> &cols, const std::vector<DataType> &types, uint64_t rows,
                                                                uint64_t selected_local, uint64_t capacity, int64_t limit) {
  const uint64_t out_rows = limit >= 0 ? std::min<uint64_t>((uint64_t)limit, capacity * (uint64_t)world_) : capacity * (uint64_t)world_;
  std::vector<DataArrayRef> finals;
  std::vector<const fq_column *> lc;
  std::vector<fq_column *> fc;
  for (size_t i = 0; i < types.size(); i++) {
    finals.push_back(DataArray::alloc(gpu_, types[i], std::max<uint64_t>(out_rows, 1)));
    fc.push_back(finals.back()->column());
    lc.push_back(i < cols.size() && cols[i] ? cols[i]->column() : nullptr);
  }
  gpu_->check(fq_group_gather_columns(gpu_->raw(), raw_, lc.data(), nullptr, (int32_t)types.size(), rows, selected_local, capacity, fc.data(), nullptr,
                                      limit, gpu_->stream));
  uint64_t selected = 0, n = 0;
  gpu_->check(fq_group_fetch_gather(gpu_->raw(), raw_, &selected, &n));
  for (auto &a : finals) a = a->slice(0, n);
  return {finals, selected};
}

}  // namespace fuse
