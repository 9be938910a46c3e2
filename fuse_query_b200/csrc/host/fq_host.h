// fq_host.h — C++ host mirror of the reference's operator / plugin surface for the hot path.
//
// Same names, argument meaning and error behaviour as the Rust crate (file:line cited per item, relative
// to /root/reference/src), implemented on top of the C ABI in include/fuse_gpu.h and nothing else: every
// array lives in HBM as an fq_column, every per-row computation is a fused sm_100a kernel.  This is
// what a Rust maintainer's FFI crate would look like from the inside (INTEGRATION.md shows the Rust
// side); here it is C++ because no Rust toolchain exists in this image.
#pragma once

#include <algorithm>
#include <cstdint>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../../include/fuse_gpu.h"

namespace fuse {

// ---------------------------------------------------------------------------------------------
// error.rs:10-20
// ---------------------------------------------------------------------------------------------
struct FuseQueryError : std::runtime_error {
  enum Kind { SQLParse, Plan, Internal } kind;
  FuseQueryError(Kind k, const std::string &display) : std::runtime_error(display), kind(k) {}
  static FuseQueryError internal(const std::string &m) { return FuseQueryError(Internal, "Internal Error: " + m); }
  static FuseQueryError plan(const std::string &m) { return FuseQueryError(Plan, "Error during plan: " + m); }
  static FuseQueryError sql(const std::string &m) { return FuseQueryError(SQLParse, "SQLParser Error: " + m); }
  // text already carries its prefix (messages coming back through fq_last_error)
  static FuseQueryError from_abi(fq_status st, const std::string &display) {
    return FuseQueryError(st == FQ_ERR_PLAN ? Plan : Internal, display);
  }
};

// ---------------------------------------------------------------------------------------------
// datavalues
// ---------------------------------------------------------------------------------------------
using DataType = fq_dtype;  // datavalues/data_type.rs:7 (arrow DataType), tags of data_value.rs:19-35
const char *data_type_name(DataType t);
DataType numerical_coercion(const std::string &op, DataType l, DataType r);  // data_type.rs:27-87
DataType equal_coercion(const std::string &op, DataType l, DataType r);      // data_type.rs:89-98

// data_value.rs:19-35
struct DataValue {
  DataType tag = FQ_NULL;   // FQ_NULL = DataValue::Null
  bool some = false;        // Type(None) when false
  int64_t i = 0;            // Boolean / Int*
  uint64_t u = 0;           // UInt*
  double f = 0;             // Float*
  std::string s;            // String
  std::vector<DataValue> items;  // Struct

  static DataValue Null() { return DataValue(); }
  static DataValue None(DataType t) { DataValue v; v.tag = t; return v; }
  static DataValue UInt64(uint64_t x) { DataValue v; v.tag = FQ_U64; v.some = true; v.u = x; return v; }
  static DataValue Int64(int64_t x) { DataValue v; v.tag = FQ_I64; v.some = true; v.i = x; return v; }
  static DataValue Float64(double x) { DataValue v; v.tag = FQ_F64; v.some = true; v.f = x; return v; }
  static DataValue String(const std::string &x) { DataValue v; v.tag = FQ_UTF8; v.some = true; v.s = x; return v; }
  static DataValue Struct(std::vector<DataValue> it) { DataValue v; v.tag = FQ_STRUCT; v.items = std::move(it); return v; }
  static DataValue of(DataType t, int64_t i, uint64_t u, double f);
  static DataValue from_abi(const fq_value &v);

  bool is_null() const { return tag != FQ_NULL && tag != FQ_STRUCT && !some; }  // data_value.rs:40-56
  DataType data_type() const { return tag; }
  std::string to_string() const;                 // Display / Debug, data_value.rs:200-239
  std::string to_json() const;                   // serde_json (externally tagged)
  static DataValue from_json(const std::string &s);
  bool operator==(const DataValue &o) const;
};

// data_value_arithmetic.rs:10-27 and data_value_aggregate.rs:8-101 (scalar (+) scalar on the host: 32 bytes)
DataValue data_value_arithmetic_op(int op, const DataValue &l, const DataValue &r);
DataValue data_value_aggregate_op(int op, const DataValue &l, const DataValue &r);

struct DataField { std::string name; DataType data_type; bool nullable; };   // data_field.rs
struct DataSchema {                                                           // data_schema.rs
  std::vector<DataField> fields;
  int index_of(const std::string &name) const;  // throws like arrow's Schema::index_of
  const DataField &field_with_name(const std::string &name) const { return fields[index_of(name)]; }
};
using DataSchemaRef = std::shared_ptr<const DataSchema>;

class GpuContext;
using GpuContextRef = std::shared_ptr<GpuContext>;
class DataArray;

// The sorted dictionary of a dictionary-encoded Utf8 column (fq_utf8_dict_encode): distinct valid strings in bytewise
// order on the device, shared by the column, its slices and every result column decoded through it.
struct Utf8Dict {
  GpuContextRef ctx;
  fq_utf8 *raw = nullptr;
  uint64_t size = 0;
  ~Utf8Dict();
  std::string at(uint32_t code) const;   // one entry, through fq_utf8_take
  // fq_utf8_bounds of a literal, remembered: a dictionary never changes, and every pipe of a query lowers the same literals
  std::pair<uint64_t, uint64_t> bounds(const std::string &literal) const;
  // bit `code` = entry `code` LIKE `pattern` (NOT LIKE when `negate`): a UInt8 column of ceil(size / 8) bytes (at least one)
  // from fq_utf8_like, remembered like the bounds.  Pipes read it through an FQ_EXPR_LOOKUP node.
  std::shared_ptr<DataArray> like(const std::string &pattern, bool negate) const;

 private:
  mutable std::mutex mu_;
  mutable std::map<std::string, std::pair<uint64_t, uint64_t>> bounds_;
  mutable std::map<std::pair<std::string, bool>, std::shared_ptr<DataArray>> like_;
  mutable uint64_t like_bytes_ = 0;
};
using Utf8DictRef = std::shared_ptr<const Utf8Dict>;

// ArrayRef (data_array.rs): a device-resident Arrow-layout column, a host Utf8 array (partial aggregate states and
// EXPLAIN text), or a dictionary-encoded Utf8 column: UInt32 codes on the device (with the column's validity) over a
// shared sorted dictionary, decoded lazily when its strings are asked for
class DataArray : public std::enable_shared_from_this<DataArray> {
 public:
  ~DataArray();
  static std::shared_ptr<DataArray> device(GpuContextRef ctx, fq_column *col, std::shared_ptr<DataArray> parent = nullptr);
  static std::shared_ptr<DataArray> alloc(GpuContextRef ctx, DataType t, uint64_t len);
  static std::shared_ptr<DataArray> from_host(GpuContextRef ctx, DataType t, const void *data, uint64_t len);
  // Arrow LSB-first bitmaps (BooleanArray values, validity buffers) <-> the device's byte per row
  static std::shared_ptr<DataArray> from_arrow_bitmap(GpuContextRef ctx, const void *bits, uint64_t bit_offset, uint64_t len);
  std::vector<unsigned char> to_arrow_bitmap() const;   // Boolean arrays only; ceil(len / 8) bytes
  // validity: a Boolean array of the same length (one byte per row, 1 = valid) or null for a NOT NULL array
  void set_validity(std::shared_ptr<DataArray> validity);
  const std::shared_ptr<DataArray> &validity() const { return validity_; }
  uint64_t null_count() const;
  static std::shared_ptr<DataArray> utf8(std::vector<std::string> values);
  // Arrow strings (int32 offsets[len + 1] starting at 0, the bytes, optional validity bytes 1 = valid) uploaded and
  // dictionary-encoded on the device
  static std::shared_ptr<DataArray> utf8_dict(GpuContextRef ctx, const int32_t *offsets, const void *data, uint64_t len,
                                              const unsigned char *valid);
  // a UInt32 codes array (its validity included) read as strings of `dict`
  static std::shared_ptr<DataArray> with_dict(const std::shared_ptr<DataArray> &codes, Utf8DictRef dict);
  DataType data_type() const { return dtype_; }
  uint64_t len() const { return len_; }
  bool is_utf8() const { return dtype_ == FQ_UTF8; }
  bool is_host_utf8() const { return dtype_ == FQ_UTF8 && !dict_; }
  const Utf8DictRef &dict() const { return dict_; }
  fq_column *column() const { return col_; }   // dictionary arrays: the codes
  const std::vector<std::string> &strings() const;   // dictionary arrays: decoded on first use ("" in NULL slots)
  std::shared_ptr<DataArray> slice(uint64_t offset, uint64_t len);   // arrow::compute::limit == slice(0, n)
  void to_host(void *out) const;                                      // len * size bytes
  DataValue value(uint64_t index) const;                              // DataValue::try_from_array
  GpuContextRef ctx() const { return ctx_; }

 private:
  DataArray() = default;
  GpuContextRef ctx_;
  DataType dtype_ = FQ_NULL;
  uint64_t len_ = 0;
  fq_column *col_ = nullptr;
  std::shared_ptr<DataArray> parent_;
  std::shared_ptr<DataArray> validity_;
  mutable std::vector<std::string> strings_;
  Utf8DictRef dict_;
  mutable bool decoded_ = false;
};
using DataArrayRef = std::shared_ptr<DataArray>;

// data_columnar_value.rs:8-30
struct DataColumnarValue {
  bool is_scalar = false;
  DataArrayRef array;
  DataValue scalar;
  static DataColumnarValue Array(DataArrayRef a) { DataColumnarValue c; c.array = std::move(a); return c; }
  static DataColumnarValue Scalar(DataValue v) { DataColumnarValue c; c.is_scalar = true; c.scalar = std::move(v); return c; }
  DataType data_type() const { return is_scalar ? scalar.data_type() : array->data_type(); }
  DataArrayRef to_array(GpuContextRef ctx, uint64_t size) const;   // DataValue::to_array broadcast (data_value.rs:76-112)
};

// datablocks/data_block.rs:10-62
class DataBlock {
 public:
  DataBlock() : schema_(std::make_shared<DataSchema>()) {}
  DataBlock(DataSchemaRef schema, std::vector<DataArrayRef> columns) : schema_(std::move(schema)), columns_(std::move(columns)) {}
  static DataBlock create(DataSchemaRef schema, std::vector<DataArrayRef> columns) { return DataBlock(std::move(schema), std::move(columns)); }
  const DataSchemaRef &schema() const { return schema_; }
  uint64_t num_rows() const { return columns_.empty() ? 0 : columns_[0]->len(); }
  size_t num_columns() const { return columns_.size(); }
  const DataArrayRef &column(size_t i) const { return columns_.at(i); }
  const DataArrayRef &column_by_name(const std::string &name) const { return columns_.at(schema_->index_of(name)); }
  // generated numbers_mt block: no column buffer exists, values are begin + row (fq_source.generated)
  bool generated = false;
  uint64_t numbers_begin = 0, generated_rows = 0;
  uint64_t rows() const { return generated ? generated_rows : num_rows(); }

 private:
  DataSchemaRef schema_;
  std::vector<DataArrayRef> columns_;
};

// device-side array ops (datavalues/data_array_{arithmetic,comparison,logic,aggregate}.rs): one fused
// kernel per call
DataArrayRef data_array_arithmetic_op(GpuContextRef ctx, int op, const DataColumnarValue &l, const DataColumnarValue &r);
DataArrayRef data_array_comparison_op(GpuContextRef ctx, int op, const DataColumnarValue &l, const DataColumnarValue &r);
DataArrayRef data_array_logic_op(GpuContextRef ctx, int op, const DataColumnarValue &l, const DataColumnarValue &r);
DataValue data_array_aggregate_op(GpuContextRef ctx, int op, const DataArrayRef &a);

// ---------------------------------------------------------------------------------------------
// GPU context: owns the fq_ctx and a cache of compiled pipes
// ---------------------------------------------------------------------------------------------
struct PipeHandle {
  GpuContextRef ctx;
  fq_pipe *pipe = nullptr;
  std::vector<DataArrayRef> lookups;   // bit tables bound with fq_pipe_set_lookup: the pipe borrows them
  ~PipeHandle();
};
using PipeRef = std::shared_ptr<PipeHandle>;

class GpuContext : public std::enable_shared_from_this<GpuContext> {
 public:
  static GpuContextRef create(int device);
  ~GpuContext();
  fq_ctx *raw() const { return ctx_; }
  int device() const { return device_; }
  void check(fq_status st) const;   // throws FuseQueryError carrying fq_last_error
  uint64_t launch_count() const { return fq_ctx_launch_count(ctx_); }
  void *stream = nullptr;           // launch stream for everything issued through this context

 private:
  fq_ctx *ctx_ = nullptr;
  int device_ = 0;
};

// The merge point across GPUs (processors/processor_merge.rs:37-66) for rows: every rank's blocks meet, in rank order, on the
// device (fq_group).  One process per GPU; `handle` travels to the peers by whatever the deployment has.
class GpuGroup {
 public:
  GpuGroup(GpuContextRef gpu, int rank, int world, uint64_t row_bytes);
  ~GpuGroup();
  GpuGroup(const GpuGroup &) = delete;
  GpuGroup &operator=(const GpuGroup &) = delete;
  std::string handle() const;                             // 64 bytes
  void connect(const std::vector<std::string> &handles);  // handles[r] = rank r's
  // every rank's columns (same types, `rows` local rows, at most `capacity` on any rank) concatenated in rank order and cut at
  // `limit` (-1: none) -> (columns, rows selected by all ranks as reported in `selected_local`)
  std::pair<std::vector<DataArrayRef>, uint64_t> gather(const std::vector<DataArrayRef> &cols, const std::vector<DataType> &types, uint64_t rows,
                                                        uint64_t selected_local, uint64_t capacity, int64_t limit);
  int rank() const { return rank_; }
  int world() const { return world_; }

 private:
  GpuContextRef gpu_;
  fq_group *raw_ = nullptr;
  int rank_, world_;
};

// ---------------------------------------------------------------------------------------------
// functions — enum Function (functions/function.rs:16-146)
// ---------------------------------------------------------------------------------------------
class Function;
using FunctionRef = std::shared_ptr<Function>;

class Function {
 public:
  enum Kind { Alias, Constant, Variable, Arithmetic, Comparison, Logic, Aggregator, Like };
  Kind kind;
  int op = 0;               // FQ_AR_* / FQ_CMP_* / FQ_LG_* / FQ_AGG_*; Like: 1 = NOT LIKE
  size_t depth = 0;
  std::string name;         // field name / alias
  DataValue value;          // constant value; aggregator state (starts Null, function_aggregator.rs:30)
  FunctionRef left, right;  // children; aggregator / alias argument in `left`

  // constructors named after the reference's try_create functions
  static FunctionRef FieldFunction(const std::string &name);                        // function_field.rs:21-27
  static FunctionRef ConstantFunction(const DataValue &v);                           // function_constant.rs:18-20
  static FunctionRef AliasFunction(const std::string &alias, FunctionRef f);         // function_alias.rs:20-26
  static FunctionRef ArithmeticFunction(int op, const std::vector<FunctionRef> &args);   // function_arithmetic.rs:23-34
  static FunctionRef ComparisonFunction(int op, const std::vector<FunctionRef> &args);   // function_comparison.rs:25-37
  static FunctionRef LogicFunction(int op, const std::vector<FunctionRef> &args);        // function_logic.rs:25-33
  static FunctionRef AggregatorFunction(int op, const std::vector<FunctionRef> &args);   // function_aggregator.rs:25-36
  // `s LIKE 'pattern'` / `s NOT LIKE 'pattern'` (no counterpart in the reference): Boolean, NULL where s is
  static FunctionRef LikeFunction(bool negate, const std::vector<FunctionRef> &args);
  // ScalarFunctionFactory::get, function_factory.rs:17-39
  static FunctionRef factory_get(const std::string &name, const std::vector<FunctionRef> &args);

  FunctionRef clone() const;  // #[derive(Clone)]: deep copy, aggregator state included

  DataType return_type(const DataSchema &input_schema) const;
  bool nullable(const DataSchema &input_schema) const;
  DataColumnarValue eval(GpuContextRef ctx, const DataBlock &block);
  void set_depth(size_t depth);
  void accumulate(GpuContextRef ctx, const DataBlock &block);
  std::vector<DataValue> accumulate_result();
  void merge_state(const std::vector<DataValue> &states);
  DataValue merge_result();
  std::string to_string() const;  // Debug (drives column names)

 private:
  explicit Function(Kind k) : kind(k) {}
  // aggregator: device-resident running state of blocks accumulated since the last sync
  PipeRef agg_pipe_;
  std::string agg_pipe_key_;
  bool agg_pending_ = false;
  void sync_state();
  friend struct Lowering;
};

// ---------------------------------------------------------------------------------------------
// datastreams — SendableDataBlockStream (datastreams/stream.rs:8-9); pull-based, synchronous on the
// host (device work is asynchronous underneath)
// ---------------------------------------------------------------------------------------------
class IDataBlockStream {
 public:
  virtual ~IDataBlockStream() = default;
  virtual std::optional<DataBlock> next() = 0;
};
using SendableDataBlockStream = std::unique_ptr<IDataBlockStream>;

// stream_datablock.rs:13-60
class DataBlockStream : public IDataBlockStream {
 public:
  explicit DataBlockStream(std::vector<DataBlock> blocks) : blocks_(std::move(blocks)) {}
  std::optional<DataBlock> next() override;

 private:
  std::vector<DataBlock> blocks_;
  size_t i_ = 0;
};
// stream_expression.rs:15-50
using ExpressionExecutor = std::function<DataBlock(GpuContextRef, const DataSchemaRef &, const DataBlock &, std::vector<FunctionRef>)>;
class ExpressionStream : public IDataBlockStream {
 public:
  ExpressionStream(GpuContextRef ctx, SendableDataBlockStream input, DataSchemaRef schema, std::vector<FunctionRef> exprs, ExpressionExecutor f)
      : ctx_(std::move(ctx)), input_(std::move(input)), schema_(std::move(schema)), exprs_(std::move(exprs)), func_(std::move(f)) {}
  std::optional<DataBlock> next() override;

 private:
  GpuContextRef ctx_;
  SendableDataBlockStream input_;
  DataSchemaRef schema_;
  std::vector<FunctionRef> exprs_;
  ExpressionExecutor func_;
};
// stream_limit.rs:13-63
class LimitStream : public IDataBlockStream {
 public:
  LimitStream(SendableDataBlockStream input, size_t limit) : input_(std::move(input)), limit_(limit) {}
  std::optional<DataBlock> limit(const DataBlock &block);
  std::optional<DataBlock> next() override;

 private:
  SendableDataBlockStream input_;
  size_t limit_, current_ = 0;
};

// ---------------------------------------------------------------------------------------------
// planners
// ---------------------------------------------------------------------------------------------
// plan_expression.rs:13-29
struct ExpressionPlan {
  enum Kind { Alias, Field, Constant, BinaryExpression, Function, Wildcard } kind = Wildcard;
  std::string name;   // alias / field / operator / function name
  DataValue value;
  std::vector<ExpressionPlan> args;   // Alias: [expr]; Binary: [left, right]; Function: args
  int tree_depth = 1;                 // height of the tree below (and including) this node; the SQL front end bounds it

  static constexpr int kMaxDepth = 128;   // deeper trees are refused: every later walk (to_function, lowering, codegen) recurses
  static ExpressionPlan field(const std::string &n) { ExpressionPlan e; e.kind = Field; e.name = n; return e; }
  static ExpressionPlan constant(const DataValue &v) { ExpressionPlan e; e.kind = Constant; e.value = v; return e; }
  static ExpressionPlan alias(const std::string &a, ExpressionPlan x) {
    ExpressionPlan e; e.kind = Alias; e.name = a; e.tree_depth = x.tree_depth + 1; e.args = {std::move(x)}; return checked(std::move(e));
  }
  static ExpressionPlan binary(ExpressionPlan l, const std::string &op, ExpressionPlan r) {
    ExpressionPlan e; e.kind = BinaryExpression; e.name = op; e.tree_depth = std::max(l.tree_depth, r.tree_depth) + 1;
    e.args = {std::move(l), std::move(r)}; return checked(std::move(e));
  }
  static ExpressionPlan function(const std::string &op, std::vector<ExpressionPlan> a) {
    ExpressionPlan e; e.kind = Function; e.name = op;
    for (const auto &x : a) e.tree_depth = std::max(e.tree_depth, x.tree_depth + 1);
    e.args = std::move(a); return checked(std::move(e));
  }
  static ExpressionPlan checked(ExpressionPlan e) {
    if (e.tree_depth > kMaxDepth) throw FuseQueryError::plan("expression depth more than 128");
    return e;
  }
  static ExpressionPlan wildcard() { return ExpressionPlan(); }

  FunctionRef to_function(size_t depth = 0) const;                 // plan_expression.rs:40-75
  DataField to_field(const DataSchema &input_schema) const;        // :31-38
  bool is_aggregate() const;                                       // :77-89
  std::string to_string() const;                                   // Debug, :92-105
};

struct Partition { std::string name; uint64_t version = 0; };       // datasources/partition.rs:7-11
using Partitions = std::vector<Partition>;

// plan_node.rs:12-23 and the per-node plan structs
struct PlanNode;
using PlanNodeRef = std::shared_ptr<const PlanNode>;
struct PlanNode {
  enum Kind { Empty, Projection, Aggregate, Filter, Limit, Scan, ReadSource, Explain, Select, Sort } kind = Empty;
  PlanNodeRef input;                      // Projection / Aggregate / Filter / Limit input; Explain / Select child plan
  DataSchemaRef schema_;                  // Empty, Projection, Aggregate, Scan (projected), ReadSource
  std::vector<ExpressionPlan> expr;       // Projection exprs / Aggregate aggr_expr / Sort keys (over the input's output columns)
  std::vector<bool> descending;           // Sort: per key
  std::vector<ExpressionPlan> group_expr; // Aggregate
  ExpressionPlan predicate;               // Filter
  size_t n = 0;                           // Limit
  // Scan
  std::string schema_name;
  std::optional<ExpressionPlan> table_args;
  // ReadSource (plan_read_datasource.rs)
  std::string db, table, table_type, description;
  Partitions partitions;

  DataSchemaRef schema() const;           // plan_node.rs:27-39
  const char *name() const;               // :41-53
  std::vector<PlanNode> children_to_plans() const;   // :127-129 (bottom-up, without Select/Explain)
  std::vector<PlanNode> node_to_plans() const;       // :131-133
  static PlanNode plans_to_node(const std::vector<PlanNode> &plans);   // :135-162
  std::string to_string() const;          // Debug, plan_display.rs:16-88
};

// plan_builder.rs:14-143
class PlanBuilder {
 public:
  explicit PlanBuilder(PlanNode plan) : plan_(std::move(plan)) {}
  static PlanBuilder from(const PlanNode &plan) { return PlanBuilder(plan); }
  static PlanBuilder create(DataSchemaRef schema);
  static PlanBuilder empty(bool produce_one_row);
  static PlanBuilder scan(const std::string &schema_name, const std::string &table_name, const DataSchema &table_schema,
                          std::optional<ExpressionPlan> table_args);
  PlanBuilder project(const std::vector<ExpressionPlan> &exprs) const;
  PlanBuilder aggregate(const std::vector<ExpressionPlan> &group_expr, const std::vector<ExpressionPlan> &aggr_expr) const;
  PlanBuilder filter(const ExpressionPlan &expr) const;
  PlanBuilder limit(size_t n) const;
  // ORDER BY (the reference plans no sort: README.md:28); keys are expressions over the input plan's output columns
  PlanBuilder sort(const std::vector<ExpressionPlan> &keys, const std::vector<bool> &descending) const;
  PlanBuilder select() const;
  PlanBuilder explain() const;
  PlanNode build() const { return plan_; }

 private:
  PlanNode plan_;
};

// ---------------------------------------------------------------------------------------------
// datasources
// ---------------------------------------------------------------------------------------------
class FuseQueryContext;
using FuseQueryContextRef = std::shared_ptr<FuseQueryContext>;

// datasources/table.rs:13-22
class ITable {
 public:
  virtual ~ITable() = default;
  virtual std::string name() const = 0;
  virtual DataSchemaRef schema() const = 0;
  virtual PlanNode read_plan(const PlanNode &push_down_plan) const = 0;   // -> ReadSource node
  virtual SendableDataBlockStream read(FuseQueryContextRef ctx, const Partitions &parts) const = 0;
};
using ITableRef = std::shared_ptr<ITable>;

// datasources/system/numbers_table.rs
class NumbersTable : public ITable {
 public:
  NumbersTable();
  static Partitions generate_parts(uint64_t total);   // :29-55
  std::string name() const override { return "numbers_mt"; }
  DataSchemaRef schema() const override { return schema_; }
  PlanNode read_plan(const PlanNode &push_down_plan) const override;   // :68-92
  SendableDataBlockStream read(FuseQueryContextRef ctx, const Partitions &parts) const override;   // :94-96

 private:
  DataSchemaRef schema_;
};

// A table whose columns are resident in HBM (SURVEY §8f rank 2: the ITable the README calls "Remote (S3 or other table
// storage engine)" would land its Arrow column chunks here).  Partitioned and streamed exactly like numbers_mt:
// generate_parts over the row count, partition names "N-start-end", blocks = zero-copy slices of the device columns.
class MemoryTable : public ITable {
 public:
  MemoryTable(std::string db, std::string name, DataSchemaRef schema, std::vector<DataArrayRef> columns);
  std::string name() const override { return name_; }
  DataSchemaRef schema() const override { return schema_; }
  PlanNode read_plan(const PlanNode &push_down_plan) const override;
  SendableDataBlockStream read(FuseQueryContextRef ctx, const Partitions &parts) const override;
  uint64_t num_rows() const { return columns_.empty() ? 0 : columns_[0]->len(); }

 private:
  std::string db_, name_;
  DataSchemaRef schema_;
  std::vector<DataArrayRef> columns_;
};

// datasources/datasource.rs: catalog db -> table
class DataSource {
 public:
  DataSource();
  void add_database(const std::string &db) { dbs_[db]; }
  void add_table(const std::string &db, ITableRef table);
  ITableRef get_table(const std::string &db, const std::string &table) const;

 private:
  std::map<std::string, std::map<std::string, ITableRef>> dbs_;
};

// contexts/context.rs:10-37 + the knobs the device path adds
struct GpuOptions {
  bool fuse = true;              // collapse Source->Filter->(Projection|AggregatePartial)->Limit into one GpuPipeTransform
  bool generated = false;        // numbers_mt: generate in-kernel instead of reading a materialised shard
  uint64_t block_rows = 0;       // rows per DataBlock the source emits; 0 = one block per partition run (the
                                 // reference uses 10 000, numbers_stream.rs:29)
  bool tail_quirk = true;        // reproduce numbers_stream.rs:44-46 (SURVEY F7) for sizes that trigger it
  bool limit_early_exit = true;  // let a LIMIT stop the scan (the reference stops pulling blocks, stream_limit.rs:28-31)
  bool block_quirks = true;      // fused aggregate pipes reproduce SURVEY F8: with a WHERE clause, a Sum whose predicate
                                 // empties one of the reference's 10 000-row blocks fails like the reference does
                                 // ("DataValue to array cannot be NONE NULL"); false = return the merged sum instead
  bool group_by = true;          // execute GROUP BY (hash aggregation); false = ignore it like the reference's pipeline builder
  bool align_runs = false;       // internal: only merge partitions into one device block when block boundaries line up
};
class FuseQueryContext : public std::enable_shared_from_this<FuseQueryContext> {
 public:
  static FuseQueryContextRef create_ctx(size_t worker_threads, std::shared_ptr<DataSource> datasource, GpuContextRef gpu);
  size_t worker_threads;
  GpuOptions options;
  std::string get_current_database() const;
  void set_current_database(const std::string &db);
  ITableRef get_table(const std::string &db, const std::string &table) const;
  std::shared_ptr<DataSource> datasource() const { return datasource_; }
  GpuContextRef gpu() const;     // throws when the context was built without a device (planning-only use)

 private:
  FuseQueryContext() = default;
  mutable std::mutex mu_;
  std::string default_db_ = "default";
  std::shared_ptr<DataSource> datasource_;
  GpuContextRef gpu_;
};

// planners/plan_parser.rs: SQL -> PlanNode
class Planner {
 public:
  PlanNode build_from_sql(FuseQueryContextRef ctx, const std::string &query) const;   // :16-28
};

// optimizers/optimizer.rs:15-32, optimizer_filter_push_down.rs:19-82
class Optimizer {
 public:
  static Optimizer create() { return Optimizer(); }
  PlanNode optimize(const PlanNode &plan) const;
};
class FilterPushDownOptimizer {
 public:
  PlanNode optimize(const PlanNode &plan) const;
};

// ---------------------------------------------------------------------------------------------
// processors + transforms
// ---------------------------------------------------------------------------------------------
// processors/processor.rs:22-58
class IProcessor {
 public:
  virtual ~IProcessor() = default;
  virtual std::string name() const = 0;
  virtual void connect_to(std::shared_ptr<IProcessor> input) = 0;
  virtual SendableDataBlockStream execute() = 0;
};
using IProcessorRef = std::shared_ptr<IProcessor>;

class EmptyProcessor : public IProcessor {   // processor_empty.rs
 public:
  std::string name() const override { return "EmptyProcessor"; }
  void connect_to(IProcessorRef) override;
  SendableDataBlockStream execute() override;
};
class MergeProcessor : public IProcessor {   // processor_merge.rs:16-66
 public:
  std::string name() const override { return "MergeProcessor"; }
  void connect_to(IProcessorRef input) override { list_.push_back(std::move(input)); }
  SendableDataBlockStream execute() override;

 private:
  std::vector<IProcessorRef> list_;
};

#define FUSE_TRANSFORM_COMMON(NAME)                                       \
  std::string name() const override { return NAME; }                     \
  void connect_to(IProcessorRef input) override { input_ = std::move(input); }

class SourceTransform : public IProcessor {   // transform_source.rs:14-53
 public:
  SourceTransform(FuseQueryContextRef ctx, std::string db, std::string table, Partitions partitions)
      : ctx_(std::move(ctx)), db_(std::move(db)), table_(std::move(table)), partitions_(std::move(partitions)) {}
  std::string name() const override { return "SourceTransform"; }
  void connect_to(IProcessorRef) override;
  SendableDataBlockStream execute() override;
  const Partitions &partitions() const { return partitions_; }

 private:
  FuseQueryContextRef ctx_;
  std::string db_, table_;
  Partitions partitions_;
};
class FilterTransform : public IProcessor {   // transform_filter.rs:17-77
 public:
  FilterTransform(FuseQueryContextRef ctx, const ExpressionPlan &predicate);
  FUSE_TRANSFORM_COMMON("FilterTransform")
  static DataBlock expression_executor(GpuContextRef gpu, const DataSchemaRef &schema, const DataBlock &block, std::vector<FunctionRef> funcs);
  SendableDataBlockStream execute() override;

 private:
  FuseQueryContextRef ctx_;
  FunctionRef func_;
  IProcessorRef input_ = std::make_shared<EmptyProcessor>();
};
class ProjectionTransform : public IProcessor {   // transform_projection.rs:16-78
 public:
  ProjectionTransform(FuseQueryContextRef ctx, DataSchemaRef schema, const std::vector<ExpressionPlan> &exprs);
  FUSE_TRANSFORM_COMMON("ProjectionTransform")
  static DataBlock expression_executor(GpuContextRef gpu, const DataSchemaRef &schema, const DataBlock &block, std::vector<FunctionRef> funcs);
  SendableDataBlockStream execute() override;

 private:
  FuseQueryContextRef ctx_;
  std::vector<FunctionRef> funcs_;
  DataSchemaRef schema_;
  IProcessorRef input_ = std::make_shared<EmptyProcessor>();
};
class AggregatePartialTransform : public IProcessor {   // transform_aggregate_partial.rs:18-79
 public:
  AggregatePartialTransform(FuseQueryContextRef ctx, DataSchemaRef schema, const std::vector<ExpressionPlan> &exprs);
  FUSE_TRANSFORM_COMMON("AggregatePartialTransform")
  SendableDataBlockStream execute() override;

 private:
  FuseQueryContextRef ctx_;
  std::vector<FunctionRef> funcs_;
  DataSchemaRef schema_;
  IProcessorRef input_ = std::make_shared<EmptyProcessor>();
};
class AggregateFinalTransform : public IProcessor {   // transform_aggregate_final.rs:18-79
 public:
  AggregateFinalTransform(FuseQueryContextRef ctx, DataSchemaRef schema, const std::vector<ExpressionPlan> &exprs);
  FUSE_TRANSFORM_COMMON("AggregateFinalTransform")
  SendableDataBlockStream execute() override;

 private:
  FuseQueryContextRef ctx_;
  std::vector<FunctionRef> funcs_;
  DataSchemaRef schema_;
  IProcessorRef input_ = std::make_shared<EmptyProcessor>();
};
class LimitTransform : public IProcessor {   // transform_limit.rs:12-43
 public:
  explicit LimitTransform(size_t limit) : limit_(limit) {}
  FUSE_TRANSFORM_COMMON("LimitTransform")
  SendableDataBlockStream execute() override;

 private:
  size_t limit_;
  IProcessorRef input_ = std::make_shared<EmptyProcessor>();
};

// The fused device pipe: Source -> [Filter] -> (Projection | AggregatePartial) [-> Limit] of ONE source
// pipe as one kernel launch per partition run (SURVEY.md §8b).  Emits exactly what the chain it replaces
// would emit to the next processor: the partial-state Utf8/JSON block for aggregates
// (transform_aggregate_partial.rs:61-72) or the filtered + projected (+ limited) rows.
class GpuPipeTransform : public IProcessor {
 public:
  GpuPipeTransform(FuseQueryContextRef ctx, std::string db, std::string table, Partitions partitions,
                   std::optional<ExpressionPlan> predicate, bool is_aggregate, DataSchemaRef schema,
                   std::vector<ExpressionPlan> exprs, std::optional<size_t> limit);
  std::string name() const override { return "GpuPipeTransform"; }
  void connect_to(IProcessorRef) override;
  SendableDataBlockStream execute() override;
  std::string describe() const;   // the chain it stands for, for EXPLAIN

 private:
  FuseQueryContextRef ctx_;
  std::string db_, table_;
  Partitions partitions_;
  std::optional<ExpressionPlan> predicate_;
  bool is_aggregate_;
  DataSchemaRef schema_;
  std::vector<ExpressionPlan> exprs_;
  std::optional<size_t> limit_;
};

// GROUP BY (SURVEY 8 f4).  The reference plans AggregatePlan{group_expr, aggr_expr} (plan_parser.rs:279-308) but
// PipelineBuilder only uses aggr_expr (pipeline_builder.rs:50-65): a GROUP BY query there returns the un-grouped aggregate.
// With GpuOptions.group_by (default on) the plan is executed as written: ONE processor over all partitions — the hash
// table in HBM is the merge point — emitting one block with the plan's schema: the group fields, then the aggregate
// fields, one row per group (row order unspecified).  Arithmetic over aggregates is applied per group exactly like
// merge_result does (function_arithmetic.rs:82-88), as a projection over the exported leaf columns.
class GpuGroupByTransform : public IProcessor {
 public:
  GpuGroupByTransform(FuseQueryContextRef ctx, std::string db, std::string table, Partitions partitions,
                      std::optional<ExpressionPlan> predicate, DataSchemaRef schema, std::vector<ExpressionPlan> group_expr,
                      std::vector<ExpressionPlan> aggr_expr);
  std::string name() const override { return "GpuGroupByTransform"; }
  void connect_to(IProcessorRef) override;
  SendableDataBlockStream execute() override;

 private:
  FuseQueryContextRef ctx_;
  std::string db_, table_;
  Partitions partitions_;
  std::optional<ExpressionPlan> predicate_;
  DataSchemaRef schema_;
  std::vector<ExpressionPlan> group_expr_, aggr_expr_;
};

// ORDER BY: gathers every block of its input, evaluates the key expressions over them, sorts row indexes on the device
// (fq_sort_indices: stable, NULLs first, ASC unless DESC) and emits one block with every column gathered in that order.
// The reference has no sort operator (README.md:28 "[ ] Sorting"); semantics in oracle/sort.py.
class GpuSortTransform : public IProcessor {
 public:
  // `limit`: the LIMIT that follows the sort in the plan, if any — only that many rows are ordered and gathered
  GpuSortTransform(FuseQueryContextRef ctx, std::vector<ExpressionPlan> keys, std::vector<bool> descending, std::optional<size_t> limit = std::nullopt);
  FUSE_TRANSFORM_COMMON("GpuSortTransform")
  SendableDataBlockStream execute() override;

 private:
  FuseQueryContextRef ctx_;
  std::vector<ExpressionPlan> keys_;
  std::vector<bool> descending_;
  std::optional<size_t> limit_;
  IProcessorRef input_ = std::make_shared<EmptyProcessor>();
};

// processors/pipeline.rs:13-135
class Pipeline {
 public:
  using Pipe = std::vector<IProcessorRef>;
  size_t pipe_num() const { return processors_.empty() ? 0 : processors_.back().size(); }
  void add_source(IProcessorRef source);
  void add_simple_transform(const std::function<IProcessorRef()> &f);
  void merge_processor();
  SendableDataBlockStream execute();
  std::string to_string() const;   // Debug, :109-135
  const std::vector<Pipe> &pipes() const { return processors_; }

 private:
  std::vector<Pipe> processors_;
};

// processors/pipeline_builder.rs:16-107
class PipelineBuilder {
 public:
  PipelineBuilder(FuseQueryContextRef ctx, PlanNode plan) : ctx_(std::move(ctx)), plan_(std::move(plan)) {}
  static PipelineBuilder create(FuseQueryContextRef ctx, PlanNode plan) { return PipelineBuilder(std::move(ctx), std::move(plan)); }
  Pipeline build() const;

 private:
  FuseQueryContextRef ctx_;
  PlanNode plan_;
};

// ---------------------------------------------------------------------------------------------
// executors (executors/executor*.rs)
// ---------------------------------------------------------------------------------------------
class IExecutor {
 public:
  virtual ~IExecutor() = default;
  virtual std::string name() const = 0;
  virtual SendableDataBlockStream execute() = 0;
};
class SelectExecutor : public IExecutor {   // executor_select.rs:15-41
 public:
  SelectExecutor(FuseQueryContextRef ctx, PlanNode select_plan) : ctx_(std::move(ctx)), plan_(std::move(select_plan)) {}
  std::string name() const override { return "SelectExecutor"; }
  SendableDataBlockStream execute() override;

 private:
  FuseQueryContextRef ctx_;
  PlanNode plan_;
};
class ExplainExecutor : public IExecutor {   // executor_explain.rs:18-60
 public:
  ExplainExecutor(FuseQueryContextRef ctx, PlanNode explain_plan) : ctx_(std::move(ctx)), plan_(std::move(explain_plan)) {}
  std::string name() const override { return "ExplainExecutor"; }
  SendableDataBlockStream execute() override;

 private:
  FuseQueryContextRef ctx_;
  PlanNode plan_;
};
struct ExecutorFactory {   // executor_factory.rs:12-25
  static std::shared_ptr<IExecutor> get(FuseQueryContextRef ctx, const PlanNode &plan);
};

// What mysql_handler.rs:52-75 does for one query, minus the wire protocol: plan, optimize, execute, drain.
std::vector<DataBlock> execute_sql(FuseQueryContextRef ctx, const std::string &sql);

// servers/mysql/mysql_stream.rs:12-86 minus the socket: the result set a MySQL client would be sent.  Column types
// follow the reference's mapping (every integer -> MYSQL_TYPE_LONG, floats -> MYSQL_TYPE_FLOAT, Utf8 ->
// MYSQL_TYPE_VARCHAR, anything else "Unsupported column type:<type>"); cells are arrow's array_value_to_string
// (decimal integers, shortest round-trip floats without exponent, "" for NULL).  One D2H copy per column per block.
struct MySQLColumn { std::string column; std::string coltype; };
struct MySQLResultSet {
  std::vector<MySQLColumn> columns;
  std::vector<std::vector<std::string>> rows;
};
class MySQLStream {
 public:
  static MySQLStream create(std::vector<DataBlock> blocks) { return MySQLStream(std::move(blocks)); }
  MySQLResultSet execute() const;
 private:
  explicit MySQLStream(std::vector<DataBlock> blocks) : blocks_(std::move(blocks)) {}
  std::vector<DataBlock> blocks_;
};

}  // namespace fuse
