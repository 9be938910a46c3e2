// pipeline.cc — host mirror of src/datasources, src/datastreams, src/transforms, src/processors,
// src/executors and src/contexts for the hot path, plus the fused GpuPipeTransform.
#include <algorithm>
#include <cstring>
#include <list>

#include "host_internal.h"

#include <charconv>
#include <cmath>
#include <type_traits>

namespace fuse {

// ---------------------------------------------------------------------------------------------
// contexts/context.rs
// ---------------------------------------------------------------------------------------------
FuseQueryContextRef FuseQueryContext::create_ctx(size_t worker_threads, std::shared_ptr<DataSource> datasource, GpuContextRef gpu) {
  auto c = std::shared_ptr<FuseQueryContext>(new FuseQueryContext());
  c->worker_threads = worker_threads;
  c->datasource_ = datasource ? std::move(datasource) : std::make_shared<DataSource>();
  c->gpu_ = std::move(gpu);
  return c;
}
std::string FuseQueryContext::get_current_database() const {
  std::lock_guard<std::mutex> lk(mu_);
  return default_db_;
}
void FuseQueryContext::set_current_database(const std::string &db) {
  std::lock_guard<std::mutex> lk(mu_);
  default_db_ = db;
}
ITableRef FuseQueryContext::get_table(const std::string &db, const std::string &table) const { return datasource_->get_table(db, table); }
GpuContextRef FuseQueryContext::gpu() const {
  if (!gpu_) throw FuseQueryError::internal("this FuseQueryContext has no CUDA device bound (planning only); there is no CPU execution path");
  return gpu_;
}

// ---------------------------------------------------------------------------------------------
// datasources
// ---------------------------------------------------------------------------------------------
DataSource::DataSource() {   // datasource.rs:19-32: register system.numbers_mt
  dbs_["system"];
  add_table("system", std::make_shared<NumbersTable>());
}
void DataSource::add_table(const std::string &db, ITableRef table) {
  auto it = dbs_.find(db);
  if (it == dbs_.end()) throw FuseQueryError::internal("Cannot find the database: " + db);
  it->second[table->name()] = std::move(table);
}
ITableRef DataSource::get_table(const std::string &db, const std::string &table) const {
  auto it = dbs_.find(db);
  if (it == dbs_.end()) throw FuseQueryError::internal("Cannot find the database: " + db);
  auto jt = it->second.find(table);
  if (jt == it->second.end()) throw FuseQueryError::internal("Cannot find the table: " + table);
  return jt->second;
}

NumbersTable::NumbersTable() {
  auto s = std::make_shared<DataSchema>();
  s->fields.push_back({"number", FQ_U64, false});   // numbers_table.rs:19-27
  schema_ = s;
}
Partitions NumbersTable::generate_parts(uint64_t total) {   // numbers_table.rs:29-55
  const uint64_t workers = 8;
  uint64_t chunk = total / workers;
  Partitions parts;
  auto name = [&](uint64_t a, uint64_t b) { return std::to_string(total) + "-" + std::to_string(a) + "-" + std::to_string(b); };
  if (chunk == 0) {
    parts.push_back({name(0, total - 1), 0});   // total == 0 underflows exactly like the reference's u64
    return parts;
  }
  uint64_t remain = total % workers;
  for (uint64_t p = 0; p < workers; p++) {
    uint64_t start = p * chunk, end = (p + 1) * chunk - 1;
    if (p == workers - 1 && remain > 0) end += remain;
    parts.push_back({name(start, end), 0});
  }
  return parts;
}
PlanNode NumbersTable::read_plan(const PlanNode &push_down_plan) const {   // :68-92
  uint64_t total = 10000;
  if (push_down_plan.kind == PlanNode::Scan && push_down_plan.table_args) {
    const ExpressionPlan &a = *push_down_plan.table_args;
    if (a.kind == ExpressionPlan::Constant && a.value.some) {
      if (a.value.tag == FQ_U64) total = a.value.u;
      if (a.value.tag == FQ_I64) total = (uint64_t)a.value.i;
    }
  }
  PlanNode p;
  p.kind = PlanNode::ReadSource;
  p.db = "system";
  p.table = name();
  p.table_type = "System";
  p.schema_ = schema_;
  p.partitions = generate_parts(total);
  p.description = "(Read from system.numbers_mt table)";
  return p;
}

// Row ranges a list of partitions emits, in the order NumbersStream::create walks them
// (numbers_stream.rs:27-62).  tail_quirk reproduces :44-46: when a partition holds >= block_size rows and
// is not a multiple of it, its last block ends at block_begin + remain, so the partition emits only
// block_size * (n_blocks - 1) + remain + 1 rows (a contiguous prefix).
struct RowRange { uint64_t begin, rows; };
static std::vector<RowRange> emitted_ranges(const Partitions &parts, bool tail_quirk, bool align_runs = false) {
  std::vector<RowRange> out;
  const uint64_t block_size = 10000;
  for (const auto &part : parts) {
    size_t a = part.name.find('-'), b = part.name.find('-', a + 1);
    if (a == std::string::npos || b == std::string::npos) throw FuseQueryError::internal("bad partition name " + part.name);
    uint64_t begin = strtoull(part.name.c_str() + a + 1, nullptr, 10), end = strtoull(part.name.c_str() + b + 1, nullptr, 10);
    uint64_t count = end - begin + 1;
    uint64_t nblk = count / block_size, remain = count % block_size;
    uint64_t rows = count;
    if (tail_quirk && nblk > 0 && remain > 0) rows = block_size * (nblk - 1) + remain + 1;
    // merging two partitions into one run keeps the reference's block boundaries only if the run so far is whole blocks
    if (!out.empty() && out.back().begin + out.back().rows == begin && (!align_runs || out.back().rows % block_size == 0)) out.back().rows += rows;
    else out.push_back({begin, rows});
  }
  return out;
}

// materialised shards stay resident in HBM across queries (they ARE the table)
struct ShardCache {
  std::mutex mu;
  std::list<std::pair<RowRange, DataArrayRef>> items;
  DataArrayRef get(GpuContextRef gpu, RowRange r) {
    std::lock_guard<std::mutex> lk(mu);
    for (auto it = items.begin(); it != items.end(); ++it) {
      const RowRange &c = it->first;
      if (it->second->ctx() == gpu && c.begin <= r.begin && r.begin + r.rows <= c.begin + c.rows && ((r.begin - c.begin) % 2 == 0)) {
        items.splice(items.begin(), items, it);
        auto &a = items.front().second;
        return (c.begin == r.begin && c.rows == r.rows) ? a : a->slice(r.begin - c.begin, r.rows);
      }
    }
    const uint64_t cap_bytes = 140ull << 30;
    uint64_t held = 0;
    for (auto &kv : items) held += kv.first.rows * 8;
    while (!items.empty() && held + r.rows * 8 > cap_bytes) {
      held -= items.back().first.rows * 8;
      items.pop_back();
    }
    DataArrayRef a = DataArray::alloc(gpu, FQ_U64, r.rows);
    gpu->check(fq_numbers_fill(gpu->raw(), a->column(), 0, r.begin, r.rows, gpu->stream));
    items.emplace_front(r, a);
    return a;
  }
  void clear() {
    std::lock_guard<std::mutex> lk(mu);
    items.clear();
  }
};
static ShardCache &shard_cache() {
  static ShardCache c;
  return c;
}
void numbers_cache_clear() { shard_cache().clear(); }

// NumbersStream (numbers_stream.rs:20-84) emitting device blocks
class NumbersStream : public IDataBlockStream {
 public:
  NumbersStream(FuseQueryContextRef ctx, DataSchemaRef schema, const Partitions &parts) : ctx_(std::move(ctx)), schema_(std::move(schema)) {
    const GpuOptions &o = ctx_->options;
    for (const RowRange &r : emitted_ranges(parts, o.tail_quirk, o.align_runs)) {
      if (o.block_rows == 0) { blocks_.push_back({r, r}); continue; }
      for (uint64_t off = 0; off < r.rows; off += o.block_rows) blocks_.push_back({{r.begin + off, std::min(o.block_rows, r.rows - off)}, r});
    }
  }
  std::optional<DataBlock> next() override {
    if (i_ >= blocks_.size()) return std::nullopt;
    const auto &[blk, run] = blocks_[i_++];
    if (ctx_->options.generated) {
      DataBlock b(schema_, {});
      b.generated = true;
      b.numbers_begin = blk.begin;
      b.generated_rows = blk.rows;
      return b;
    }
    // materialise the whole run once, hand out slices (16-byte aligned when the offset is even)
    DataArrayRef whole = shard_cache().get(ctx_->gpu(), run);
    DataArrayRef col;
    uint64_t off = blk.begin - run.begin;
    if (off == 0 && blk.rows == run.rows) col = whole;
    else if (off % 2 == 0) col = whole->slice(off, blk.rows);
    else col = shard_cache().get(ctx_->gpu(), blk);
    return DataBlock(schema_, {col});
  }

 private:
  FuseQueryContextRef ctx_;
  DataSchemaRef schema_;
  std::vector<std::pair<RowRange, RowRange>> blocks_;
  size_t i_ = 0;
};
SendableDataBlockStream NumbersTable::read(FuseQueryContextRef ctx, const Partitions &parts) const {
  return std::make_unique<NumbersStream>(std::move(ctx), schema_, parts);
}

// ---- MemoryTable ----
MemoryTable::MemoryTable(std::string db, std::string name, DataSchemaRef schema, std::vector<DataArrayRef> columns)
    : db_(std::move(db)), name_(std::move(name)), schema_(std::move(schema)), columns_(std::move(columns)) {
  if (schema_->fields.size() != columns_.size()) throw FuseQueryError::internal("MemoryTable: schema and columns differ in length");
  for (size_t i = 0; i < columns_.size(); i++) {
    if (columns_[i]->len() != columns_[0]->len()) throw FuseQueryError::internal("MemoryTable: columns differ in length");
    if (columns_[i]->data_type() != schema_->fields[i].data_type) throw FuseQueryError::internal("MemoryTable: column type differs from the schema");
  }
}
PlanNode MemoryTable::read_plan(const PlanNode &) const {
  PlanNode p;
  p.kind = PlanNode::ReadSource;
  p.db = db_;
  p.table = name_;
  p.table_type = "Memory";
  p.schema_ = schema_;
  if (num_rows() > 0) p.partitions = NumbersTable::generate_parts(num_rows());
  p.description = "(Read from " + name_ + " table)";
  return p;
}
namespace {
class MemoryStream : public IDataBlockStream {
 public:
  MemoryStream(FuseQueryContextRef ctx, DataSchemaRef schema, std::vector<DataArrayRef> cols, const Partitions &parts)
      : schema_(std::move(schema)), cols_(std::move(cols)) {
    // no tail quirk here: that is a NumbersStream bug, not a property of tables
    for (const RowRange &r : emitted_ranges(parts, false, ctx->options.align_runs)) {
      const uint64_t step = ctx->options.block_rows ? ctx->options.block_rows : r.rows;
      for (uint64_t off = 0; off < r.rows; off += step) blocks_.push_back({r.begin + off, std::min(step, r.rows - off)});
    }
  }
  std::optional<DataBlock> next() override {
    if (i_ >= blocks_.size()) return std::nullopt;
    const RowRange b = blocks_[i_++];
    std::vector<DataArrayRef> out;
    for (auto &c : cols_) out.push_back((b.begin == 0 && b.rows == c->len()) ? c : c->slice(b.begin, b.rows));
    return DataBlock(schema_, out);
  }

 private:
  DataSchemaRef schema_;
  std::vector<DataArrayRef> cols_;
  std::vector<RowRange> blocks_;
  size_t i_ = 0;
};
}  // namespace
SendableDataBlockStream MemoryTable::read(FuseQueryContextRef ctx, const Partitions &parts) const {
  return std::make_unique<MemoryStream>(std::move(ctx), schema_, columns_, parts);
}

// ---------------------------------------------------------------------------------------------
// datastreams
// ---------------------------------------------------------------------------------------------
std::optional<DataBlock> DataBlockStream::next() {
  if (i_ >= blocks_.size()) return std::nullopt;
  return blocks_[i_++];
}
std::optional<DataBlock> ExpressionStream::next() {   // stream_expression.rs:38-50: exprs are cloned per block
  auto b = input_->next();
  if (!b) return std::nullopt;
  std::vector<FunctionRef> clones;
  for (auto &f : exprs_) clones.push_back(f->clone());
  return func_(ctx_, schema_, *b, std::move(clones));
}
std::optional<DataBlock> LimitStream::limit(const DataBlock &block) {   // stream_limit.rs:28-48
  uint64_t rows = block.rows();
  if (current_ == limit_) return std::nullopt;
  if (current_ + rows < limit_) {
    current_ += rows;
    return block;
  }
  uint64_t keep = limit_ - current_;
  current_ = limit_;
  if (block.generated) {
    DataBlock b = block;
    b.generated_rows = std::min(keep, block.generated_rows);
    return b;
  }
  std::vector<DataArrayRef> cols;
  for (size_t i = 0; i < block.num_columns(); i++) cols.push_back(block.column(i)->slice(0, std::min<uint64_t>(keep, block.column(i)->len())));
  return DataBlock(block.schema(), cols);
}
std::optional<DataBlock> LimitStream::next() {
  auto b = input_->next();
  if (!b) return std::nullopt;
  return limit(*b);
}

namespace {
// ChannelStream fed by MergeProcessor: blocks of input 0, then input 1, ... (one of the arrival orders the
// reference's mpsc fan-in can produce; processor_merge.rs:45-63)
class ConcatStream : public IDataBlockStream {
 public:
  explicit ConcatStream(std::vector<IProcessorRef> inputs) : inputs_(std::move(inputs)) {}
  std::optional<DataBlock> next() override {
    for (;;) {
      if (!cur_) {
        if (i_ >= inputs_.size()) return std::nullopt;
        cur_ = inputs_[i_++]->execute();
      }
      auto b = cur_->next();
      if (b) return b;
      cur_.reset();
    }
  }

 private:
  std::vector<IProcessorRef> inputs_;
  size_t i_ = 0;
  SendableDataBlockStream cur_;
};
}  // namespace

// ---------------------------------------------------------------------------------------------
// processors
// ---------------------------------------------------------------------------------------------
void EmptyProcessor::connect_to(IProcessorRef) { throw FuseQueryError::internal("Cannot call EmptyProcessor connect_to"); }
SendableDataBlockStream EmptyProcessor::execute() { return std::make_unique<DataBlockStream>(std::vector<DataBlock>{}); }

SendableDataBlockStream MergeProcessor::execute() {
  if (list_.empty()) throw FuseQueryError::internal("Merge processor cannot be zero");
  if (list_.size() == 1) return list_[0]->execute();
  return std::make_unique<ConcatStream>(list_);
}

void SourceTransform::connect_to(IProcessorRef) { throw FuseQueryError::internal("Cannot call SourceTransform connect_to"); }
SendableDataBlockStream SourceTransform::execute() { return ctx_->get_table(db_, table_)->read(ctx_, partitions_); }

FilterTransform::FilterTransform(FuseQueryContextRef ctx, const ExpressionPlan &predicate) : ctx_(std::move(ctx)) {
  if (predicate.is_aggregate())   // transform_filter.rs:23-29
    throw FuseQueryError::internal("Aggregate function " + predicate.to_string() + " is found in WHERE in query");
  func_ = predicate.to_function();
}
DataBlock FilterTransform::expression_executor(GpuContextRef gpu, const DataSchemaRef &, const DataBlock &block, std::vector<FunctionRef> funcs) {
  // predicate -> BooleanArray -> filter_record_batch over every column (transform_filter.rs:38-55), fused:
  // one compaction kernel that evaluates the predicate and gathers all columns of the kept rows
  std::vector<FunctionRef> fields;
  std::vector<const Function *> raw;
  for (const auto &f : block.schema()->fields) fields.push_back(Function::FieldFunction(f.name));
  for (auto &f : fields) raw.push_back(f.get());
  ProjectResult r = run_project(gpu, block, funcs[0].get(), raw, -1, false);
  return DataBlock(block.schema(), r.columns);
}
SendableDataBlockStream FilterTransform::execute() {
  return std::make_unique<ExpressionStream>(ctx_->gpu(), input_->execute(), std::make_shared<DataSchema>(), std::vector<FunctionRef>{func_->clone()},
                                            FilterTransform::expression_executor);
}

ProjectionTransform::ProjectionTransform(FuseQueryContextRef ctx, DataSchemaRef schema, const std::vector<ExpressionPlan> &exprs)
    : ctx_(std::move(ctx)), schema_(std::move(schema)) {
  for (const auto &e : exprs)
    if (e.is_aggregate()) throw FuseQueryError::internal("Unsupported aggregator function: " + e.to_string());   // transform_projection.rs:24-31
  for (const auto &e : exprs) funcs_.push_back(e.to_function());
}
DataBlock ProjectionTransform::expression_executor(GpuContextRef gpu, const DataSchemaRef &projected_schema, const DataBlock &block,
                                                   std::vector<FunctionRef> funcs) {
  // every expression of the projection in ONE kernel (the reference evaluates them one by one, :51-55)
  std::vector<const Function *> raw;
  for (auto &f : funcs) raw.push_back(f.get());
  ProjectResult r = run_project(gpu, block, nullptr, raw, -1, false);
  return DataBlock(projected_schema, r.columns);
}
SendableDataBlockStream ProjectionTransform::execute() {
  std::vector<FunctionRef> clones;
  for (auto &f : funcs_) clones.push_back(f->clone());
  return std::make_unique<ExpressionStream>(ctx_->gpu(), input_->execute(), schema_, std::move(clones), ProjectionTransform::expression_executor);
}

AggregatePartialTransform::AggregatePartialTransform(FuseQueryContextRef ctx, DataSchemaRef schema, const std::vector<ExpressionPlan> &exprs)
    : ctx_(std::move(ctx)), schema_(std::move(schema)) {
  for (const auto &e : exprs) funcs_.push_back(e.to_function());
}
static DataBlock partial_state_block(const DataSchemaRef &schema, std::vector<FunctionRef> &funcs) {
  // transform_aggregate_partial.rs:61-72: one Utf8 column, row i = JSON of DataValue::Struct(states of expr i)
  std::vector<std::string> rows;
  for (auto &f : funcs) rows.push_back(DataValue::Struct(f->accumulate_result()).to_json());
  return DataBlock(schema, {DataArray::utf8(std::move(rows))});
}
SendableDataBlockStream AggregatePartialTransform::execute() {
  std::vector<FunctionRef> funcs;
  for (auto &f : funcs_) funcs.push_back(f->clone());
  auto stream = input_->execute();
  GpuContextRef gpu = ctx_->gpu();
  while (auto block = stream->next())   // :53-59
    for (auto &f : funcs) f->accumulate(gpu, *block);
  return std::make_unique<DataBlockStream>(std::vector<DataBlock>{partial_state_block(schema_, funcs)});
}

AggregateFinalTransform::AggregateFinalTransform(FuseQueryContextRef ctx, DataSchemaRef schema, const std::vector<ExpressionPlan> &exprs)
    : ctx_(std::move(ctx)), schema_(std::move(schema)) {
  for (const auto &e : exprs) funcs_.push_back(e.to_function());
}
SendableDataBlockStream AggregateFinalTransform::execute() {   // transform_aggregate_final.rs:50-78
  std::vector<FunctionRef> funcs;
  for (auto &f : funcs_) funcs.push_back(f->clone());
  auto stream = input_->execute();
  while (auto block = stream->next()) {
    for (size_t i = 0; i < funcs.size(); i++) {
      DataValue v = block->column(0)->value(i);
      if (v.tag == FQ_UTF8 && v.some) {
        DataValue states = DataValue::from_json(v.s);
        if (states.tag == FQ_STRUCT) funcs[i]->merge_state(states.items);
      }
    }
  }
  std::vector<DataArrayRef> arrays;
  GpuContextRef gpu = ctx_->gpu();
  for (auto &f : funcs) arrays.push_back(DataColumnarValue::Scalar(f->merge_result()).to_array(gpu, 1));
  return std::make_unique<DataBlockStream>(std::vector<DataBlock>{DataBlock(schema_, arrays)});
}

SendableDataBlockStream LimitTransform::execute() { return std::make_unique<LimitStream>(input_->execute(), limit_); }

// ---------------------------------------------------------------------------------------------
// GpuSortTransform — ORDER BY (no counterpart in the reference: README.md:28 "[ ] Sorting")
// ---------------------------------------------------------------------------------------------
GpuSortTransform::GpuSortTransform(FuseQueryContextRef ctx, std::vector<ExpressionPlan> keys, std::vector<bool> descending, std::optional<size_t> limit)
    : ctx_(std::move(ctx)), keys_(std::move(keys)), descending_(std::move(descending)), limit_(limit) {
  descending_.resize(keys_.size(), false);
}
SendableDataBlockStream GpuSortTransform::execute() {
  GpuContextRef gpu = ctx_->gpu();
  auto stream = input_->execute();
  std::vector<DataBlock> blocks;
  DataSchemaRef schema;
  while (auto block = stream->next()) {
    if (!schema) schema = block->schema();
    if (block->num_rows() > 0) blocks.push_back(*block);
  }
  if (blocks.empty()) return std::make_unique<DataBlockStream>(std::vector<DataBlock>{});
  const size_t n_cols = blocks[0].num_columns();
  uint64_t n = 0;
  for (const auto &b : blocks) n += b.num_rows();
  if (n >= (1ull << 32)) throw FuseQueryError::internal("Unsupported on the device path: ORDER BY over 2^32 rows or more");
  // every block of the input as one block (a sort is a pipeline breaker)
  std::vector<DataArrayRef> cols(n_cols);
  for (size_t c = 0; c < n_cols; c++) {
    if (blocks[0].column(c)->is_host_utf8()) throw FuseQueryError::internal("Unsupported on the device path: ORDER BY over a block with a Utf8 column");
    if (blocks.size() == 1) {
      cols[c] = blocks[0].column(c);
      continue;
    }
    // a dictionary column is concatenated as its codes: every block must carry the same dictionary
    const Utf8DictRef dict = blocks[0].column(c)->dict();
    bool nullable = false;
    for (const auto &b : blocks) {
      nullable = nullable || b.column(c)->validity();
      if (b.column(c)->dict() != dict) throw FuseQueryError::internal("Unsupported on the device path: ORDER BY over Utf8 blocks with different dictionaries");
    }
    cols[c] = DataArray::alloc(gpu, dict ? (DataType)FQ_U32 : blocks[0].column(c)->data_type(), n);
    DataArrayRef valid = nullable ? DataArray::alloc(gpu, FQ_BOOL, n) : nullptr;
    uint64_t at = 0;
    for (const auto &b : blocks) {
      const DataArrayRef &src = b.column(c);
      gpu->check(fq_column_copy(gpu->raw(), cols[c]->column(), at, src->column(), 0, src->len(), gpu->stream));
      if (valid) {
        DataArrayRef v = src->validity();
        if (!v) {   // a NOT NULL piece of a nullable column: all ones
          std::vector<unsigned char> ones(src->len(), 1);
          v = DataArray::from_host(gpu, FQ_BOOL, ones.data(), src->len());
        }
        gpu->check(fq_column_copy(gpu->raw(), valid->column(), at, v->column(), 0, src->len(), gpu->stream));
        gpu->check(fq_stream_synchronize(gpu->raw(), gpu->stream));   // `v` may be a temporary
      }
      at += src->len();
    }
    if (valid) cols[c]->set_validity(valid);
    if (dict) cols[c] = DataArray::with_dict(cols[c], dict);
  }
  gpu->check(fq_stream_synchronize(gpu->raw(), gpu->stream));
  DataBlock all(schema, cols);
  // the keys: expressions over the block's columns, all in one projection launch
  std::vector<FunctionRef> funcs;
  std::vector<const Function *> raw;
  for (const auto &k : keys_) funcs.push_back(k.to_function());
  for (auto &f : funcs) raw.push_back(f.get());
  ProjectResult keys = run_project(gpu, all, nullptr, raw, -1, false);
  std::vector<const fq_column *> key_cols;
  std::vector<uint8_t> desc;
  for (size_t k = 0; k < keys.columns.size(); k++) {
    key_cols.push_back(keys.columns[k]->column());
    desc.push_back(descending_[k] ? 1 : 0);
  }
  // with a LIMIT behind the sort only its rows are ordered (radix select when one NOT NULL key decides) and gathered
  uint64_t out_rows = limit_ ? std::min<uint64_t>(*limit_, n) : n;
  DataArrayRef rows = DataArray::alloc(gpu, FQ_U32, std::max<uint64_t>(out_rows, 1));
  if (limit_)
    gpu->check(fq_sort_indices_limit(gpu->raw(), key_cols.data(), desc.data(), (int32_t)key_cols.size(), n, *limit_, rows->column(), &out_rows, gpu->stream));
  else
    gpu->check(fq_sort_indices(gpu->raw(), key_cols.data(), desc.data(), (int32_t)key_cols.size(), n, rows->column(), gpu->stream));
  if (out_rows == 0) return std::make_unique<DataBlockStream>(std::vector<DataBlock>{});
  std::vector<DataArrayRef> sorted(n_cols);
  for (size_t c = 0; c < n_cols; c++) {
    const Utf8DictRef &dict = cols[c]->dict();
    sorted[c] = DataArray::alloc(gpu, dict ? (DataType)FQ_U32 : cols[c]->data_type(), out_rows);
    DataArrayRef valid = cols[c]->validity() ? DataArray::alloc(gpu, FQ_BOOL, out_rows) : nullptr;
    gpu->check(fq_column_take(gpu->raw(), cols[c]->column(), rows->column(), out_rows, sorted[c]->column(), valid ? valid->column() : nullptr, gpu->stream));
    if (valid) sorted[c]->set_validity(valid);
    if (dict) sorted[c] = DataArray::with_dict(sorted[c], dict);
  }
  gpu->check(fq_stream_synchronize(gpu->raw(), gpu->stream));
  return std::make_unique<DataBlockStream>(std::vector<DataBlock>{DataBlock(schema, sorted)});
}

// ---------------------------------------------------------------------------------------------
// GpuPipeTransform
// ---------------------------------------------------------------------------------------------
GpuPipeTransform::GpuPipeTransform(FuseQueryContextRef ctx, std::string db, std::string table, Partitions partitions,
                                   std::optional<ExpressionPlan> predicate, bool is_aggregate, DataSchemaRef schema,
                                   std::vector<ExpressionPlan> exprs, std::optional<size_t> limit)
    : ctx_(std::move(ctx)), db_(std::move(db)), table_(std::move(table)), partitions_(std::move(partitions)), predicate_(std::move(predicate)),
      is_aggregate_(is_aggregate), schema_(std::move(schema)), exprs_(std::move(exprs)), limit_(limit) {
  // the same construction-time checks as the transforms it replaces
  if (predicate_ && predicate_->is_aggregate())
    throw FuseQueryError::internal("Aggregate function " + predicate_->to_string() + " is found in WHERE in query");
  if (!is_aggregate_)
    for (const auto &e : exprs_)
      if (e.is_aggregate()) throw FuseQueryError::internal("Unsupported aggregator function: " + e.to_string());
}
void GpuPipeTransform::connect_to(IProcessorRef) { throw FuseQueryError::internal("Cannot call GpuPipeTransform connect_to"); }
std::string GpuPipeTransform::describe() const {
  std::string s = "SourceTransform";
  if (predicate_) s += " -> FilterTransform";
  s += is_aggregate_ ? " -> AggregatePartialTransform" : " -> ProjectionTransform";
  if (limit_) s += " -> LimitTransform";
  return s;
}

// rows [off, off + rows) of a device block (a view; generated blocks just move their first number)
static DataBlock slice_block(const DataBlock &b, uint64_t off, uint64_t rows) {
  if (b.generated) {
    DataBlock s = b;
    s.numbers_begin = b.numbers_begin + off;
    s.generated_rows = rows;
    return s;
  }
  std::vector<DataArrayRef> cols;
  for (size_t i = 0; i < b.num_columns(); i++) cols.push_back(b.column(i)->slice(off, rows));
  return DataBlock(b.schema(), cols);
}

static void collect_leaves(const Function &f, std::vector<const Function *> *out);
// states of one select expression in accumulate_result order (function_arithmetic.rs:69-75)
static void collect_states(const Function &f, const std::map<const Function *, DataValue> &leaf, std::vector<DataValue> *out) {
  switch (f.kind) {
    case Function::Alias: collect_states(*f.left, leaf, out); return;
    case Function::Constant: out->push_back(f.value); return;
    case Function::Aggregator: out->push_back(leaf.at(&f)); return;
    case Function::Arithmetic:
      collect_states(*f.left, leaf, out);
      collect_states(*f.right, leaf, out);
      return;
    case Function::Variable: throw FuseQueryError::internal("Unsupported aggregate operation for function field");
    case Function::Comparison:
      throw FuseQueryError::internal(std::string("Unsupported aggregate operation for function ") + (const char *[]){"=", "<", "<=", ">", ">="}[f.op % 5]);
    case Function::Like: throw FuseQueryError::internal(std::string("Unsupported aggregate operation for function ") + (f.op ? "NOT LIKE" : "LIKE"));
    default: throw FuseQueryError::internal(std::string("Unsupported aggregate operation for function ") + (f.op == FQ_LG_AND ? "and" : "or"));
  }
}
static void collect_leaves(const Function &f, std::vector<const Function *> *out) {
  if (f.kind == Function::Aggregator) { out->push_back(&f); return; }
  if (f.left) collect_leaves(*f.left, out);
  if (f.right) collect_leaves(*f.right, out);
}

SendableDataBlockStream GpuPipeTransform::execute() {
  GpuContextRef gpu = ctx_->gpu();
  ITableRef table = ctx_->get_table(db_, table_);
  // the source emits one device block per contiguous run of this pipe's partitions
  FunctionRef pred = predicate_ ? predicate_->to_function() : nullptr;
  std::vector<FunctionRef> funcs;
  for (const auto &e : exprs_) funcs.push_back(e.to_function());
  // SURVEY F8: per-block Sum folding of the reference is observable when a WHERE clause can empty a block
  bool track_blocks = false;
  if (is_aggregate_ && pred && ctx_->options.block_quirks) {
    std::vector<const Function *> ls;
    for (auto &f : funcs) collect_leaves(*f, &ls);
    for (const Function *l : ls) track_blocks = track_blocks || l->op == FQ_AGG_SUM;
  }
  // the pipe reads whole runs of partitions; the context's options are restored even when read() throws (bad partition name)
  struct OptionsGuard {
    FuseQueryContextRef c;
    GpuOptions saved;
    explicit OptionsGuard(FuseQueryContextRef ctx) : c(std::move(ctx)), saved(c->options) {}
    ~OptionsGuard() { c->options = saved; }
  };
  SendableDataBlockStream source;
  {
    OptionsGuard guard(ctx_);
    ctx_->options.block_rows = 0;
    // runs keep the reference's block boundaries whenever they are observable: Sum under WHERE (F8), errors under LIMIT
    ctx_->options.align_runs = track_blocks || (!is_aggregate_ && limit_ && ctx_->options.block_quirks);
    source = table->read(ctx_, partitions_);
  }

  if (is_aggregate_) {
    // one fused pipe per FQ_MAX_EXPRS select expressions (almost always exactly one)
    struct Part { PipeRef pipe; Lowering lw; std::vector<const Function *> funcs, leaves; };
    std::vector<Part> parts((funcs.size() + FQ_MAX_EXPRS - 1) / FQ_MAX_EXPRS);
    for (size_t i = 0; i < funcs.size(); i++) parts[i / FQ_MAX_EXPRS].funcs.push_back(funcs[i].get());
    std::vector<const Function *> leaves;
    for (auto &f : funcs) collect_leaves(*f, &leaves);
    for (auto &pt : parts)
      for (const Function *f : pt.funcs) collect_leaves(*f, &pt.leaves);
    int launches = 0;
    while (auto block = source->next()) {
      for (auto &pt : parts) {
        if (!pt.pipe) {
          if (block->generated) pt.lw.column_of(*block, block->schema()->fields[0].name);
          int p = pred ? pt.lw.lower(*pred, *block) : -1;
          std::vector<int> roots;
          for (const Function *f : pt.funcs) roots.push_back(pt.lw.lower(*f, *block));
          fq_pipe_desc d = pt.lw.desc(FQ_PIPE_AGGREGATE, p, roots);
          pt.pipe = compile_pipe(gpu, pt.lw, d);
        }
        BoundSource bs;
        bind_source(pt.lw, *block, &bs);
        gpu->check(fq_pipe_launch_aggregate(gpu->raw(), pt.pipe->pipe, &bs.src,
                                            (launches > 0 ? FQ_RUN_ACCUMULATE : 0) | (track_blocks ? FQ_RUN_BLOCK_STATS : 0), gpu->stream));
      }
      launches++;
    }
    std::map<const Function *, DataValue> leaf_state;
    for (const Function *l : leaves) leaf_state[l] = DataValue::Null();
    for (auto &pt : parts) {
      if (!pt.pipe) continue;
      std::vector<fq_value> st(pt.leaves.size() + 1);
      int32_t n = 0;
      uint64_t sel = 0;
      gpu->check(fq_pipe_fetch_aggregate(gpu->raw(), pt.pipe->pipe, st.data(), (int32_t)st.size(), &n, &sel));
      if (track_blocks) {
        uint64_t blocks = 0, empty = 0;
        gpu->check(fq_pipe_fetch_block_stats(gpu->raw(), pt.pipe->pipe, &blocks, &empty));
        // function_aggregator.rs:88-97: state = state + arrow_sum(block); the second block onwards goes through
        // DataValue::to_array, which refuses Type(None) (data_value.rs:104-109) — on either side of the add
        if (blocks >= 2 && empty > 0) throw FuseQueryError::internal("DataValue to array cannot be NONE NULL");
      }
      std::vector<int32_t> nodes(pt.leaves.size() + 1);
      int32_t nn = 0;
      gpu->check(fq_pipe_aggregator_nodes(gpu->raw(), pt.pipe->pipe, nodes.data(), (int32_t)nodes.size(), &nn));
      for (const Function *l : pt.leaves) {
        int node = pt.lw.node_of.at(l);
        for (int k = 0; k < nn; k++)
          if (nodes[k] == node) leaf_state[l] = pt.lw.decode_leaf(*l, DataValue::from_abi(st[k]));
      }
    }
    std::vector<std::string> rows;
    for (auto &f : funcs) {
      std::vector<DataValue> states;
      collect_states(*f, leaf_state, &states);
      rows.push_back(DataValue::Struct(states).to_json());
    }
    return std::make_unique<DataBlockStream>(std::vector<DataBlock>{DataBlock(schema_, {DataArray::utf8(std::move(rows))})});
  }

  // projection (+ filter, + limit): one compaction/projection launch per run, rows in order
  std::vector<const Function *> raw;
  for (auto &f : funcs) raw.push_back(f.get());
  std::vector<DataBlock> out;
  size_t taken = 0;
  const bool exact_errors = limit_ && ctx_->options.block_quirks;
  while (auto block = source->next()) {
    if (limit_ && taken == *limit_) break;   // LimitStream ends the pipe (stream_limit.rs:30-31)
    int64_t remaining = limit_ ? (int64_t)(*limit_ - taken) : -1;
    std::string deferred;
    ProjectResult r = run_project(gpu, *block, pred.get(), raw, remaining, ctx_->options.limit_early_exit, exact_errors ? &deferred : nullptr);
    if (exact_errors) {
      // The reference pulls this pipe's 10 000-row blocks one by one: FilterTransform evaluates the predicate over the whole
      // block, ProjectionTransform every kept row of it (transform_projection.rs:45-56), and only then LimitStream cuts
      // (stream_limit.rs:28-48).  LimitStream::poll_next polls its input BEFORE it looks at its counter (:58-62), so the
      // block after the one that completes the limit is still pulled — filtered, projected, and its error passed on —
      // before the stream ends.  The fused kernel evaluates the predicate over rows the reference never pulls and projects
      // only the rows it writes, so errors are settled here over exactly the reference's rows: everything up to the end of
      // the block FOLLOWING the one that holds the limit-th kept row.
      const uint64_t rows = block->rows();
      const uint64_t blk_end = r.limit_reached ? std::min<uint64_t>(rows, (r.limit_row / 10000 + 2) * 10000) : rows;
      if (!deferred.empty()) {
        if (!r.limit_reached) throw FuseQueryError(FuseQueryError::Internal, deferred);
        run_project(gpu, slice_block(*block, 0, blk_end), pred.get(), raw, -1, false);            // throws iff the error is inside
      } else if (r.limit_reached && r.limit_row + 1 < blk_end) {
        run_project(gpu, slice_block(*block, r.limit_row + 1, blk_end - r.limit_row - 1), pred.get(), raw, -1, false);
      }
    }
    taken += r.rows_written;
    out.push_back(DataBlock(schema_, r.columns));
  }
  return std::make_unique<DataBlockStream>(std::move(out));
}

// ---------------------------------------------------------------------------------------------
// GpuGroupByTransform
// ---------------------------------------------------------------------------------------------
GpuGroupByTransform::GpuGroupByTransform(FuseQueryContextRef ctx, std::string db, std::string table, Partitions partitions,
                                         std::optional<ExpressionPlan> predicate, DataSchemaRef schema, std::vector<ExpressionPlan> group_expr,
                                         std::vector<ExpressionPlan> aggr_expr)
    : ctx_(std::move(ctx)), db_(std::move(db)), table_(std::move(table)), partitions_(std::move(partitions)), predicate_(std::move(predicate)),
      schema_(std::move(schema)), group_expr_(std::move(group_expr)), aggr_expr_(std::move(aggr_expr)) {
  if (predicate_ && predicate_->is_aggregate())
    throw FuseQueryError::internal("Aggregate function " + predicate_->to_string() + " is found in WHERE in query");
  for (const auto &k : group_expr_)
    if (k.is_aggregate()) throw FuseQueryError::internal("Aggregate function " + k.to_string() + " is found in GROUP BY in query");
  if (group_expr_.size() > (size_t)FQ_MAX_KEYS) throw FuseQueryError::internal("Unsupported on the device path: more than 4 GROUP BY expressions");
  if (aggr_expr_.size() > (size_t)FQ_MAX_EXPRS) throw FuseQueryError::internal("Unsupported on the device path: more than 8 aggregate expressions in a GROUP BY");
}
void GpuGroupByTransform::connect_to(IProcessorRef) { throw FuseQueryError::internal("Cannot call GpuGroupByTransform connect_to"); }

// the select expression with every Aggregator leaf replaced by a field of the exported leaf block
static FunctionRef over_leaves(const Function &f, const std::map<const Function *, std::string> &leaf_name) {
  switch (f.kind) {
    case Function::Aggregator: return Function::FieldFunction(leaf_name.at(&f));
    case Function::Alias: return over_leaves(*f.left, leaf_name);
    case Function::Constant: return Function::ConstantFunction(f.value);
    case Function::Arithmetic: return Function::ArithmeticFunction(f.op, {over_leaves(*f.left, leaf_name), over_leaves(*f.right, leaf_name)});
    case Function::Variable: throw FuseQueryError::internal("Unsupported aggregate operation for function field");
    case Function::Comparison:
      throw FuseQueryError::internal(std::string("Unsupported aggregate operation for function ") + (const char *[]){"=", "<", "<=", ">", ">="}[f.op % 5]);
    case Function::Like: throw FuseQueryError::internal(std::string("Unsupported aggregate operation for function ") + (f.op ? "NOT LIKE" : "LIKE"));
    default: throw FuseQueryError::internal(std::string("Unsupported aggregate operation for function ") + (f.op == FQ_LG_AND ? "and" : "or"));
  }
}

SendableDataBlockStream GpuGroupByTransform::execute() {
  GpuContextRef gpu = ctx_->gpu();
  ITableRef table = ctx_->get_table(db_, table_);
  FunctionRef pred = predicate_ ? predicate_->to_function() : nullptr;
  std::vector<FunctionRef> keys, funcs;
  for (const auto &e : group_expr_) keys.push_back(e.to_function());
  for (const auto &e : aggr_expr_) funcs.push_back(e.to_function());
  std::vector<const Function *> leaves;
  for (auto &f : funcs) collect_leaves(*f, &leaves);

  PipeRef pipe;
  Lowering lw;
  std::vector<Utf8DictRef> key_dicts;   // GROUP BY a dictionary column: its codes are the key
  uint64_t hint = 1 << 16, n_groups = 0;
  int full_overflows = 0;   // overflows of tables with room for every row scanned
  for (;;) {   // the table is grown until the groups fit (a full re-scan: cardinality is unknown up front)
    uint64_t rows = 0;
    struct OptionsGuard {
      FuseQueryContextRef c;
      GpuOptions saved;
      explicit OptionsGuard(FuseQueryContextRef ctx) : c(std::move(ctx)), saved(c->options) {}
      ~OptionsGuard() { c->options = saved; }
    };
    SendableDataBlockStream source;
    {
      OptionsGuard guard(ctx_);
      ctx_->options.block_rows = 0;
      ctx_->options.align_runs = false;
      source = table->read(ctx_, partitions_);
    }
    int launches = 0;
    while (auto block = source->next()) {
      if (!pipe) {
        if (block->generated) lw.column_of(*block, block->schema()->fields[0].name);
        const int p = pred ? lw.lower(*pred, *block) : -1;
        std::vector<int> roots, key_roots;
        for (auto &f : funcs) roots.push_back(lw.lower(*f, *block));
        for (auto &k : keys) {
          key_roots.push_back(lw.lower(*k, *block));
          key_dicts.push_back(dict_of(*k, *block));
        }
        fq_pipe_desc d = lw.desc(FQ_PIPE_GROUPBY, p, roots);
        d.n_keys = (int)key_roots.size();
        for (size_t k = 0; k < key_roots.size(); k++) d.keys[k] = key_roots[k];
        pipe = compile_pipe(gpu, lw, d);
      }
      if (launches == 0) gpu->check(fq_pipe_groupby_reserve(gpu->raw(), pipe->pipe, hint));
      BoundSource bs;
      bind_source(lw, *block, &bs);
      gpu->check(fq_pipe_launch_groupby(gpu->raw(), pipe->pipe, &bs.src, launches > 0 ? FQ_RUN_ACCUMULATE : 0, gpu->stream));
      rows += bs.src.n_rows;
      launches++;
    }
    if (!pipe) break;   // no rows at all: no groups
    const fq_status st = fq_pipe_fetch_groupby(gpu->raw(), pipe->pipe, &n_groups);
    if (st == FQ_ERR_CAPACITY) {
      // no scan has more groups than rows: a table with room for all of them overflows only when the keys' hashes cluster,
      // and the next reservation rehashes them with a new seed.  Two such overflows are an error, not a larger table.
      if (hint >= rows && full_overflows++)
        throw FuseQueryError::internal("GROUP BY: two hash tables with room for all " + std::to_string(rows) + " rows scanned overflowed");
      hint = std::max<uint64_t>(1, std::min(hint * 8, rows));
      continue;
    }
    gpu->check(st);
    break;
  }

  std::vector<DataArrayRef> out;
  if (!pipe || n_groups == 0) {   // an empty result still carries the plan's schema
    for (const auto &f : schema_->fields) out.push_back(f.data_type == FQ_UTF8 ? DataArray::utf8({}) : DataArray::alloc(gpu, f.data_type, 0));
    return std::make_unique<DataBlockStream>(std::vector<DataBlock>{DataBlock(schema_, out)});
  }
  // export: key columns, then one column per Aggregator leaf
  std::vector<DataArrayRef> key_arrays, key_valid, leaf_arrays, leaf_valid;
  std::vector<fq_column *> kc, kv, lc, lv;
  for (size_t j = 0; j < keys.size(); j++) {
    fq_dtype t;
    int32_t nullable = 0;
    gpu->check(fq_pipe_key_dtype(gpu->raw(), pipe->pipe, (int)j, &t, &nullable));
    key_arrays.push_back(DataArray::alloc(gpu, t, n_groups));
    key_valid.push_back(nullable ? DataArray::alloc(gpu, FQ_BOOL, n_groups) : nullptr);
    kc.push_back(key_arrays.back()->column());
    kv.push_back(nullable ? key_valid.back()->column() : nullptr);
  }
  std::vector<int32_t> nodes(leaves.size() + 1);
  int32_t n_leaves = 0;
  gpu->check(fq_pipe_aggregator_nodes(gpu->raw(), pipe->pipe, nodes.data(), (int32_t)nodes.size(), &n_leaves));
  for (int k = 0; k < n_leaves; k++) {
    fq_dtype t;
    int32_t nullable = 0;
    gpu->check(fq_pipe_leaf_dtype(gpu->raw(), pipe->pipe, k, &t, &nullable));
    leaf_arrays.push_back(DataArray::alloc(gpu, t, n_groups));
    leaf_valid.push_back(nullable ? DataArray::alloc(gpu, FQ_BOOL, n_groups) : nullptr);
    lc.push_back(leaf_arrays.back()->column());
    lv.push_back(nullable ? leaf_valid.back()->column() : nullptr);
  }
  gpu->check(fq_pipe_export_groups(gpu->raw(), pipe->pipe, kc.data(), kv.data(), lc.data(), lv.data(), n_groups, gpu->stream));
  gpu->check(fq_stream_synchronize(gpu->raw(), gpu->stream));
  for (size_t j = 0; j < keys.size(); j++) {
    if (key_valid[j]) key_arrays[j]->set_validity(key_valid[j]);
    out.push_back(key_dicts[j] ? DataArray::with_dict(key_arrays[j], key_dicts[j]) : key_arrays[j]);
  }
  // the leaf block and the select expressions over it
  auto leaf_schema = std::make_shared<DataSchema>();
  std::map<const Function *, std::string> leaf_name;
  for (int k = 0; k < n_leaves; k++) {
    if (leaf_valid[k]) leaf_arrays[k]->set_validity(leaf_valid[k]);
    for (const auto &ld : lw.leaf_dict)   // min / max of a dictionary column: codes, read as strings
      if (lw.node_of.at(ld.first) == nodes[k]) leaf_arrays[k] = DataArray::with_dict(leaf_arrays[k], ld.second);
    leaf_schema->fields.push_back({"__leaf" + std::to_string(k), leaf_arrays[k]->data_type(), leaf_valid[k] != nullptr});
  }
  for (const Function *l : leaves) {
    const int node = lw.node_of.at(l);
    for (int k = 0; k < n_leaves; k++)
      if (nodes[k] == node) leaf_name[l] = "__leaf" + std::to_string(k);
  }
  DataBlock leaf_block(leaf_schema, leaf_arrays);
  std::vector<FunctionRef> finals;
  std::vector<const Function *> raw;
  for (auto &f : funcs) finals.push_back(over_leaves(*f, leaf_name));
  for (auto &f : finals) raw.push_back(f.get());
  if (!raw.empty()) {
    if (n_leaves == 0) throw FuseQueryError::internal("Unsupported on the device path: GROUP BY select expressions without an aggregate");
    ProjectResult r = run_project(gpu, leaf_block, nullptr, raw, -1, false);
    for (auto &c : r.columns) out.push_back(c);
  }
  return std::make_unique<DataBlockStream>(std::vector<DataBlock>{DataBlock(schema_, out)});
}

// ---------------------------------------------------------------------------------------------
// Pipeline — processors/pipeline.rs
// ---------------------------------------------------------------------------------------------
void Pipeline::add_source(IProcessorRef source) {
  if (processors_.empty()) processors_.push_back({});
  processors_[0].push_back(std::move(source));
}
void Pipeline::add_simple_transform(const std::function<IProcessorRef()> &f) {
  if (processors_.empty()) throw FuseQueryError::internal("Can't add transform to an empty pipe list");
  Pipe items;
  for (auto &x : processors_.back()) {
    IProcessorRef p = f();
    p->connect_to(x);
    items.push_back(std::move(p));
  }
  processors_.push_back(std::move(items));
}
void Pipeline::merge_processor() {
  if (processors_.empty()) throw FuseQueryError::internal("Can't merge processor when the last pipe is empty");
  if (processors_.back().size() > 1) {
    auto m = std::make_shared<MergeProcessor>();
    for (auto &x : processors_.back()) m->connect_to(x);
    processors_.push_back({m});
  }
}
SendableDataBlockStream Pipeline::execute() {
  if (processors_.empty()) throw FuseQueryError::internal("empty pipeline");
  if (processors_.back().size() > 1) merge_processor();
  return processors_.back()[0]->execute();
}
std::string Pipeline::to_string() const {   // Debug, pipeline.rs:109-135 + processor.rs:38-57 + processor_merge.rs:68-94
  std::string out;
  size_t indent = 0;
  for (size_t k = processors_.size(); k-- > 0;) {
    const Pipe &cur = processors_[k];
    size_t prev_ways = 0;
    std::string prev_name;
    if (k > 0) {
      prev_ways = processors_[k - 1].size();
      prev_name = processors_[k - 1][0]->name();
    }
    indent++;
    out += "\n";
    for (size_t i = 0; i < indent; i++) out += "  ";
    const std::string name = cur[0]->name();
    if (name == "MergeProcessor")
      out += "└─ Merge (" + prev_name + " × " + std::to_string(prev_ways) + (prev_ways == 1 ? " processor" : " processors") + ") to (" + name + " × " +
             std::to_string(cur.size()) + ")";
    else
      out += "└─ " + name + " × " + std::to_string(cur.size()) + (cur.size() == 1 ? " processor" : " processors");
  }
  return out;
}

// ---------------------------------------------------------------------------------------------
// PipelineBuilder — processors/pipeline_builder.rs:26-106
// ---------------------------------------------------------------------------------------------
Pipeline PipelineBuilder::build() const {
  Pipeline pipeline;
  std::vector<PlanNode> plans = plan_.children_to_plans();
  FuseQueryContextRef ctx = ctx_;
  size_t i = 0;
  // fused device pipes: ReadSource [Filter] (Projection [Limit] | Aggregate) collapse into one GpuPipeTransform
  // per source pipe; everything after them is built exactly like the reference does
  if (ctx->options.fuse && !plans.empty() && plans[0].kind == PlanNode::ReadSource) {
    size_t j = 1;
    std::optional<ExpressionPlan> pred;
    if (j < plans.size() && plans[j].kind == PlanNode::Filter) pred = plans[j++].predicate;
    if (j < plans.size() && plans[j].kind == PlanNode::Aggregate && !plans[j].group_expr.empty() && ctx->options.group_by) {
      // GROUP BY: one hash-aggregation processor over every partition (the table in HBM is the merge point)
      const PlanNode &src = plans[0];
      const PlanNode &sel = plans[j];
      pipeline.add_source(std::make_shared<GpuGroupByTransform>(ctx, src.db, src.table, src.partitions, pred, sel.schema(), sel.group_expr, sel.expr));
      i = j + 1;
    } else if (j < plans.size() && (plans[j].kind == PlanNode::Projection || plans[j].kind == PlanNode::Aggregate)) {
      const PlanNode &src = plans[0];
      const PlanNode &sel = plans[j];
      const bool is_agg = sel.kind == PlanNode::Aggregate;
      j++;
      std::optional<size_t> limit;
      if (!is_agg && j < plans.size() && plans[j].kind == PlanNode::Limit) limit = plans[j].n;
      size_t workers = ctx->worker_threads;
      size_t chunk = (workers == 0 || workers >= src.partitions.size()) ? 1 : src.partitions.size() / workers;   // :75-80
      for (size_t s = 0; s < src.partitions.size(); s += chunk) {
        Partitions part(src.partitions.begin() + (long)s, src.partitions.begin() + (long)std::min(s + chunk, src.partitions.size()));
        pipeline.add_source(std::make_shared<GpuPipeTransform>(ctx, src.db, src.table, part, pred, is_agg, sel.schema(), sel.expr, limit));
      }
      if (is_agg) {   // :50-65
        pipeline.merge_processor();
        pipeline.add_simple_transform([&]() { return std::make_shared<AggregateFinalTransform>(ctx, sel.schema(), sel.expr); });
      } else if (limit) {   // :31-41 (the per-pipe LimitTransform is inside the fused pipe)
        if (pipeline.pipe_num() > 1) {
          pipeline.merge_processor();
          size_t n = *limit;
          pipeline.add_simple_transform([n]() { return std::make_shared<LimitTransform>(n); });
        }
        j++;
      }
      i = j;
    }
  }
  for (; i < plans.size(); i++) {
    const PlanNode &plan = plans[i];
    switch (plan.kind) {
      case PlanNode::Limit: {
        size_t n = plan.n;
        pipeline.add_simple_transform([n]() { return std::make_shared<LimitTransform>(n); });
        if (pipeline.pipe_num() > 1) {
          pipeline.merge_processor();
          pipeline.add_simple_transform([n]() { return std::make_shared<LimitTransform>(n); });
        }
        break;
      }
      case PlanNode::Sort:   // a pipeline breaker: every pipe meets in one sort processor
        if (pipeline.pipe_num() > 1) pipeline.merge_processor();
        {
          std::optional<size_t> limit;
          if (i + 1 < plans.size() && plans[i + 1].kind == PlanNode::Limit) limit = plans[i + 1].n;   // the LimitTransform still follows
          pipeline.add_simple_transform([&]() { return std::make_shared<GpuSortTransform>(ctx, plan.expr, plan.descending, limit); });
        }
        break;
      case PlanNode::Projection:
        pipeline.add_simple_transform([&]() { return std::make_shared<ProjectionTransform>(ctx, plan.schema(), plan.expr); });
        break;
      case PlanNode::Aggregate:
        pipeline.add_simple_transform([&]() { return std::make_shared<AggregatePartialTransform>(ctx, plan.schema(), plan.expr); });
        pipeline.merge_processor();
        pipeline.add_simple_transform([&]() { return std::make_shared<AggregateFinalTransform>(ctx, plan.schema(), plan.expr); });
        break;
      case PlanNode::Filter:
        pipeline.add_simple_transform([&]() { return std::make_shared<FilterTransform>(ctx, plan.predicate); });
        break;
      case PlanNode::ReadSource: {
        size_t workers = ctx->worker_threads;
        size_t chunk = (workers == 0 || workers >= plan.partitions.size()) ? 1 : plan.partitions.size() / workers;
        for (size_t s = 0; s < plan.partitions.size(); s += chunk) {
          Partitions part(plan.partitions.begin() + (long)s, plan.partitions.begin() + (long)std::min(s + chunk, plan.partitions.size()));
          pipeline.add_source(std::make_shared<SourceTransform>(ctx, plan.db, plan.table, part));
        }
        break;
      }
      default:
        throw FuseQueryError::internal(std::string("Build pipeline from the plan node unsupported:\"") + plan.name() + "\"");
    }
  }
  pipeline.merge_processor();
  return pipeline;
}

// ---------------------------------------------------------------------------------------------
// executors
// ---------------------------------------------------------------------------------------------
SendableDataBlockStream SelectExecutor::execute() { return PipelineBuilder::create(ctx_, plan_).build().execute(); }
SendableDataBlockStream ExplainExecutor::execute() {   // executor_explain.rs:35-59
  auto schema = std::make_shared<DataSchema>();
  schema->fields.push_back({"explain", FQ_UTF8, false});
  Pipeline pipeline = PipelineBuilder::create(ctx_, *plan_.input).build();
  DataBlock block(schema, {DataArray::utf8({plan_.to_string(), pipeline.to_string()})});
  return std::make_unique<DataBlockStream>(std::vector<DataBlock>{block});
}
std::shared_ptr<IExecutor> ExecutorFactory::get(FuseQueryContextRef ctx, const PlanNode &plan) {
  switch (plan.kind) {
    case PlanNode::Select: return std::make_shared<SelectExecutor>(ctx, plan);
    case PlanNode::Explain: return std::make_shared<ExplainExecutor>(ctx, plan);
    default: throw FuseQueryError::internal(std::string("Can't get the executor by plan:") + plan.name());
  }
}

std::vector<DataBlock> execute_sql(FuseQueryContextRef ctx, const std::string &sql) {   // mysql_handler.rs:52-75
  PlanNode plan = Planner().build_from_sql(ctx, sql);
  plan = Optimizer::create().optimize(plan);
  auto executor = ExecutorFactory::get(ctx, plan);
  auto stream = executor->execute();
  std::vector<DataBlock> blocks;
  while (auto b = stream->next()) blocks.push_back(*b);
  return blocks;
}


// ---- servers/mysql/mysql_stream.rs ----
namespace {
template <class T> void cells_of(const DataArray &a, std::vector<std::string> *out) {
  std::vector<T> v(a.len());
  a.to_host(v.data());
  std::vector<unsigned char> ok;
  if (a.validity()) {
    ok.resize(a.len());
    a.validity()->to_host(ok.data());
  }
  out->reserve(v.size());
  for (size_t i = 0; i < v.size(); i++) {
    if (!ok.empty() && !ok[i]) { out->emplace_back(); continue; }   // arrow: a NULL slot prints as the empty string
    if constexpr (std::is_floating_point<T>::value) {
      if (std::isnan(v[i])) { out->emplace_back("NaN"); continue; }
      if (std::isinf(v[i])) { out->emplace_back(v[i] < 0 ? "-inf" : "inf"); continue; }
      char buf[400];
      auto r = std::to_chars(buf, buf + sizeof buf, v[i], std::chars_format::fixed);   // Rust's Display: shortest, no exponent
      out->emplace_back(buf, r.ptr);
    } else {
      out->push_back(std::to_string(v[i]));
    }
  }
}
}  // namespace

MySQLResultSet MySQLStream::execute() const {
  MySQLResultSet rs;
  if (blocks_.empty()) return rs;   // writer.completed(0, 0)
  const DataBlock &first = blocks_[0];
  for (const DataField &f : first.schema()->fields) {
    std::string t;
    switch (f.data_type) {
      case FQ_I8: case FQ_I16: case FQ_I32: case FQ_I64: case FQ_U8: case FQ_U16: case FQ_U32: case FQ_U64: t = "MYSQL_TYPE_LONG"; break;
      case FQ_F32: case FQ_F64: t = "MYSQL_TYPE_FLOAT"; break;
      case FQ_UTF8: t = "MYSQL_TYPE_VARCHAR"; break;
      default: throw FuseQueryError::internal(std::string("Unsupported column type:") + data_type_name(f.data_type));
    }
    rs.columns.push_back({f.name, t});
  }
  const size_t ncols = first.num_columns();
  if (ncols == 0) return rs;
  for (const DataBlock &b : blocks_) {
    std::vector<std::vector<std::string>> cols(ncols);
    for (size_t c = 0; c < ncols; c++) {
      const DataArray &a = *b.column(c);
      switch (a.data_type()) {
        case FQ_I8: cells_of<int8_t>(a, &cols[c]); break;
        case FQ_I16: cells_of<int16_t>(a, &cols[c]); break;
        case FQ_I32: cells_of<int32_t>(a, &cols[c]); break;
        case FQ_I64: cells_of<int64_t>(a, &cols[c]); break;
        case FQ_U8: cells_of<uint8_t>(a, &cols[c]); break;
        case FQ_U16: cells_of<uint16_t>(a, &cols[c]); break;
        case FQ_U32: cells_of<uint32_t>(a, &cols[c]); break;
        case FQ_U64: cells_of<uint64_t>(a, &cols[c]); break;
        case FQ_F32: cells_of<float>(a, &cols[c]); break;
        case FQ_F64: cells_of<double>(a, &cols[c]); break;
        case FQ_UTF8:
          for (uint64_t i = 0; i < a.len(); i++) cols[c].push_back(a.value(i).s);
          break;
        default: throw FuseQueryError::internal(std::string("Unsupported column type:") + data_type_name(a.data_type()));
      }
    }
    const size_t nrows = cols[0].size();
    for (size_t r = 0; r < nrows; r++) {
      std::vector<std::string> row(ncols);
      for (size_t c = 0; c < ncols; c++) row[c] = std::move(cols[c][r]);
      rs.rows.push_back(std::move(row));
    }
  }
  return rs;
}

}  // namespace fuse
