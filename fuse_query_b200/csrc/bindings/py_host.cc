// py_host.cc — pybind11 view of the C++ host mirror (fuse_query_b200._fuse_host), so that the parity
// tests can be written the way the reference's own Rust tests are.  No computation happens here.
#include <pybind11/functional.h>
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include "../host/fq_host.h"

namespace py = pybind11;
using namespace fuse;

namespace fuse { void numbers_cache_clear(); }

namespace {

py::object value_payload(const DataValue &v) {
  if (v.tag == FQ_NULL) return py::none();
  if (v.tag == FQ_STRUCT) {
    py::list l;
    for (const auto &it : v.items) l.append(it);
    return std::move(l);
  }
  if (!v.some) return py::none();
  switch (v.tag) {
    case FQ_BOOL: return py::bool_(v.i != 0);
    case FQ_UTF8: return py::str(v.s);
    case FQ_F32: case FQ_F64: return py::float_(v.f);
    case FQ_U8: case FQ_U16: case FQ_U32: case FQ_U64: return py::int_(v.u);
    default: return py::int_(v.i);
  }
}
DataValue make_value(int tag, py::object payload) {
  DataValue v;
  v.tag = tag;
  if (tag == FQ_NULL) return v;
  if (tag == FQ_STRUCT) {
    for (auto it : payload) v.items.push_back(it.cast<DataValue>());
    return v;
  }
  if (payload.is_none()) return v;
  v.some = true;
  switch (tag) {
    case FQ_BOOL: v.i = payload.cast<bool>(); break;
    case FQ_UTF8: v.s = payload.cast<std::string>(); break;
    case FQ_F32: v.f = (double)(float)payload.cast<double>(); break;
    case FQ_F64: v.f = payload.cast<double>(); break;
    case FQ_U8: case FQ_U16: case FQ_U32: case FQ_U64: v.u = payload.cast<uint64_t>(); break;
    default: v.i = payload.cast<int64_t>();
  }
  return v;
}
const char *np_format(DataType t) {
  switch (t) {
    case FQ_BOOL: return "?";
    case FQ_I8: return "b"; case FQ_I16: return "h"; case FQ_I32: return "i"; case FQ_I64: return "q";
    case FQ_U8: return "B"; case FQ_U16: return "H"; case FQ_U32: return "I"; case FQ_U64: return "Q";
    case FQ_F32: return "f"; case FQ_F64: return "d";
    default: return nullptr;
  }
}
DataType dtype_of_numpy(const py::array &a) {
  char k = a.dtype().kind();
  ssize_t sz = a.dtype().itemsize();
  if (k == 'b') return FQ_BOOL;
  if (k == 'i') return sz == 1 ? FQ_I8 : sz == 2 ? FQ_I16 : sz == 4 ? FQ_I32 : FQ_I64;
  if (k == 'u') return sz == 1 ? FQ_U8 : sz == 2 ? FQ_U16 : sz == 4 ? FQ_U32 : FQ_U64;
  if (k == 'f') return sz == 4 ? FQ_F32 : FQ_F64;
  throw FuseQueryError::internal("unsupported numpy dtype");
}
py::object array_to_python(const DataArrayRef &a) {
  if (a->is_utf8()) return py::cast(a->strings());
  py::array out(py::dtype(np_format(a->data_type())), py::array::ShapeContainer{(ssize_t)a->len()});
  a->to_host(out.mutable_data());
  return std::move(out);
}
std::vector<DataBlock> drain(IDataBlockStream &s) {
  std::vector<DataBlock> blocks;
  while (auto b = s.next()) blocks.push_back(*b);
  return blocks;
}
// a Python-visible stream handle
struct PyStream {
  SendableDataBlockStream s;
  std::optional<DataBlock> next() { return s->next(); }
};
// IProcessor implemented by a Python callable returning a list of blocks (test doubles)
class PyBlocksProcessor : public IProcessor {
 public:
  explicit PyBlocksProcessor(std::vector<DataBlock> blocks) : blocks_(std::move(blocks)) {}
  std::string name() const override { return "DataBlockSource"; }
  void connect_to(IProcessorRef) override { throw FuseQueryError::internal("Cannot call DataBlockSource connect_to"); }
  SendableDataBlockStream execute() override { return std::make_unique<DataBlockStream>(blocks_); }

 private:
  std::vector<DataBlock> blocks_;
};

}  // namespace

PYBIND11_MODULE(_fuse_host, m) {
  m.doc() = "C++ host mirror of fuse-query's function / processor / planner surface over libfuse_gpu.so";

  static py::exception<FuseQueryError> exc(m, "FuseQueryError");
  py::register_exception_translator([](std::exception_ptr p) {
    try {
      if (p) std::rethrow_exception(p);
    } catch (const FuseQueryError &e) {
      exc(e.what());
    }
  });

  // ---- data types ----
  py::module_ dt = m.def_submodule("DataType");
  const char *names[] = {"Null", "Boolean", "Int8", "Int16", "Int32", "Int64", "UInt8", "UInt16", "UInt32", "UInt64", "Float32", "Float64", "Utf8", "Struct"};
  for (int i = 0; i <= FQ_STRUCT; i++) dt.attr(names[i]) = i;
  m.def("data_type_name", &data_type_name);
  m.def("numerical_coercion", &numerical_coercion);
  m.def("equal_coercion", &equal_coercion);
  py::module_ ops = m.def_submodule("ops");
  ops.attr("Add") = (int)FQ_AR_ADD; ops.attr("Sub") = (int)FQ_AR_SUB; ops.attr("Mul") = (int)FQ_AR_MUL; ops.attr("Div") = (int)FQ_AR_DIV;
  ops.attr("Eq") = (int)FQ_CMP_EQ; ops.attr("Lt") = (int)FQ_CMP_LT; ops.attr("LtEq") = (int)FQ_CMP_LTEQ; ops.attr("Gt") = (int)FQ_CMP_GT; ops.attr("GtEq") = (int)FQ_CMP_GTEQ;
  ops.attr("And") = (int)FQ_LG_AND; ops.attr("Or") = (int)FQ_LG_OR;
  ops.attr("Min") = (int)FQ_AGG_MIN; ops.attr("Max") = (int)FQ_AGG_MAX; ops.attr("Sum") = (int)FQ_AGG_SUM; ops.attr("Count") = (int)FQ_AGG_COUNT;

  py::class_<DataValue>(m, "DataValue")
      .def(py::init(&make_value), py::arg("tag"), py::arg("value") = py::none())
      .def_static("Null", &DataValue::Null)
      .def_static("from_json", &DataValue::from_json)
      .def_readonly("tag", &DataValue::tag)
      .def_readonly("some", &DataValue::some)
      .def_property_readonly("value", &value_payload)
      .def("is_null", &DataValue::is_null)
      .def("data_type", &DataValue::data_type)
      .def("to_json", &DataValue::to_json)
      .def("__str__", &DataValue::to_string)
      .def("__repr__", [](const DataValue &v) { return std::string("DataValue::") + (v.tag == FQ_NULL ? "Null" : std::string(data_type_name(v.tag)) + "(" + v.to_string() + ")"); })
      .def("__eq__", &DataValue::operator==);
  m.def("data_value_arithmetic_op", &data_value_arithmetic_op);
  m.def("data_value_aggregate_op", &data_value_aggregate_op);

  py::class_<DataField>(m, "DataField")
      .def(py::init([](std::string n, int t, bool nullable) { return DataField{std::move(n), t, nullable}; }))
      .def_readonly("name", &DataField::name)
      .def_readonly("data_type", &DataField::data_type)
      .def_readonly("nullable", &DataField::nullable);
  py::class_<DataSchema, std::shared_ptr<DataSchema>>(m, "DataSchema")
      .def(py::init([](std::vector<DataField> f) { auto s = std::make_shared<DataSchema>(); s->fields = std::move(f); return s; }))
      .def_readonly("fields", &DataSchema::fields)
      .def("index_of", &DataSchema::index_of)
      .def("names", [](const DataSchema &s) { std::vector<std::string> n; for (auto &f : s.fields) n.push_back(f.name); return n; })
      .def("types", [](const DataSchema &s) { std::vector<int> n; for (auto &f : s.fields) n.push_back(f.data_type); return n; });

  py::class_<GpuContext, GpuContextRef>(m, "GpuContext")
      .def_static("create", &GpuContext::create, py::arg("device") = 0)
      .def_property_readonly("launch_count", &GpuContext::launch_count)
      .def_property_readonly("device", &GpuContext::device)
      .def("set_stream", [](GpuContext &g, uintptr_t s) { g.stream = (void *)s; });

  py::class_<GpuGroup, std::shared_ptr<GpuGroup>>(m, "GpuGroup")
      .def(py::init([](GpuContextRef gpu, int rank, int world, uint64_t row_bytes) { return std::make_shared<GpuGroup>(gpu, rank, world, row_bytes); }),
           py::arg("gpu"), py::arg("rank"), py::arg("world"), py::arg("row_bytes") = 1u << 16)
      .def("handle", [](const GpuGroup &g) { return py::bytes(g.handle()); })
      .def("connect", [](GpuGroup &g, const std::vector<py::bytes> &hs) {
        std::vector<std::string> v;
        for (const auto &h : hs) v.push_back(std::string(h));
        g.connect(v);
      })
      .def("gather", [](GpuGroup &g, const std::vector<DataArrayRef> &cols, const std::vector<int> &types, uint64_t rows, uint64_t selected,
                        uint64_t capacity, int64_t limit) {
        std::vector<DataType> t(types.begin(), types.end());
        return g.gather(cols, t, rows, selected, capacity, limit);
      })
      .def_property_readonly("rank", &GpuGroup::rank)
      .def_property_readonly("world", &GpuGroup::world);

  py::class_<DataArray, DataArrayRef>(m, "DataArray")
      .def_static("from_numpy", [](GpuContextRef gpu, py::array a) {
        py::array c = py::array::ensure(a, py::array::c_style);
        return DataArray::from_host(gpu, dtype_of_numpy(c), c.data(), (uint64_t)c.size());
      })
      .def_static("from_numpy_masked", [](GpuContextRef gpu, py::array a, py::array valid) {
        py::array c = py::array::ensure(a, py::array::c_style);
        // canonical 0/1 bytes: the kernels load validity as `bool` and combine it bitwise, so a mask holding 2 or 255 must
        // not reach the device unchanged
        py::array v = py::array::ensure(valid.attr("__ne__")(0).attr("astype")("uint8"), py::array::c_style);
        if (v.size() != c.size()) throw FuseQueryError::internal("validity and values differ in length");
        auto arr = DataArray::from_host(gpu, dtype_of_numpy(c), c.data(), (uint64_t)c.size());
        arr->set_validity(DataArray::from_host(gpu, FQ_BOOL, v.data(), (uint64_t)v.size()));
        return arr;
      })
      .def_static("from_arrow_bitmap", [](GpuContextRef gpu, uintptr_t address, uint64_t bit_offset, uint64_t len) {
        return DataArray::from_arrow_bitmap(gpu, (const void *)address, bit_offset, len);
      }, "Boolean array from an Arrow LSB-first bitmap at a host address (pyarrow Buffer.address), expanded on the device")
      .def("to_arrow_bitmap", [](const DataArrayRef &a) {
        auto v = a->to_arrow_bitmap();
        return py::bytes((const char *)v.data(), v.size());
      })
      .def_static("from_utf8", [](GpuContextRef gpu, py::array_t<int32_t, py::array::c_style | py::array::forcecast> offsets, py::bytes data,
                                  py::object valid) {
        const std::string bytes = data;
        const uint64_t n = offsets.size() ? (uint64_t)offsets.size() - 1 : 0;
        if (!offsets.size()) throw FuseQueryError::internal("Utf8 offsets need len + 1 entries");
        std::vector<unsigned char> v;
        if (!valid.is_none()) {
          py::array_t<uint8_t, py::array::c_style | py::array::forcecast> a = py::array::ensure(valid.attr("__ne__")(0).attr("astype")("uint8"));
          if ((uint64_t)a.size() != n) throw FuseQueryError::internal("validity and values differ in length");
          v.assign(a.data(), a.data() + n);
        }
        if (n && (uint64_t)offsets.data()[n] != bytes.size()) throw FuseQueryError::internal("Utf8 offsets do not end at the byte count");
        return DataArray::utf8_dict(gpu, offsets.data(), bytes.data(), n, v.empty() ? nullptr : v.data());
      }, py::arg("gpu"), py::arg("offsets"), py::arg("data"), py::arg("valid") = py::none(),
         "Utf8 column from Arrow offsets (int32, starting at 0) + bytes (+ validity), dictionary-encoded on the device")
      .def("dictionary", [](const DataArrayRef &a) -> py::object {
        if (!a->dict()) return py::none();
        const Utf8Dict &d = *a->dict();
        std::vector<uint32_t> all(d.size);
        for (uint64_t i = 0; i < d.size; i++) all[i] = (uint32_t)i;
        auto rows = DataArray::from_host(a->ctx(), FQ_U32, all.data(), d.size);
        return py::cast(DataArray::with_dict(rows, a->dict())->strings());
      }, "the sorted dictionary of a dictionary-encoded Utf8 array (None for other arrays)")
      .def("set_validity", &DataArray::set_validity)
      .def("validity", &DataArray::validity)
      .def("null_count", &DataArray::null_count)
      .def_static("utf8", &DataArray::utf8)
      .def("data_type", &DataArray::data_type)
      .def("__len__", &DataArray::len)
      .def("slice", &DataArray::slice)
      .def("value", &DataArray::value)
      .def("to_numpy", &array_to_python)
      .def("to_list", [](const DataArrayRef &a) -> py::object {   // NULL slots come back as None
        py::object o = array_to_python(a);
        if (a->is_utf8()) {
          if (!a->validity()) return o;
          py::list vals = o;
          py::list ok = array_to_python(a->validity()).attr("tolist")();
          for (size_t i = 0; i < vals.size(); i++)
            if (!ok[i].cast<bool>()) vals[i] = py::none();
          return std::move(vals);
        }
        py::list vals = o.attr("tolist")();
        if (a->validity()) {
          py::list ok = array_to_python(a->validity()).attr("tolist")();
          for (size_t i = 0; i < vals.size(); i++)
            if (!ok[i].cast<bool>()) vals[i] = py::none();
        }
        return std::move(vals);
      });

  py::class_<DataColumnarValue>(m, "DataColumnarValue")
      .def_static("Array", &DataColumnarValue::Array)
      .def_static("Scalar", &DataColumnarValue::Scalar)
      .def_readonly("is_scalar", &DataColumnarValue::is_scalar)
      .def_readonly("array", &DataColumnarValue::array)
      .def_readonly("scalar", &DataColumnarValue::scalar)
      .def("data_type", &DataColumnarValue::data_type)
      .def("to_array", &DataColumnarValue::to_array);

  py::class_<DataBlock>(m, "DataBlock")
      .def(py::init([](std::shared_ptr<DataSchema> s, std::vector<DataArrayRef> c) { return DataBlock(s, std::move(c)); }))
      .def_static("create", [](std::shared_ptr<DataSchema> s, std::vector<DataArrayRef> c) { return DataBlock(s, std::move(c)); })
      .def("schema", [](const DataBlock &b) { return std::const_pointer_cast<DataSchema>(b.schema()); })
      .def("num_rows", &DataBlock::rows)
      .def("num_columns", &DataBlock::num_columns)
      .def("column", &DataBlock::column)
      .def("column_by_name", &DataBlock::column_by_name)
      .def_readonly("generated", &DataBlock::generated);

  m.def("data_array_arithmetic_op", &data_array_arithmetic_op);
  m.def("data_array_comparison_op", &data_array_comparison_op);
  m.def("data_array_logic_op", &data_array_logic_op);
  m.def("data_array_aggregate_op", &data_array_aggregate_op);

  // ---- functions ----
  py::class_<Function, FunctionRef>(m, "Function")
      .def("clone", &Function::clone)
      .def("return_type", &Function::return_type)
      .def("nullable", &Function::nullable)
      .def("eval", &Function::eval)
      .def("set_depth", &Function::set_depth)
      .def("accumulate", &Function::accumulate)
      .def("accumulate_result", &Function::accumulate_result)
      .def("merge_state", &Function::merge_state)
      .def("merge_result", &Function::merge_result)
      .def("__str__", &Function::to_string)
      .def("__repr__", &Function::to_string);
  struct FieldFunctionNS {};
  py::class_<FieldFunctionNS>(m, "FieldFunction").def_static("try_create", &Function::FieldFunction);
  struct ConstantFunctionNS {};
  py::class_<ConstantFunctionNS>(m, "ConstantFunction").def_static("try_create", &Function::ConstantFunction);
  struct AliasFunctionNS {};
  py::class_<AliasFunctionNS>(m, "AliasFunction").def_static("try_create", &Function::AliasFunction);
  struct ArithmeticFunctionNS {};
  py::class_<ArithmeticFunctionNS>(m, "ArithmeticFunction").def_static("try_create", &Function::ArithmeticFunction);
  struct ComparisonFunctionNS {};
  py::class_<ComparisonFunctionNS>(m, "ComparisonFunction").def_static("try_create", &Function::ComparisonFunction);
  struct LogicFunctionNS {};
  py::class_<LogicFunctionNS>(m, "LogicFunction").def_static("try_create", &Function::LogicFunction);
  struct AggregatorFunctionNS {};
  py::class_<AggregatorFunctionNS>(m, "AggregatorFunction").def_static("try_create", &Function::AggregatorFunction);
  struct ScalarFunctionFactoryNS {};
  py::class_<ScalarFunctionFactoryNS>(m, "ScalarFunctionFactory").def_static("get", &Function::factory_get);

  // ---- planners ----
  py::class_<ExpressionPlan>(m, "ExpressionPlan")
      .def_static("Field", &ExpressionPlan::field)
      .def_static("Constant", &ExpressionPlan::constant)
      .def_static("Alias", &ExpressionPlan::alias)
      .def_static("BinaryExpression", &ExpressionPlan::binary)
      .def_static("Function", &ExpressionPlan::function)
      .def_static("Wildcard", &ExpressionPlan::wildcard)
      .def("to_function", [](const ExpressionPlan &e) { return e.to_function(); })
      .def("to_field", &ExpressionPlan::to_field)
      .def("is_aggregate", &ExpressionPlan::is_aggregate)
      .def("__str__", &ExpressionPlan::to_string)
      .def("__repr__", &ExpressionPlan::to_string);
  py::class_<Partition>(m, "Partition").def_readonly("name", &Partition::name).def_readonly("version", &Partition::version);
  py::class_<PlanNode>(m, "PlanNode")
      .def("name", &PlanNode::name)
      .def("schema", [](const PlanNode &p) { return std::const_pointer_cast<DataSchema>(p.schema()); })
      .def("children_to_plans", &PlanNode::children_to_plans)
      .def_readonly("partitions", &PlanNode::partitions)
      .def_readonly("db", &PlanNode::db)
      .def_readonly("table", &PlanNode::table)
      .def_readonly("expr", &PlanNode::expr)
      .def_readonly("predicate", &PlanNode::predicate)
      .def_readonly("n", &PlanNode::n)
      .def_readonly("descending", &PlanNode::descending)
      .def_property_readonly("input", [](const PlanNode &p) { return *p.input; })
      .def("__str__", &PlanNode::to_string)
      .def("__repr__", &PlanNode::to_string);
  py::class_<PlanBuilder>(m, "PlanBuilder")
      .def_static("create", [](std::shared_ptr<DataSchema> s) { return PlanBuilder::create(s); })
      .def_static("from_plan", &PlanBuilder::from)
      .def("project", &PlanBuilder::project)
      .def("aggregate", &PlanBuilder::aggregate)
      .def("filter", &PlanBuilder::filter)
      .def("limit", &PlanBuilder::limit)
      .def("select", &PlanBuilder::select)
      .def("explain", &PlanBuilder::explain)
      .def("build", &PlanBuilder::build);

  // ---- datasources / context ----
  py::class_<ITable, ITableRef>(m, "ITable")
      .def("name", &ITable::name)
      .def("schema", [](const ITable &t) { return std::const_pointer_cast<DataSchema>(t.schema()); })
      .def("read_plan", &ITable::read_plan);
  py::class_<NumbersTable, ITable, std::shared_ptr<NumbersTable>>(m, "NumbersTable")
      .def(py::init<>())
      .def_static("generate_parts", &NumbersTable::generate_parts);
  py::class_<MemoryTable, ITable, std::shared_ptr<MemoryTable>>(m, "MemoryTable")
      .def(py::init([](std::string db, std::string name, std::shared_ptr<DataSchema> schema, std::vector<DataArrayRef> cols) {
        return std::make_shared<MemoryTable>(std::move(db), std::move(name), schema, std::move(cols));
      }))
      .def("num_rows", &MemoryTable::num_rows);
  py::class_<DataSource, std::shared_ptr<DataSource>>(m, "DataSource")
      .def(py::init<>())
      .def("add_database", &DataSource::add_database)
      .def("add_table", &DataSource::add_table)
      .def("get_table", &DataSource::get_table);
  py::class_<GpuOptions>(m, "GpuOptions")
      .def_readwrite("fuse", &GpuOptions::fuse)
      .def_readwrite("generated", &GpuOptions::generated)
      .def_readwrite("block_rows", &GpuOptions::block_rows)
      .def_readwrite("tail_quirk", &GpuOptions::tail_quirk)
      .def_readwrite("limit_early_exit", &GpuOptions::limit_early_exit)
      .def_readwrite("block_quirks", &GpuOptions::block_quirks)
      .def_readwrite("group_by", &GpuOptions::group_by);
  py::class_<FuseQueryContext, FuseQueryContextRef>(m, "FuseQueryContext")
      .def_static("create_ctx", [](size_t workers, GpuContextRef gpu) { return FuseQueryContext::create_ctx(workers, nullptr, gpu); },
                  py::arg("worker_threads"), py::arg("gpu") = nullptr)
      .def_readwrite("worker_threads", &FuseQueryContext::worker_threads)
      .def_readwrite("options", &FuseQueryContext::options)
      .def("get_table", &FuseQueryContext::get_table)
      .def("datasource", &FuseQueryContext::datasource)
      .def("get_current_database", &FuseQueryContext::get_current_database)
      .def("set_current_database", &FuseQueryContext::set_current_database);
  py::class_<Planner>(m, "Planner").def(py::init<>()).def("build_from_sql", &Planner::build_from_sql);
  py::class_<Optimizer>(m, "Optimizer").def_static("create", &Optimizer::create).def("optimize", &Optimizer::optimize);
  py::class_<FilterPushDownOptimizer>(m, "FilterPushDownOptimizer").def(py::init<>()).def_static("create", []() { return FilterPushDownOptimizer(); }).def("optimize", &FilterPushDownOptimizer::optimize);

  // ---- streams / processors ----
  py::class_<PyStream>(m, "DataBlockStream")
      .def("next", &PyStream::next)
      .def("collect", [](PyStream &s) { return drain(*s.s); });
  py::class_<IProcessor, IProcessorRef>(m, "IProcessor")
      .def("name", &IProcessor::name)
      .def("connect_to", &IProcessor::connect_to)
      .def("execute", [](IProcessor &p) { return PyStream{p.execute()}; });
  py::class_<SourceTransform, IProcessor, std::shared_ptr<SourceTransform>>(m, "SourceTransform")
      .def(py::init<FuseQueryContextRef, std::string, std::string, Partitions>())
      .def_static("try_create", [](FuseQueryContextRef c, std::string db, std::string t, Partitions p) { return std::make_shared<SourceTransform>(c, db, t, p); });
  py::class_<PyBlocksProcessor, IProcessor, std::shared_ptr<PyBlocksProcessor>>(m, "DataBlockSource").def(py::init<std::vector<DataBlock>>());
  py::class_<FilterTransform, IProcessor, std::shared_ptr<FilterTransform>>(m, "FilterTransform")
      .def_static("try_create", [](FuseQueryContextRef c, const ExpressionPlan &p) { return std::make_shared<FilterTransform>(c, p); });
  py::class_<ProjectionTransform, IProcessor, std::shared_ptr<ProjectionTransform>>(m, "ProjectionTransform")
      .def_static("try_create", [](FuseQueryContextRef c, std::shared_ptr<DataSchema> s, const std::vector<ExpressionPlan> &e) { return std::make_shared<ProjectionTransform>(c, s, e); });
  py::class_<AggregatePartialTransform, IProcessor, std::shared_ptr<AggregatePartialTransform>>(m, "AggregatePartialTransform")
      .def_static("try_create", [](FuseQueryContextRef c, std::shared_ptr<DataSchema> s, const std::vector<ExpressionPlan> &e) { return std::make_shared<AggregatePartialTransform>(c, s, e); });
  py::class_<GpuSortTransform, IProcessor, std::shared_ptr<GpuSortTransform>>(m, "GpuSortTransform")
      .def_static("try_create", [](FuseQueryContextRef c, const std::vector<ExpressionPlan> &keys, const std::vector<bool> &desc) {
        return std::make_shared<GpuSortTransform>(c, keys, desc);
      });
  py::class_<AggregateFinalTransform, IProcessor, std::shared_ptr<AggregateFinalTransform>>(m, "AggregateFinalTransform")
      .def_static("try_create", [](FuseQueryContextRef c, std::shared_ptr<DataSchema> s, const std::vector<ExpressionPlan> &e) { return std::make_shared<AggregateFinalTransform>(c, s, e); });
  py::class_<LimitTransform, IProcessor, std::shared_ptr<LimitTransform>>(m, "LimitTransform")
      .def_static("try_create", [](size_t n) { return std::make_shared<LimitTransform>(n); });
  py::class_<MergeProcessor, IProcessor, std::shared_ptr<MergeProcessor>>(m, "MergeProcessor").def(py::init<>());
  py::class_<GpuPipeTransform, IProcessor, std::shared_ptr<GpuPipeTransform>>(m, "GpuPipeTransform")
      .def_static("try_create",
                  [](FuseQueryContextRef c, std::string db, std::string table, Partitions parts, std::optional<ExpressionPlan> pred, bool is_agg,
                     std::shared_ptr<DataSchema> schema, std::vector<ExpressionPlan> exprs, std::optional<size_t> limit) {
                    return std::make_shared<GpuPipeTransform>(c, db, table, parts, pred, is_agg, schema, exprs, limit);
                  })
      .def("describe", &GpuPipeTransform::describe);

  py::class_<Pipeline>(m, "Pipeline")
      .def(py::init<>())
      .def_static("create", []() { return Pipeline(); })
      .def("pipe_num", &Pipeline::pipe_num)
      .def("add_source", &Pipeline::add_source)
      .def("add_simple_transform", &Pipeline::add_simple_transform)
      .def("merge_processor", &Pipeline::merge_processor)
      .def("execute", [](Pipeline &p) { return PyStream{p.execute()}; })
      .def("pipes", [](const Pipeline &p) { std::vector<std::vector<std::string>> o; for (auto &pp : p.pipes()) { o.emplace_back(); for (auto &x : pp) o.back().push_back(x->name()); } return o; })
      .def("__str__", &Pipeline::to_string)
      .def("__repr__", &Pipeline::to_string);
  py::class_<PipelineBuilder>(m, "PipelineBuilder")
      .def_static("create", &PipelineBuilder::create)
      .def("build", &PipelineBuilder::build);

  // ---- executors ----
  py::class_<IExecutor, std::shared_ptr<IExecutor>>(m, "IExecutor")
      .def("name", &IExecutor::name)
      .def("execute", [](IExecutor &e) { return PyStream{e.execute()}; });
  struct ExecutorFactoryNS {};
  py::class_<ExecutorFactoryNS>(m, "ExecutorFactory").def_static("get", &ExecutorFactory::get);
  m.def("mysql_result_set", [](std::vector<DataBlock> blocks) {
    MySQLResultSet rs = MySQLStream::create(std::move(blocks)).execute();
    py::list cols;
    for (auto &c : rs.columns) cols.append(py::make_tuple(c.column, c.coltype));
    return py::make_tuple(cols, rs.rows);
  }, "servers/mysql/mysql_stream.rs: (columns [(name, MYSQL_TYPE_*)], rows of strings) for a list of result blocks");
  m.def("execute_sql", &execute_sql, "plan -> optimize -> execute -> drain (what the MySQL handler does per query)");
  m.def("numbers_cache_clear", &numbers_cache_clear);
}
