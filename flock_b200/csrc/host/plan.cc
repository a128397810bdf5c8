// plan.cc -- builds ExecutionPlan trees from the reference's serde-JSON and runs them on the GPU.
// See plan.h for the mapping to the reference's types.
#include "plan.h"

#include <algorithm>
#include <deque>
#include <set>

#include "../expr_compile.h"

namespace flock {

using fg::Expr;
using fg::ExprTok;
using fg::fail;

// ------------------------------------------------------------------------------------------------
// data types / scalar values / expressions in the reference's JSON dialect
// ------------------------------------------------------------------------------------------------
static void parse_data_type(const Json& j, int* dtype, std::string* format) {
  if (j.is_string()) {
    const std::string& s = j.str;
    if (s == "Int32") { *dtype = FLOCKGPU_INT32; *format = "i"; return; }
    if (s == "UInt32") { *dtype = FLOCKGPU_UINT32; *format = "I"; return; }
    if (s == "Int64") { *dtype = FLOCKGPU_INT64; *format = "l"; return; }
    if (s == "UInt64") { *dtype = FLOCKGPU_UINT64; *format = "L"; return; }
    if (s == "Float64") { *dtype = FLOCKGPU_FLOAT64; *format = "g"; return; }
    if (s == "Utf8") { *dtype = FLOCKGPU_UTF8; *format = "u"; return; }
    fail(FLOCKGPU_ERR_UNSUPPORTED, "plan JSON: data type %s is not supported on the GPU path", s.c_str());
  }
  if (j.is_object()) {
    if (const Json* ts = j.get("Timestamp")) {
      // {"Timestamp": ["Millisecond", null | "tz"]}
      std::string unit = ts->is_array() && !ts->arr.empty() && ts->arr[0]->is_string() ? ts->arr[0]->str : "Millisecond";
      char u = unit == "Second" ? 's' : unit == "Millisecond" ? 'm' : unit == "Microsecond" ? 'u' : 'n';
      std::string tz = ts->is_array() && ts->arr.size() > 1 && ts->arr[1]->is_string() ? ts->arr[1]->str : "";
      *dtype = FLOCKGPU_TIMESTAMP;
      *format = std::string("ts") + u + ":" + tz;
      return;
    }
  }
  fail(FLOCKGPU_ERR_UNSUPPORTED, "plan JSON: unsupported data type");
}

static Schema parse_schema(const Json& j) {
  Schema s;
  for (const JsonPtr& f : j.at("fields").arr) {
    Field fld;
    fld.name = f->at("name").as_string("field name");
    parse_data_type(f->at("data_type"), &fld.dtype, &fld.format);
    const Json* n = f->get("nullable");
    fld.nullable = n && n->kind == Json::Bool && n->b;
    s.fields.push_back(std::move(fld));
  }
  if (const Json* md = j.get("metadata")) {
    if (md->is_object() && !md->obj.empty()) {
      // encode as an Arrow metadata block
      std::string blk;
      int32_t n = int32_t(md->obj.size());
      blk.append(reinterpret_cast<const char*>(&n), 4);
      for (const auto& kv : md->obj) {
        int32_t kl = int32_t(kv.first.size());
        std::string v = kv.second->is_string() ? kv.second->str : "";
        int32_t vl = int32_t(v.size());
        blk.append(reinterpret_cast<const char*>(&kl), 4);
        blk.append(kv.first);
        blk.append(reinterpret_cast<const char*>(&vl), 4);
        blk.append(v);
      }
      s.metadata = blk;
    }
  }
  return s;
}

static int resolve_column(const fg::Table& in, const std::string& name, int index) {
  if (index >= 0 && index < int(in.cols.size()) && in.cols[index].name == name) return index;
  for (size_t i = 0; i < in.cols.size(); ++i)
    if (in.cols[i].name == name) return int(i);
  if (index >= 0 && index < int(in.cols.size())) return index;
  fail(FLOCKGPU_ERR_INVALID, "plan: column \"%s\" (index %d) not found in an input of %zu columns", name.c_str(), index, in.cols.size());
}

static int column_of(const Json& e, const fg::Table& in) {
  const Json* idx = e.get("index");
  return resolve_column(in, e.at("name").as_string("column name"), idx ? int(idx->as_int("column index")) : -1);
}

static bool is_column_expr(const Json& e) {
  const Json* k = e.get("physical_expr");
  return k && k->is_string() && k->str == "column";
}

static ExprTok scalar_token(const Json& value) {
  if (!value.is_object() || value.obj.size() != 1) fail(FLOCKGPU_ERR_INVALID, "plan JSON: malformed ScalarValue");
  const std::string& ty = value.obj[0].first;
  const Json& v = *value.obj[0].second;
  if (v.is_null()) fail(FLOCKGPU_ERR_UNSUPPORTED, "plan: NULL literal of type %s", ty.c_str());
  ExprTok t{};
  if (ty == "Float64" || ty == "Float32") {
    t.op = FLOCKGPU_OP_LIT_F64;
    t.dtype = FLOCKGPU_FLOAT64;
    t.f64 = v.num;
  } else if (ty == "Utf8" || ty == "LargeUtf8") {
    t.op = FLOCKGPU_OP_LIT_UTF8;
    t.dtype = FLOCKGPU_UTF8;
    t.str = v.as_string("Utf8 literal");
  } else if (ty == "Int8" || ty == "Int16" || ty == "Int32" || ty == "Int64" || ty == "UInt8" || ty == "UInt16" || ty == "UInt32" || ty == "UInt64" ||
             ty == "TimestampMillisecond" || ty == "TimestampSecond" || ty == "TimestampMicrosecond" || ty == "TimestampNanosecond") {
    t.op = FLOCKGPU_OP_LIT_I64;
    t.i64 = v.as_int("integer literal");
    t.dtype = ty == "Int32" ? FLOCKGPU_INT32 : ty == "UInt32" ? FLOCKGPU_UINT32 : ty == "UInt64" ? FLOCKGPU_UINT64
              : ty.rfind("Timestamp", 0) == 0 ? FLOCKGPU_TIMESTAMP : FLOCKGPU_INT64;
  } else {
    fail(FLOCKGPU_ERR_UNSUPPORTED, "plan: literal of type %s", ty.c_str());
  }
  return t;
}

static int binary_op(const std::string& op) {
  static const std::pair<const char*, int> table[] = {
      {"Eq", FLOCKGPU_OP_EQ}, {"NotEq", FLOCKGPU_OP_NE}, {"Lt", FLOCKGPU_OP_LT}, {"LtEq", FLOCKGPU_OP_LE}, {"Gt", FLOCKGPU_OP_GT},
      {"GtEq", FLOCKGPU_OP_GE}, {"Plus", FLOCKGPU_OP_ADD}, {"Minus", FLOCKGPU_OP_SUB}, {"Multiply", FLOCKGPU_OP_MUL},
      {"Divide", FLOCKGPU_OP_DIV}, {"Modulo", FLOCKGPU_OP_MOD}, {"Modulus", FLOCKGPU_OP_MOD}, {"And", FLOCKGPU_OP_AND}, {"Or", FLOCKGPU_OP_OR}};
  for (const auto& kv : table)
    if (op == kv.first) return kv.second;
  fail(FLOCKGPU_ERR_UNSUPPORTED, "plan: binary operator %s", op.c_str());
}

static void emit_expr(const Json& e, const fg::Table& in, Expr* out) {
  const std::string& kind = e.at("physical_expr").as_string("physical_expr tag");
  if (kind == "column") {
    ExprTok t{};
    t.op = FLOCKGPU_OP_COLUMN;
    t.col = column_of(e, in);
    out->push_back(t);
  } else if (kind == "literal") {
    out->push_back(scalar_token(e.at("value")));
  } else if (kind == "cast_expr" || kind == "try_cast_expr") {
    emit_expr(e.at("expr"), in, out);
    ExprTok t{};
    t.op = FLOCKGPU_OP_CAST;
    std::string fmt;
    parse_data_type(e.at("cast_type"), &t.dtype, &fmt);
    out->push_back(t);
  } else if (kind == "binary_expr") {
    emit_expr(e.at("left"), in, out);
    emit_expr(e.at("right"), in, out);
    ExprTok t{};
    t.op = binary_op(e.at("op").as_string("binary operator"));
    out->push_back(t);
  } else if (kind == "not_expr" || kind == "not") {
    emit_expr(e.get("arg") ? e.at("arg") : e.at("expr"), in, out);
    ExprTok t{};
    t.op = FLOCKGPU_OP_NOT;
    out->push_back(t);
  } else {
    fail(FLOCKGPU_ERR_UNSUPPORTED, "plan: physical expression \"%s\" is not supported on the GPU path", kind.c_str());
  }
}

static std::string data_type_display(const Json& j) {
  if (j.is_string()) return j.str;
  if (j.is_object() && j.get("Timestamp")) return "Timestamp(Millisecond, None)";
  return "?";
}

static std::string expr_display(const Json& e) {
  const Json* k = e.get("physical_expr");
  if (!k || !k->is_string()) return "?";
  const std::string& kind = k->str;
  if (kind == "column") {
    const Json* idx = e.get("index");
    std::string s = e.at("name").str;
    if (idx) s += "@" + std::to_string(idx->as_int("index"));
    return s;
  }
  if (kind == "literal") {
    const Json& v = e.at("value");
    if (v.is_object() && v.obj.size() == 1) {
      const Json& x = *v.obj[0].second;
      if (x.is_string()) return x.str;
      if (x.kind == Json::Number) {
        char buf[64];
        if (x.is_int) snprintf(buf, sizeof buf, "%lld", (long long)x.i64);
        else snprintf(buf, sizeof buf, "%g", x.num);
        return buf;
      }
    }
    return "NULL";
  }
  if (kind == "cast_expr" || kind == "try_cast_expr") return "CAST(" + expr_display(e.at("expr")) + " AS " + data_type_display(e.at("cast_type")) + ")";
  if (kind == "binary_expr") {
    static const std::pair<const char*, const char*> sym[] = {{"Eq", "="}, {"NotEq", "!="}, {"Lt", "<"}, {"LtEq", "<="}, {"Gt", ">"},
                                                               {"GtEq", ">="}, {"Plus", "+"}, {"Minus", "-"}, {"Multiply", "*"}, {"Divide", "/"},
                                                               {"Modulo", "%"}, {"Modulus", "%"}, {"And", "AND"}, {"Or", "OR"}};
    std::string op = e.at("op").str;
    for (const auto& kv : sym)
      if (op == kv.first) op = kv.second;
    return expr_display(e.at("left")) + " " + op + " " + expr_display(e.at("right"));
  }
  return kind;
}

// ------------------------------------------------------------------------------------------------
// nodes
// ------------------------------------------------------------------------------------------------
std::vector<std::string> MemoryExec::projected_names() const {
  std::vector<std::string> names;
  bool in_range = has_projection;
  for (int p : projection) in_range &= p >= 0 && p < int(full_schema.fields.size());
  if (has_projection && in_range) {
    for (int p : projection) names.push_back(full_schema.fields[p].name);
  } else {
    for (const Field& f : full_schema.fields) names.push_back(f.name);  // schema is already the projected one
  }
  return names;
}

std::string MemoryExec::fmt_as() const { return std::string("MemoryExec: partitions=") + (fed ? "1" : "0") + ", gpu_resident_rows=" + std::to_string(fed ? fed->num_rows : 0); }

TablePtr MemoryExec::execute(const ExecEnv& env) {
  if (fed) return fed;
  // never fed (or cleaned): an empty relation with the projected schema (context.rs:310-323)
  auto t = std::make_shared<fg::Table>();
  t->ctx = env.ctx;
  t->metadata = full_schema.metadata;
  std::vector<std::string> names = projected_names();
  for (const std::string& n : names) {
    for (const Field& f : full_schema.fields) {
      if (f.name != n) continue;
      fg::Column c;
      c.name = f.name;
      c.dtype = f.dtype;
      c.format = f.format;
      c.nullable = f.nullable;
      c.data = fg::alloc(env.ctx, 0);
      if (c.dtype == FLOCKGPU_UTF8) {
        c.offsets = fg::alloc(env.ctx, 4);
        FG_CUDA(cudaMemsetAsync(c.offsets->ptr, 0, 4, env.ctx->stream));
      }
      t->cols.push_back(std::move(c));
      break;
    }
  }
  return t;
}

static ExecutionPlan* skip_passthrough(ExecutionPlan* p) {
  while (true) {
    if (auto* c = dynamic_cast<CoalesceBatchesExec*>(p)) { p = c->input.get(); continue; }
    if (auto* c = dynamic_cast<CoalescePartitionsExec*>(p)) { p = c->input.get(); continue; }
    return p;
  }
}

std::string ProjectionExec::fmt_as() const {
  std::string s = "ProjectionExec: expr=[";
  for (size_t i = 0; i < expr.size(); ++i) s += (i ? ", " : "") + expr_display(*expr[i].first) + " as " + expr[i].second;
  return s + "]";
}

TablePtr ProjectionExec::execute(const ExecEnv& env) {
  // ProjectionExec <- CoalesceBatchesExec <- FilterExec is ONE kernel pass on the GPU (planner.rs:120-124)
  FilterExec* filter = dynamic_cast<FilterExec*>(skip_passthrough(input.get()));
  TablePtr in = filter ? filter->input->execute(env) : input->execute(env);
  std::vector<Expr> projs;
  std::vector<std::string> names;
  for (const auto& e : expr) {
    Expr t;
    emit_expr(*e.first, *in, &t);
    projs.push_back(std::move(t));
    names.push_back(e.second);
  }
  if (filter) {
    Expr pred;
    emit_expr(*filter->predicate, *in, &pred);
    return fg::filter_project(env.ctx, in, &pred, projs, names);
  }
  return fg::filter_project(env.ctx, in, nullptr, projs, names);
}

std::string FilterExec::fmt_as() const { return "FilterExec: " + expr_display(*predicate); }

TablePtr FilterExec::execute(const ExecEnv& env) {
  TablePtr in = input->execute(env);
  Expr pred;
  emit_expr(*predicate, *in, &pred);
  return fg::filter_project(env.ctx, in, &pred, {}, {});
}

std::string CoalesceBatchesExec::fmt_as() const { return "CoalesceBatchesExec: target_batch_size=" + std::to_string(target_batch_size); }

TablePtr CoalescePartitionsExec::execute(const ExecEnv& env) {
  TablePtr in = input->execute(env);
  if (env.world == 1) return in;
  // "merge every partition into one": with one partition per GPU that is a gather to rank 0 (the other ranks
  // continue with an empty relation), done by the exchange with a constant destination.
  // A rank whose partition holds the state row of an aggregate over NO input carries NULL states (SUM / MIN / MAX /
  // AVG over zero rows, SURVEY.md Appendix C.7): a NULL state merges as "absent" in the reference, so the row stays
  // home (its COUNT state is 0, the identity of the merge).
  in->resolve();
  bool null_state = false;
  for (const fg::Column& c : in->cols) null_state |= c.all_null;
  if (null_state) in = fg::empty_like(env.ctx, *in);
  return fg::hash_exchange(env.ctx, in, {}, 0);
}

std::string RepartitionExec::fmt_as() const {
  if (!hash) return "RepartitionExec: partitioning=RoundRobinBatch(" + std::to_string(n_partitions) + ")";
  std::string s = "RepartitionExec: partitioning=Hash([";
  for (size_t i = 0; i < hash_exprs.size(); ++i) s += (i ? ", " : "") + expr_display(*hash_exprs[i]);
  return s + "], " + std::to_string(n_partitions) + ")";
}

std::vector<int> RepartitionExec::key_columns(const fg::Table& in) const {
  std::vector<int> keys;
  for (const Json* e : hash_exprs) {
    if (!is_column_expr(*e)) fail(FLOCKGPU_ERR_UNSUPPORTED, "RepartitionExec: only plain columns can be hash keys on the GPU path");
    keys.push_back(column_of(*e, in));
  }
  return keys;
}

TablePtr RepartitionExec::execute(const ExecEnv& env) {
  TablePtr in = input->execute(env);
  if (hash && env.world > 1) {
    // the inter-function shuffle of the reference (actor.rs:425-543): the partition kernel pushes every row into its
    // receiver's window over NVLink (exchange.cu).  An input that an earlier exchange already routed on the same
    // columns is in place: DataFusion 6 plans Hash([p_id, name]) for q8's aggregate and Hash([p_id]) for its join,
    // two shuffles where one suffices (routing hashes the fixed-width key columns, here p_id both times).
    in->resolve();
    const std::vector<int> keys = key_columns(*in);
    if (in->partition_world == env.world && !in->partitioned_on.empty()) {
      std::vector<std::string> want;
      for (int k : fg::routing_columns(*in, keys)) want.push_back(in->cols[k].name);
      if (want == in->partitioned_on) return in;
    }
    return fg::hash_exchange(env.ctx, in, keys);
  }
  return in;  // single device partition: nothing to move
}

static const char* mode_name(int mode) {
  switch (mode) {
    case FLOCKGPU_AGG_PARTIAL: return "Partial";
    case FLOCKGPU_AGG_FINAL: return "Final";
    case FLOCKGPU_AGG_FINAL_PARTITIONED: return "FinalPartitioned";
    default: return "Single";
  }
}

std::string HashAggregateExec::fmt_as() const {
  std::string s = std::string("HashAggregateExec: mode=") + mode_name(mode) + ", gby=[";
  for (size_t i = 0; i < group_expr.size(); ++i) s += (i ? ", " : "") + expr_display(*group_expr[i].first) + " as " + group_expr[i].second;
  s += "], aggr=[";
  for (size_t i = 0; i < aggr_expr.size(); ++i) s += (i ? ", " : "") + aggr_expr[i].name;
  return s + "]";
}

static std::vector<int> group_columns(const HashAggregateExec& n, const fg::Table& in) {
  std::vector<int> cols;
  for (const auto& g : n.group_expr) {
    if (!is_column_expr(*g.first)) fail(FLOCKGPU_ERR_UNSUPPORTED, "HashAggregateExec: group expressions must be plain columns on the GPU path");
    cols.push_back(column_of(*g.first, in));
  }
  return cols;
}

static TablePtr rename_columns(const ExecEnv& env, const TablePtr& t, const std::vector<std::string>& names) {
  bool same = true;
  for (size_t i = 0; i < names.size() && i < t->cols.size(); ++i) same &= names[i].empty() || t->cols[i].name == names[i];
  if (same) return t;
  t->resolve();
  auto r = std::make_shared<fg::Table>(*t);
  for (size_t i = 0; i < names.size() && i < r->cols.size(); ++i)
    if (!names[i].empty() && r->cols[i].name != names[i]) {
      for (std::string& p : r->partitioned_on)  // same values under a new name: the rows are still where they were routed
        if (p == r->cols[i].name) p = names[i];
      r->cols[i].name = names[i];
    }
  (void)env;
  return r;
}

// Structural signature of a subtree + identity of the buffers its leaves scan.
static void subtree_signature(ExecutionPlan* p, std::string* s) {
  s->append(p->name());
  if (auto* m = dynamic_cast<MemoryExec*>(p)) {
    char buf[64];
    const void* id = m->fed && !m->fed->cols.empty() ? m->fed->cols[0].values() : nullptr;
    snprintf(buf, sizeof buf, "@%p/%zu", id, m->fed ? m->fed->cols.size() : size_t(0));
    s->append(buf);
    for (const std::string& n : m->projected_names()) s->append("," + n);
  } else {
    s->append(":" + p->fmt_as());
  }
  s->push_back('(');
  for (const PlanPtr& c : p->children()) subtree_signature(c.get(), s);
  s->push_back(')');
}

TablePtr HashAggregateExec::execute(const ExecEnv& env) {
  std::string sig;
  if (env.memo) {
    subtree_signature(this, &sig);
    auto hit = env.memo->find(sig);
    if (hit != env.memo->end()) return hit->second;
  }
  TablePtr result = execute_uncached(env);
  if (env.memo) (*env.memo)[sig] = result;
  return result;
}

TablePtr HashAggregateExec::execute_uncached(const ExecEnv& env) {
  const bool final_mode = mode == FLOCKGPU_AGG_FINAL || mode == FLOCKGPU_AGG_FINAL_PARTITIONED;
  // ---- single-GPU fusion: Final*( Coalesce/Repartition ( Partial(x) ) ) == one SINGLE aggregate over x
  if (final_mode && env.world == 1) {
    ExecutionPlan* p = input.get();
    while (true) {
      p = skip_passthrough(p);
      if (auto* r = dynamic_cast<RepartitionExec*>(p)) { p = r->input.get(); continue; }
      break;
    }
    if (auto* partial = dynamic_cast<HashAggregateExec*>(p)) {
      if (partial->mode == FLOCKGPU_AGG_PARTIAL && partial->group_expr.size() == group_expr.size() && partial->aggr_expr.size() == aggr_expr.size()) {
        TablePtr in = partial->input->execute(env);
        std::vector<int> gcols = group_columns(*partial, *in);
        std::vector<fg::AggSpec> specs;
        for (size_t i = 0; i < partial->aggr_expr.size(); ++i) {
          const auto& a = partial->aggr_expr[i];
          int col = a.expr && is_column_expr(*a.expr) ? column_of(*a.expr, *in) : -1;
          if (a.func != FLOCKGPU_AGG_COUNT && col < 0) fail(FLOCKGPU_ERR_UNSUPPORTED, "HashAggregateExec: aggregate argument must be a plain column");
          specs.push_back(fg::AggSpec{a.func, col, aggr_expr[i].name});
        }
        TablePtr out = fg::hash_aggregate(env.ctx, in, FLOCKGPU_AGG_SINGLE, gcols, specs);
        std::vector<std::string> names;
        for (const auto& g : group_expr) names.push_back(g.second);
        return rename_columns(env, out, names);
      }
    }
  }
  TablePtr in = input->execute(env);
  std::vector<int> gcols = group_columns(*this, *in);
  // A Partial DISTINCT (no aggregate functions) ahead of a shuffle only exists to shrink what travels.  With Utf8 / wide
  // group keys it costs a full row-representative hash table (q8: 91 us for 2.5 M persons that are all different), so
  // ask a sample first: when (nearly) every key of the first 64 Ki rows is new, the rows themselves are the partial
  // result -- the Final stage removes whatever duplicates exist, exactly as it would after a real Partial.
  if (mode == FLOCKGPU_AGG_PARTIAL && env.world > 1 && aggr_expr.empty() && !gcols.empty()) {
    in->resolve();
    bool wide = gcols.size() > 2;
    int bytes = 0;
    for (int g : gcols) {
      wide |= in->cols[g].dtype == FLOCKGPU_UTF8;
      bytes += in->cols[g].width();
    }
    wide |= bytes > 8;
    if (wide && in->num_rows >= (int64_t(1) << 16) && fg::distinct_sample_duplicates(env.ctx, in, gcols) < 0.25) {
      std::vector<fg::Expr> projs;
      std::vector<std::string> names;
      for (size_t i = 0; i < gcols.size(); ++i) {
        fg::ExprTok t{};
        t.op = FLOCKGPU_OP_COLUMN;
        t.col = gcols[i];
        projs.push_back(fg::Expr{t});
        names.push_back(group_expr[i].second);
      }
      return fg::filter_project(env.ctx, in, nullptr, projs, names);
    }
  }
  std::vector<fg::AggSpec> specs;
  if (!final_mode) {
    for (const auto& a : aggr_expr) {
      int col = a.expr && is_column_expr(*a.expr) ? column_of(*a.expr, *in) : -1;
      if (a.func != FLOCKGPU_AGG_COUNT && col < 0) fail(FLOCKGPU_ERR_UNSUPPORTED, "HashAggregateExec: aggregate argument must be a plain column");
      specs.push_back(fg::AggSpec{a.func, col, a.name});
    }
  } else {
    // the partial output is [group columns..., state columns in aggregate order]
    int state = int(group_expr.size());
    for (const auto& a : aggr_expr) {
      specs.push_back(fg::AggSpec{a.func, state, a.name});
      state += a.func == FLOCKGPU_AGG_AVG ? 2 : 1;
    }
  }
  TablePtr out = fg::hash_aggregate(env.ctx, in, mode, gcols, specs);
  // A Final aggregate without group columns runs in ONE partition (behind CoalescePartitionsExec): with several GPUs
  // that partition lives on rank 0; the other ranks hold no partition of this node, hence no row.
  if (final_mode && group_expr.empty() && env.world > 1 && env.rank != 0) out = fg::empty_like(env.ctx, *out);
  std::vector<std::string> names;
  for (const auto& g : group_expr) names.push_back(g.second);
  return rename_columns(env, out, names);
}

// DataFusion 6 JoinType names, in the order of enum flockgpu_join_type
static const char* const kJoinTypeNames[] = {"Inner", "Left", "Right", "Full", "Semi", "Anti"};

std::string HashJoinExec::fmt_as() const {
  std::string s = "HashJoinExec: mode=" + mode + ", join_type=" + kJoinTypeNames[join_type] + ", on=[";
  for (size_t i = 0; i < on.size(); ++i) s += std::string(i ? ", " : "") + "(" + on[i].first.name + ", " + on[i].second.name + ")";
  return s + "]";
}

TablePtr HashJoinExec::execute(const ExecEnv& env) {
  // Across GPUs only a Partitioned join (the exchange brought each key's rows to one rank) may emit unmatched left rows:
  // with CollectLeft every rank holds the whole left side and each would emit its unmatched rows again.
  const bool keeps_left_rows = join_type == FLOCKGPU_JOIN_LEFT || join_type == FLOCKGPU_JOIN_FULL || join_type == FLOCKGPU_JOIN_SEMI ||
                               join_type == FLOCKGPU_JOIN_ANTI;
  if (env.world > 1 && keeps_left_rows && mode != "Partitioned")
    fail(FLOCKGPU_ERR_UNSUPPORTED, "HashJoinExec: join_type=%s in mode %s is not supported across GPUs (Partitioned only)", kJoinTypeNames[join_type], mode.c_str());
  TablePtr l = left->execute(env);
  TablePtr r = right->execute(env);
  std::vector<int> lk, rk;
  for (const auto& p : on) {
    lk.push_back(resolve_column(*l, p.first.name, p.first.index));
    rk.push_back(resolve_column(*r, p.second.name, p.second.index));
  }
  return fg::hash_join(env.ctx, l, r, lk, rk, join_type);
}

std::string SortExec::fmt_as() const {
  std::string s = "SortExec: [";
  for (size_t i = 0; i < expr.size(); ++i) s += (i ? ", " : "") + expr_display(*expr[i].expr) + (expr[i].descending ? " DESC" : " ASC");
  return s + "]";
}

TablePtr SortExec::execute(const ExecEnv& env) {
  TablePtr in = input->execute(env);
  in->resolve();
  std::vector<fg::SortKey> keys;
  for (const Key& k : expr) {
    if (!is_column_expr(*k.expr)) fail(FLOCKGPU_ERR_UNSUPPORTED, "SortExec: sort expressions must be plain columns on the GPU path");
    keys.push_back(fg::SortKey{column_of(*k.expr, *in), k.descending, k.nulls_first});
  }
  return fg::sort_table(env.ctx, in, keys);
}

TablePtr GlobalLimitExec::execute(const ExecEnv& env) { return fg::limit_rows(env.ctx, input->execute(env), limit); }

std::string WindowAggExec::fmt_as() const {
  std::string s = "WindowAggExec: wdw=[";
  for (size_t i = 0; i < window_expr.size(); ++i) s += (i ? ", " : "") + window_expr[i].name;
  return s + "]";
}

TablePtr WindowAggExec::execute(const ExecEnv& env) {
  TablePtr in = input->execute(env);
  in->resolve();
  // several window expressions: each adds its column in front, the first expression ends up first
  TablePtr out = in;
  for (auto w = window_expr.rbegin(); w != window_expr.rend(); ++w) {
    std::vector<int> part;
    for (const Json* e : w->partition_by) {
      if (!is_column_expr(*e)) fail(FLOCKGPU_ERR_UNSUPPORTED, "WindowAggExec: PARTITION BY expressions must be plain columns on the GPU path");
      part.push_back(column_of(*e, *in) + int(out->cols.size() - in->cols.size()));
    }
    out = fg::row_number(env.ctx, out, part, w->name);
  }
  return out;
}

// ------------------------------------------------------------------------------------------------
// plan construction from JSON
// ------------------------------------------------------------------------------------------------
static PlanPtr build_plan(const Json& j);

static PlanPtr build_input(const Json& j) { return build_plan(j.at("input")); }

static HashJoinExec::OnCol on_col(const Json& j) {
  HashJoinExec::OnCol c;
  if (j.is_string()) {
    c.name = j.str;
  } else {
    c.name = j.at("name").as_string("join column");
    if (const Json* idx = j.get("index")) c.index = int(idx->as_int("join column index"));
  }
  return c;
}

static int agg_func(const std::string& s) {
  if (s == "count") return FLOCKGPU_AGG_COUNT;
  if (s == "sum") return FLOCKGPU_AGG_SUM;
  if (s == "min") return FLOCKGPU_AGG_MIN;
  if (s == "max") return FLOCKGPU_AGG_MAX;
  if (s == "avg") return FLOCKGPU_AGG_AVG;
  fail(FLOCKGPU_ERR_UNSUPPORTED, "plan: aggregate function \"%s\" is not supported on the GPU path", s.c_str());
}

static PlanPtr build_plan(const Json& j) {
  const std::string& tag = j.at("execution_plan").as_string("execution_plan tag");
  if (tag == "memory_exec") {
    auto n = std::make_shared<MemoryExec>();
    n->full_schema = parse_schema(j.at("schema"));
    if (const Json* p = j.get("projection")) {
      if (p->is_array()) {
        n->has_projection = true;
        for (const JsonPtr& x : p->arr) n->projection.push_back(int(x->as_int("projection index")));
      }
    }
    return n;
  }
  if (tag == "projection_exec") {
    auto n = std::make_shared<ProjectionExec>();
    for (const JsonPtr& pair : j.at("expr").arr) {
      if (!pair->is_array() || pair->arr.size() != 2) fail(FLOCKGPU_ERR_INVALID, "plan JSON: projection expr must be [expr, name]");
      n->expr.emplace_back(pair->arr[0].get(), pair->arr[1]->as_string("projection name"));
    }
    n->input = build_input(j);
    return n;
  }
  if (tag == "filter_exec") {
    auto n = std::make_shared<FilterExec>();
    n->predicate = &j.at("predicate");
    n->input = build_input(j);
    return n;
  }
  if (tag == "coalesce_batches_exec") {
    auto n = std::make_shared<CoalesceBatchesExec>();
    if (const Json* t = j.get("target_batch_size")) n->target_batch_size = t->as_int("target_batch_size");
    n->input = build_input(j);
    return n;
  }
  if (tag == "coalesce_partitions_exec" || tag == "merge_exec") {
    auto n = std::make_shared<CoalescePartitionsExec>();
    n->input = build_input(j);
    return n;
  }
  if (tag == "repartition_exec") {
    auto n = std::make_shared<RepartitionExec>();
    const Json& part = j.at("partitioning");
    if (const Json* rr = part.get("RoundRobinBatch")) {
      n->n_partitions = int(rr->as_int("RoundRobinBatch"));
    } else if (const Json* h = part.get("Hash")) {
      if (!h->is_array() || h->arr.size() != 2) fail(FLOCKGPU_ERR_INVALID, "plan JSON: Hash partitioning must be [[exprs], n]");
      n->hash = true;
      for (const JsonPtr& e : h->arr[0]->arr) n->hash_exprs.push_back(e.get());
      n->n_partitions = int(h->arr[1]->as_int("Hash partition count"));
    } else {
      fail(FLOCKGPU_ERR_UNSUPPORTED, "plan: partitioning scheme is not supported on the GPU path (HashDiff / Unknown)");
    }
    n->input = build_input(j);
    return n;
  }
  if (tag == "hash_aggregate_exec") {
    auto n = std::make_shared<HashAggregateExec>();
    const std::string& m = j.at("mode").as_string("aggregate mode");
    n->mode = m == "Partial" ? FLOCKGPU_AGG_PARTIAL : m == "Final" ? FLOCKGPU_AGG_FINAL : m == "FinalPartitioned" ? FLOCKGPU_AGG_FINAL_PARTITIONED : -1;
    if (n->mode < 0) fail(FLOCKGPU_ERR_INVALID, "plan JSON: unknown aggregate mode %s", m.c_str());
    for (const JsonPtr& pair : j.at("group_expr").arr) {
      if (!pair->is_array() || pair->arr.size() != 2) fail(FLOCKGPU_ERR_INVALID, "plan JSON: group_expr must be [expr, name]");
      n->group_expr.emplace_back(pair->arr[0].get(), pair->arr[1]->as_string("group name"));
    }
    for (const JsonPtr& a : j.at("aggr_expr").arr) {
      HashAggregateExec::Aggr ag;
      ag.func = agg_func(a->at("aggregate_expr").as_string("aggregate_expr tag"));
      ag.expr = a->get("expr");
      ag.name = a->at("name").as_string("aggregate name");
      n->aggr_expr.push_back(ag);
    }
    n->input = build_input(j);
    return n;
  }
  if (tag == "hash_join_exec") {
    auto n = std::make_shared<HashJoinExec>();
    const std::string& jt = j.at("join_type").as_string("join_type");
    n->join_type = -1;
    for (int t = FLOCKGPU_JOIN_INNER; t <= FLOCKGPU_JOIN_ANTI; ++t)
      if (jt == kJoinTypeNames[t]) n->join_type = t;
    if (n->join_type < 0) fail(FLOCKGPU_ERR_INVALID, "plan JSON: unknown join_type %s", jt.c_str());
    if (const Json* m = j.get("mode")) n->mode = m->is_string() ? m->str : "Partitioned";
    for (const JsonPtr& pair : j.at("on").arr) {
      if (!pair->is_array() || pair->arr.size() != 2) fail(FLOCKGPU_ERR_INVALID, "plan JSON: join `on` entries must be pairs");
      n->on.emplace_back(on_col(*pair->arr[0]), on_col(*pair->arr[1]));
    }
    n->left = build_plan(j.at("left"));
    n->right = build_plan(j.at("right"));
    return n;
  }
  if (tag == "sort_exec") {
    auto n = std::make_shared<SortExec>();
    for (const JsonPtr& e : j.at("expr").arr) {
      SortExec::Key k;
      k.expr = &e->at("expr");
      if (const Json* o = e->get("options")) {
        const Json* d = o->get("descending");
        const Json* nf = o->get("nulls_first");
        k.descending = d && d->kind == Json::Bool && d->b;
        k.nulls_first = nf && nf->kind == Json::Bool && nf->b;
      }
      n->expr.push_back(k);
    }
    if (n->expr.empty()) fail(FLOCKGPU_ERR_INVALID, "plan JSON: sort_exec without sort expressions");
    n->input = build_input(j);
    return n;
  }
  if (tag == "global_limit_exec") {
    auto n = std::make_shared<GlobalLimitExec>();
    n->limit = j.at("limit").as_int("limit");
    n->input = build_input(j);
    return n;
  }
  if (tag == "window_agg_exec") {
    auto n = std::make_shared<WindowAggExec>();
    for (const JsonPtr& w : j.at("window_expr").arr) {
      const Json* fun = w->get("fun");
      if (!fun || !fun->is_string() || fun->str != "RowNumber")
        fail(FLOCKGPU_ERR_UNSUPPORTED, "plan: window function %s is not supported on the GPU path (ROW_NUMBER only)", fun && fun->is_string() ? fun->str.c_str() : "?");
      WindowAggExec::Win win;
      win.name = w->at("name").as_string("window expression name");
      if (const Json* pb = w->get("partition_by"))
        for (const JsonPtr& e : pb->arr) win.partition_by.push_back(e.get());
      n->window_expr.push_back(std::move(win));
    }
    n->input = build_input(j);
    return n;
  }
  fail(FLOCKGPU_ERR_UNSUPPORTED, "plan: execution plan node \"%s\" is not supported on the GPU path", tag.c_str());
}

std::unique_ptr<ExecutionContext> ExecutionContext::unmarshal(const CtxPtr& ctx, const char* text) {
  auto ec = std::make_unique<ExecutionContext>();
  ec->ctx = ctx;
  ec->json = JsonParser(text).parse();
  const Json* root = ec->json.get();
  std::vector<const Json*> plans;
  if (root->is_array()) {
    for (const JsonPtr& p : root->arr) plans.push_back(p.get());
  } else if (root->is_object() && root->get("execution_plan")) {
    plans.push_back(root);
  } else if (root->is_object() && root->get("plan")) {
    // a marshalled ExecutionContext { plan: { execution_plans: [...] }, name, next, .. }
    for (const JsonPtr& p : root->at("plan").at("execution_plans").arr) plans.push_back(p.get());
    if (const Json* n = root->get("name")) ec->name = n->is_string() ? n->str : "";
  } else {
    fail(FLOCKGPU_ERR_INVALID, "unmarshal: expected a plan object, an array of plans or an ExecutionContext object");
  }
  if (plans.empty()) fail(FLOCKGPU_ERR_INVALID, "unmarshal: no execution plans");
  for (const Json* p : plans) ec->execution_plans.push_back(build_plan(*p));
  return ec;
}

ExecEnv ExecutionContext::env() const {
  ExecEnv e;
  e.ctx = ctx;
  e.world = fg::comm_world(ctx);
  e.rank = fg::comm_rank(ctx);
  e.memo = std::make_shared<std::map<std::string, TablePtr>>();
  return e;
}

std::vector<MemoryExec*> ExecutionContext::leaves_bfs() const {
  // breadth-first over all plans, like context.rs:262-266
  std::vector<MemoryExec*> leaves;
  std::deque<ExecutionPlan*> queue;
  for (const PlanPtr& p : execution_plans) queue.push_back(p.get());
  while (!queue.empty()) {
    ExecutionPlan* p = queue.front();
    queue.pop_front();
    std::vector<PlanPtr> ch = p->children();
    if (ch.empty()) {
      if (auto* m = dynamic_cast<MemoryExec*>(p)) leaves.push_back(m);
    }
    for (const PlanPtr& c : ch) queue.push_back(c.get());
  }
  return leaves;
}

// compare_schema (context.rs:402-416): the smaller field-name set must be contained in the larger
static bool compare_schema(const std::vector<std::string>& a, const std::vector<std::string>& b) {
  const std::vector<std::string>& sup = a.size() >= b.size() ? a : b;
  const std::vector<std::string>& sub = a.size() >= b.size() ? b : a;
  std::set<std::string> names(sup.begin(), sup.end());
  for (const std::string& s : sub)
    if (!names.count(s)) return false;
  return true;
}

static TablePtr project_by_name(const CtxPtr& ctx, const TablePtr& t, const std::vector<std::string>& names) {
  t->dense();
  auto out = std::make_shared<fg::Table>();
  out->ctx = ctx;
  out->metadata = t->metadata;
  out->num_rows = t->num_rows;
  for (const std::string& n : names) {
    bool found = false;
    for (const fg::Column& c : t->cols)
      if (c.name == n) {
        out->cols.push_back(c);  // zero-copy: shares the HBM buffers
        found = true;
        break;
      }
    if (!found) fail(FLOCKGPU_ERR_INVALID, "feed_data_sources: the fed relation has no column \"%s\" required by the plan's MemoryExec", n.c_str());
  }
  return out;
}

void ExecutionContext::feed_tables(std::vector<TablePtr> sources) {
  for (MemoryExec* leaf : leaves_bfs()) {
    std::vector<std::string> want = leaf->projected_names();
    int found = -1;
    for (size_t i = 0; i < sources.size(); ++i) {
      std::vector<std::string> have;
      for (const fg::Column& c : sources[i]->cols) have.push_back(c.name);
      if (compare_schema(want, have)) {
        found = int(i);
        break;
      }
    }
    if (found >= 0) {
      leaf->fed = project_by_name(ctx, sources[found], want);
      sources.erase(sources.begin() + found);
    } else {
      leaf->fed = nullptr;  // executes as an empty relation
    }
  }
}

void ExecutionContext::feed_data_sources(const ArrowSchema* const* schemas, const ArrowArray* const* const* batches, const int32_t* n_batches,
                                         int n_sources) {
  struct Src {
    const ArrowSchema* schema;
    const ArrowArray* const* batches;
    int n;
    std::vector<std::string> names;
  };
  std::vector<Src> sources;
  for (int i = 0; i < n_sources; ++i) {
    FG_CHECK(schemas[i] && schemas[i]->format && !strcmp(schemas[i]->format, "+s"), FLOCKGPU_ERR_INVALID, "feed_data_sources: source %d is not a struct schema", i);
    Src s{schemas[i], batches[i], n_batches[i], {}};
    for (int64_t c = 0; c < schemas[i]->n_children; ++c) s.names.push_back(schemas[i]->children[c]->name ? schemas[i]->children[c]->name : "");
    sources.push_back(std::move(s));
  }
  std::map<std::string, TablePtr> imported;
  for (MemoryExec* leaf : leaves_bfs()) {
    std::vector<std::string> want = leaf->projected_names();
    int found = -1;
    for (size_t i = 0; i < sources.size(); ++i)
      if (compare_schema(want, sources[i].names)) {
        found = int(i);
        break;
      }
    if (found < 0) {
      leaf->fed = nullptr;
      continue;
    }
    const Src& s = sources[found];
    // projection pushdown: only the columns the leaf scans cross PCIe
    std::vector<int> proj;
    for (const std::string& n : want) {
      auto it = std::find(s.names.begin(), s.names.end(), n);
      FG_CHECK(it != s.names.end(), FLOCKGPU_ERR_INVALID, "feed_data_sources: the fed relation has no column \"%s\" required by the plan", n.c_str());
      proj.push_back(int(it - s.names.begin()));
    }
    // The same host batches fed for two leaves (q5 scans `bid` twice, and feed_data_sources hands one source to
    // one leaf, context.rs:293-303) cross PCIe once: identical (buffers, projection) reuse the imported table.
    std::string key;
    for (int p : proj) key += std::to_string(p) + ",";
    for (int b = 0; b < s.n; ++b) {
      char buf[64];
      const ArrowArray* first = s.batches[b]->n_children > 0 ? s.batches[b]->children[proj.empty() ? 0 : proj[0]] : nullptr;
      snprintf(buf, sizeof buf, "|%p:%lld:%lld", first && first->n_buffers > 1 ? first->buffers[1] : nullptr, (long long)s.batches[b]->length,
               (long long)(first ? first->offset : 0));
      key += buf;
    }
    auto hit = imported.find(key);
    if (hit != imported.end()) {
      leaf->fed = hit->second;
    } else {
      leaf->fed = fg::import_batches(ctx, s.schema, s.batches, s.n, proj.data(), int(proj.size()), ctx->feed_zero_copy);
      imported[key] = leaf->fed;
    }
    sources.erase(sources.begin() + found);
  }
}

TablePtr ExecutionContext::execute(int plan_index) {
  FG_CHECK(plan_index >= 0 && plan_index < int(execution_plans.size()), FLOCKGPU_ERR_INVALID, "execute: plan index %d out of range", plan_index);
  return execution_plans[plan_index]->execute(env());
}

std::vector<TablePtr> ExecutionContext::execute_partitioned(int plan_index) {
  FG_CHECK(plan_index >= 0 && plan_index < int(execution_plans.size()), FLOCKGPU_ERR_INVALID, "execute_partitioned: plan index %d out of range", plan_index);
  ExecutionPlan* root = execution_plans[plan_index].get();
  // a shuffle stage is CoalesceBatchesExec <- RepartitionExec(Hash(keys, n)) (planner.rs:151-163): its n output
  // partitions are what the next stage's functions receive
  if (auto* cb = dynamic_cast<CoalesceBatchesExec*>(root)) {
    if (auto* rp = dynamic_cast<RepartitionExec*>(cb->input.get())) {
      if (rp->hash) {
        TablePtr in = rp->input->execute(env());
        return fg::hash_partition(ctx, in, rp->key_columns(*in), rp->n_partitions);
      }
    }
  }
  return {root->execute(env())};
}

void ExecutionContext::clean_data_sources() {
  for (MemoryExec* leaf : leaves_bfs()) leaf->fed = nullptr;
}

bool ExecutionContext::is_shuffling() const {
  if (execution_plans.empty()) return false;
  for (const PlanPtr& p : execution_plans) {
    auto* cb = dynamic_cast<CoalesceBatchesExec*>(p.get());
    if (!cb || !dynamic_cast<RepartitionExec*>(cb->input.get())) return false;
  }
  return true;
}

static void render(const ExecutionPlan* p, int depth, std::string* out) {
  out->append(size_t(depth) * 2, ' ');
  out->append(p->fmt_as());
  out->push_back('\n');
  for (const PlanPtr& c : p->children()) render(c.get(), depth + 1, out);
}

std::string ExecutionContext::plan_str(int plan_index) const {
  FG_CHECK(plan_index >= 0 && plan_index < int(execution_plans.size()), FLOCKGPU_ERR_INVALID, "plan_str: plan index %d out of range", plan_index);
  std::string s;
  render(execution_plans[plan_index].get(), 0, &s);
  return s;
}

}  // namespace flock

// ================================================================================================
// extern "C"
// ================================================================================================
struct flock_context {
  std::unique_ptr<flock::ExecutionContext> ec;
};

using namespace fg;

template <typename F>
static int guarded_ec(flock_context* h, F&& body) {
  return guarded([&] {
    FG_CHECK(h && h->ec, FLOCKGPU_ERR_INVALID, "null flock_context handle");
    FG_CHECK(h->ec->ctx, FLOCKGPU_ERR_NO_DEVICE,
             "this flock_context was unmarshalled without a flockgpu_ctx (parse-only); it cannot feed or execute -- there is no CPU fallback");
    std::lock_guard<std::recursive_mutex> g(h->ec->ctx->mu);
    FG_CUDA(cudaSetDevice(h->ec->ctx->device));
    body(*h->ec);
  });
}

extern "C" {

int flock_context_unmarshal(flockgpu_ctx* ctx, const char* plans_json, flock_context** out) {
  return guarded([&] {
    // ctx == NULL gives a parse-only context (plan_str / is_shuffling / num_plans work, execution does not)
    CtxPtr c = ctx ? core_of(ctx) : nullptr;
    FG_CHECK(plans_json && out, FLOCKGPU_ERR_INVALID, "unmarshal: null argument");
    auto h = std::make_unique<flock_context>();
    h->ec = flock::ExecutionContext::unmarshal(c, plans_json);
    *out = h.release();
  });
}

int flock_context_free(flock_context* ec) {
  return guarded([&] {
    if (ec && ec->ec && ec->ec->ctx) cudaSetDevice(ec->ec->ctx->device);
    delete ec;
  });
}

int32_t flock_context_num_plans(const flock_context* ec) { return ec && ec->ec ? int32_t(ec->ec->execution_plans.size()) : -1; }

int flock_context_feed_data_sources(flock_context* ec, const struct ArrowSchema* const* schemas, const struct ArrowArray* const* const* batches,
                                    const int32_t* n_batches, int32_t n_sources) {
  return guarded_ec(ec, [&](flock::ExecutionContext& e) {
    FG_CHECK(n_sources >= 0 && (n_sources == 0 || (schemas && batches && n_batches)), FLOCKGPU_ERR_INVALID, "feed_data_sources: bad arguments");
    e.feed_data_sources(schemas, batches, n_batches, n_sources);
  });
}

int flock_context_feed_tables(flock_context* ec, flockgpu_table* const* tables, int32_t n_sources) {
  return guarded_ec(ec, [&](flock::ExecutionContext& e) {
    std::vector<TablePtr> src;
    for (int i = 0; i < n_sources; ++i) {
      FG_CHECK(tables && tables[i] && tables[i]->table, FLOCKGPU_ERR_INVALID, "feed_tables: null table");
      src.push_back(tables[i]->table);
    }
    e.feed_tables(std::move(src));
  });
}

int flock_context_execute(flock_context* ec, int32_t plan_index, flockgpu_table** out) {
  return guarded_ec(ec, [&](flock::ExecutionContext& e) {
    FG_CHECK(out, FLOCKGPU_ERR_INVALID, "execute: null out pointer");
    *out = wrap_table(e.execute(plan_index));
  });
}

int flock_context_execute_partitioned(flock_context* ec, int32_t plan_index, flockgpu_table** out_parts, int32_t max_parts, int32_t* n_parts) {
  return guarded_ec(ec, [&](flock::ExecutionContext& e) {
    FG_CHECK(out_parts && n_parts, FLOCKGPU_ERR_INVALID, "execute_partitioned: null out pointer");
    std::vector<TablePtr> parts = e.execute_partitioned(plan_index);
    FG_CHECK(int(parts.size()) <= max_parts, FLOCKGPU_ERR_INVALID, "execute_partitioned: %zu partitions, room for %d", parts.size(), max_parts);
    for (size_t i = 0; i < parts.size(); ++i) out_parts[i] = wrap_table(parts[i]);
    *n_parts = int32_t(parts.size());
  });
}

int flock_context_clean_data_sources(flock_context* ec) {
  return guarded_ec(ec, [&](flock::ExecutionContext& e) { e.clean_data_sources(); });
}

int flock_context_is_shuffling(const flock_context* ec, int32_t* out) {
  return guarded([&] {
    FG_CHECK(ec && ec->ec && out, FLOCKGPU_ERR_INVALID, "is_shuffling: null argument");
    *out = ec->ec->is_shuffling() ? 1 : 0;
  });
}

const char* flock_context_plan_str(flock_context* ec, int32_t plan_index) {
  if (!ec || !ec->ec) return "";
  int rc = guarded([&] { ec->ec->plan_str_cache = ec->ec->plan_str(plan_index); });
  return rc == 0 ? ec->ec->plan_str_cache.c_str() : "";
}

}  // extern "C"
