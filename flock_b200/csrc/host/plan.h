// plan.h -- the host-side mirror of the reference's operator interface for the hot path.
//
// The reference keeps `Arc<dyn ExecutionPlan>` trees (DataFusion fork) inside
// `CloudExecutionPlan.execution_plans` (flock/src/runtime/plan.rs:139-146) and drives them through
// `ExecutionContext::{feed_data_sources, execute, execute_partitioned, clean_data_sources}`
// (flock/src/runtime/context.rs:172-325).  This layer rebuilds those trees from the reference's own
// serde-JSON serialisation (context.rs:366-398; fixtures flock/src/tests/data/plan/*.json) with node
// classes of the same names, and executes them on the GPU through the operators of internal.h.
//
// On the GPU a plan runs with ONE partition per device: RoundRobinBatch repartitioning, batch
// coalescing and partition merging exist in the reference only to spread work over CPU cores and
// carry no values (SURVEY.md section 8 a5/a8/a9), so those nodes forward their input.
#pragma once

#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../internal.h"
#include "json.h"

namespace flock {

using fg::CtxPtr;
using fg::TablePtr;

struct Field {
  std::string name;
  int dtype = FLOCKGPU_INT32;
  std::string format;
  bool nullable = false;
};

struct Schema {
  std::vector<Field> fields;
  std::string metadata;  // raw Arrow metadata block
};

class ExecutionPlan;
using PlanPtr = std::shared_ptr<ExecutionPlan>;

// What a node may ask of the context while executing.
struct ExecEnv {
  CtxPtr ctx;
  int world = 1;  // > 1 when an NCCL communicator is attached: Hash repartitioning becomes an all-to-all
  int rank = 0;
  // Results of aggregate subtrees already computed during THIS execution, keyed by the subtree's structure and
  // the identity of the HBM buffers its leaves scan.  DataFusion 6 has no common-subexpression elimination, so
  // NEXMark q5 plans the COUNT-by-auction subtree twice (benchmarks/src/nexmark/query/q5_plan.fmt); computing it
  // once cannot change a value (tables are immutable).
  std::shared_ptr<std::map<std::string, TablePtr>> memo;
};

class ExecutionPlan {
 public:
  virtual ~ExecutionPlan() = default;
  virtual const char* name() const = 0;  // "FilterExec", "HashJoinExec", ...
  virtual std::vector<PlanPtr> children() const = 0;
  virtual std::string fmt_as() const = 0;  // the one-line DisplayFormatType::Default rendering
  // Executes the node's single device partition.
  virtual TablePtr execute(const ExecEnv& env) = 0;
};

class MemoryExec : public ExecutionPlan {
 public:
  Schema full_schema;            // schema of the registered table
  std::vector<int> projection;   // indices into full_schema (empty + has_projection=false: all)
  bool has_projection = false;
  TablePtr fed;                  // set by feed_data_sources, dropped by clean_data_sources
  std::vector<std::string> projected_names() const;
  const char* name() const override { return "MemoryExec"; }
  std::vector<PlanPtr> children() const override { return {}; }
  std::string fmt_as() const override;
  TablePtr execute(const ExecEnv& env) override;
};

class UnaryExec : public ExecutionPlan {
 public:
  PlanPtr input;
  std::vector<PlanPtr> children() const override { return {input}; }
};

class ProjectionExec : public UnaryExec {
 public:
  std::vector<std::pair<const Json*, std::string>> expr;
  const char* name() const override { return "ProjectionExec"; }
  std::string fmt_as() const override;
  TablePtr execute(const ExecEnv& env) override;
};

class FilterExec : public UnaryExec {
 public:
  const Json* predicate = nullptr;
  const char* name() const override { return "FilterExec"; }
  std::string fmt_as() const override;
  TablePtr execute(const ExecEnv& env) override;
};

class CoalesceBatchesExec : public UnaryExec {
 public:
  int64_t target_batch_size = 4096;
  const char* name() const override { return "CoalesceBatchesExec"; }
  std::string fmt_as() const override;
  TablePtr execute(const ExecEnv& env) override { return input->execute(env); }
};

class CoalescePartitionsExec : public UnaryExec {
 public:
  const char* name() const override { return "CoalescePartitionsExec"; }
  std::string fmt_as() const override { return "CoalescePartitionsExec"; }
  TablePtr execute(const ExecEnv& env) override;
};

class RepartitionExec : public UnaryExec {
 public:
  bool hash = false;
  int n_partitions = 1;
  std::vector<const Json*> hash_exprs;  // Hash only
  const char* name() const override { return "RepartitionExec"; }
  std::string fmt_as() const override;
  TablePtr execute(const ExecEnv& env) override;
  std::vector<int> key_columns(const fg::Table& in) const;
};

class HashAggregateExec : public UnaryExec {
 public:
  int mode = FLOCKGPU_AGG_PARTIAL;
  std::vector<std::pair<const Json*, std::string>> group_expr;
  struct Aggr {
    int func;
    const Json* expr;
    std::string name;
  };
  std::vector<Aggr> aggr_expr;
  const char* name() const override { return "HashAggregateExec"; }
  std::string fmt_as() const override;
  TablePtr execute(const ExecEnv& env) override;
  TablePtr execute_uncached(const ExecEnv& env);
};

class HashJoinExec : public ExecutionPlan {
 public:
  PlanPtr left, right;
  struct OnCol {
    std::string name;
    int index = -1;
  };
  std::vector<std::pair<OnCol, OnCol>> on;
  std::string mode = "Partitioned";
  int join_type = FLOCKGPU_JOIN_INNER;  // DataFusion 6 JoinType; "Inner" ... "Anti" in the plan JSON
  const char* name() const override { return "HashJoinExec"; }
  std::vector<PlanPtr> children() const override { return {left, right}; }
  std::string fmt_as() const override;
  TablePtr execute(const ExecEnv& env) override;
};

class SortExec : public UnaryExec {
 public:
  struct Key {
    const Json* expr;
    bool descending = false, nulls_first = false;
  };
  std::vector<Key> expr;
  const char* name() const override { return "SortExec"; }
  std::string fmt_as() const override;
  TablePtr execute(const ExecEnv& env) override;
};

class GlobalLimitExec : public UnaryExec {
 public:
  int64_t limit = 0;
  const char* name() const override { return "GlobalLimitExec"; }
  std::string fmt_as() const override { return "GlobalLimitExec: limit=" + std::to_string(limit); }
  TablePtr execute(const ExecEnv& env) override;
};

// WindowAggExec with ROW_NUMBER() window expressions (the only window function NEXMark uses, q6)
class WindowAggExec : public UnaryExec {
 public:
  struct Win {
    std::string name;
    std::vector<const Json*> partition_by;
  };
  std::vector<Win> window_expr;
  const char* name() const override { return "WindowAggExec"; }
  std::string fmt_as() const override;
  TablePtr execute(const ExecEnv& env) override;
};

// flock::runtime::context::ExecutionContext (only the members that touch the hot path)
class ExecutionContext {
 public:
  CtxPtr ctx;
  JsonPtr json;  // owns every `const Json*` referenced by the nodes
  std::vector<PlanPtr> execution_plans;
  std::string name;
  std::string plan_str_cache;

  static std::unique_ptr<ExecutionContext> unmarshal(const CtxPtr& ctx, const char* text);
  // context.rs:257-325.  A source is one relation already resident in HBM with its FULL schema.
  void feed_tables(std::vector<TablePtr> sources);
  void feed_data_sources(const ArrowSchema* const* schemas, const ArrowArray* const* const* batches, const int32_t* n_batches, int n_sources);
  TablePtr execute(int plan_index);                             // context.rs:172-191
  std::vector<TablePtr> execute_partitioned(int plan_index);    // context.rs:197-216
  void clean_data_sources();                                    // context.rs:227-254
  bool is_shuffling() const;                                    // context.rs:328-337
  std::string plan_str(int plan_index) const;

 private:
  ExecEnv env() const;
  std::vector<MemoryExec*> leaves_bfs() const;
};

}  // namespace flock
