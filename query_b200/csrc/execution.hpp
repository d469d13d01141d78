// execution.hpp — host-side mirror of the reference's plan.Visitor / execution.Operator contract for the
// substituted chain.  In the real integration this layer is Go (package `execution`, see INTEGRATION.md);
// Go cannot be compiled in this image, so the same shapes are written in C++ above the C ABI and driven
// from the tests through n1gpu_plan_build / n1gpu_operator_run_once.
//
//   plan/plan.go:25-34 (plan.Operator)            plan/visitor.go:12-123 (plan.Visitor)
//   plan/op_registry.go:18-29 (MakeOperator)      plan/{scan_primary,fetch,filter,group,parallel,sequence}.go
//   execution/execution.go:26-64 (Operator)       execution/build.go:22-45,455-491 (Build, VisitParallel/Sequence)
//   execution/base.go:896-949 (marshalTimes)      algebra/aggregate.go:97-118 ("aggregates" attachment)
#pragma once
#include <memory>
#include <string>
#include <vector>

#include "group_tail.hpp"
#include "json.hpp"
#include "query.hpp"

namespace n1 {
namespace plan {

struct Visitor;

struct Operator {  // plan/plan.go:25-34
    virtual ~Operator() {}
    virtual const char* Name() const = 0;
    virtual void Accept(Visitor& v) = 0;
    virtual bool Readonly() const { return true; }
    virtual std::string MarshalJSON() const = 0;
};
typedef std::unique_ptr<Operator> OperatorP;

struct KeyspaceTerm { std::string nspace, keyspace, as; std::string Alias() const { return as.empty() ? keyspace : as; } };

struct PrimaryScan : Operator {  // plan/scan_primary.go
    KeyspaceTerm term; std::string index, using_, limit;
    const char* Name() const override { return "PrimaryScan"; }
    void Accept(Visitor& v) override;
    std::string MarshalJSON() const override;
};
struct Fetch : Operator {  // plan/fetch.go
    KeyspaceTerm term;
    const char* Name() const override { return "Fetch"; }
    void Accept(Visitor& v) override;
    std::string MarshalJSON() const override;
};
struct Filter : Operator {  // plan/filter.go
    std::string condition;
    const char* Name() const override { return "Filter"; }
    void Accept(Visitor& v) override;
    std::string MarshalJSON() const override;
};
struct Group : Operator {  // plan/group.go: InitialGroup / IntermediateGroup / FinalGroup
    int phase = 0;  // 0 initial, 1 intermediate, 2 final
    std::vector<std::string> keys, aggregates;
    const char* Name() const override { return phase == 0 ? "InitialGroup" : (phase == 1 ? "IntermediateGroup" : "FinalGroup"); }
    void Accept(Visitor& v) override;
    std::string MarshalJSON() const override;
};
struct Parallel : Operator {  // plan/parallel.go
    OperatorP child; int maxParallelism = 0;
    const char* Name() const override { return "Parallel"; }
    void Accept(Visitor& v) override;
    std::string MarshalJSON() const override;
};
struct Sequence : Operator {  // plan/sequence.go
    std::vector<OperatorP> children;
    const char* Name() const override { return "Sequence"; }
    void Accept(Visitor& v) override;
    std::string MarshalJSON() const override;
};
struct Authorize : Operator {  // plan/authorize.go
    OperatorP child; std::string privileges_json;
    const char* Name() const override { return "Authorize"; }
    void Accept(Visitor& v) override;
    std::string MarshalJSON() const override;
};
struct Opaque : Operator {  // every operator outside the chain: kept verbatim, run by the caller
    std::string name, body;
    const char* Name() const override { return name.c_str(); }
    void Accept(Visitor& v) override;
    std::string MarshalJSON() const override { return body; }
};

struct Visitor {  // plan/visitor.go:12-123 (the operators of this path; everything else is VisitOpaque)
    virtual ~Visitor() {}
    virtual void VisitPrimaryScan(PrimaryScan&) = 0;
    virtual void VisitFetch(Fetch&) = 0;
    virtual void VisitFilter(Filter&) = 0;
    virtual void VisitInitialGroup(Group&) = 0;
    virtual void VisitIntermediateGroup(Group&) = 0;
    virtual void VisitFinalGroup(Group&) = 0;
    virtual void VisitParallel(Parallel&) = 0;
    virtual void VisitSequence(Sequence&) = 0;
    virtual void VisitAuthorize(Authorize&) = 0;
    virtual void VisitOpaque(Opaque&) = 0;
};

OperatorP MakeOperator(const json::Node& n);  // plan/op_registry.go:18-29
std::string node_to_json(const json::Node& n);

}  // namespace plan

namespace execution {

// The replacement for [PrimaryScan, Fetch, Parallel(Sequence[Filter?, InitialGroup]), IntermediateGroup,
// FinalGroup].  A producer operator: RunOnce scans the keyspace, filters and groups on the GPU and yields
// what FinalGroup would have sent (execution/group_final.go:100-118).
class GpuGroupAggregate {
  public:
    plan::KeyspaceTerm term;
    std::string keyspace_dir;
    std::string condition;
    std::vector<std::string> keys, aggregates;
    std::shared_ptr<Table> table;
    std::unique_ptr<Query> query;
    i64 in_docs = 0, out_docs = 0;
    i64 docs_read = 0;  // documents read to build the table: all for a load, the changed ones for a refresh, 0 when reused
    double exec_sec = 0, serv_sec = 0;
    bool ran = false;
    // The operators after FinalGroup that this operator also replaces when all of them are within the subset
    // (SURVEY.md 8f rows 1-2): Let / Filter (LETTING, HAVING), InitialProject, FinalProject, Order, Offset, Limit.
    GroupTail tail;

    std::unique_ptr<Result> RunOnce();  // execution.Operator.RunOnce (once per operator: util.Once)
    void SendStop();                    // execution.Operator.SendStop
    std::string MarshalJSON() const;    // plan node + "#stats" (execution/base.go:896-949)
};

// execution.Build (execution/build.go:22-45) restricted to the substitution: finds the eligible Sequence
// in the plan, builds the GPU operator for its prefix; *rest_index = first child of that Sequence the
// caller still runs.  Throws Error(N1GPU_E_INELIGIBLE) when the plan does not contain the chain.
std::unique_ptr<GpuGroupAggregate> Build(const std::string& plan_json, const std::string& datastore_root, int* rest_index);
// The same, also taking over the operators after FinalGroup (op->tail) when the whole run up to FinalProject is eligible.
// rest_index then points behind the consumed operators of the chain's Sequence and *outer_rest behind those consumed
// from the enclosing Sequence (0: none).  want_tail = false builds exactly what Build does.
std::unique_ptr<GpuGroupAggregate> BuildWithTail(const std::string& plan_json, const std::string& datastore_root, bool want_tail,
                                                 int* rest_index, int* outer_rest);

std::string ResultToJSON(const Result& r);
// Directory for the operator's persistent segments ("" = none); also read from N1GPU_SEGMENT_DIR.
void set_segment_dir(const std::string& dir);

}  // namespace execution
}  // namespace n1
