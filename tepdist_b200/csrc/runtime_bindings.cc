#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include "runtime/data_loader.h"
#include "runtime/dev_mesh.h"
#include "runtime/slice_philox.h"
#include "runtime/task_graph.h"
#include "service_env.h"

namespace py = pybind11;
using namespace tepdist;

void BindRuntime(py::module_& m) {
  // ---- native input pipeline (runtime/data_loader.h)
  py::class_<TokenSource, std::shared_ptr<TokenSource>>(m, "TokenSource")
      .def(py::init<>())
      .def("add_dataset", &TokenSource::AddDataset, py::arg("files"), py::arg("weight") = 1.0, py::arg("bytes_per_token") = 2)
      .def("set_synthetic", &TokenSource::SetSynthetic, py::arg("vocab"))
      .def("total_tokens", &TokenSource::total_tokens)
      .def("num_datasets", &TokenSource::num_datasets)
      .def("sample", [](const TokenSource& s, uint64_t seed, uint64_t sample_id, int n) {
        std::vector<int32_t> v((size_t)n);
        s.Sample(seed, sample_id, n, v.data());
        return v;
      })
      .def("locate", [](const TokenSource& s, uint64_t seed, uint64_t sample_id, int n) {
        int d, f;
        uint64_t off;
        s.Locate(seed, sample_id, n, &d, &f, &off);
        return py::make_tuple(d, f, off);
      });
  py::class_<BatchLoader>(m, "BatchLoader")
      .def(py::init<std::shared_ptr<TokenSource>, int, int, int, int, uint64_t, int>(), py::arg("source"), py::arg("batch"), py::arg("n_ctx"),
           py::arg("rank") = 0, py::arg("world") = 1, py::arg("seed") = 0, py::arg("threads") = 2)
      .def("set_buffers", &BatchLoader::SetBuffers, py::arg("tokens"), py::arg("labels"),
           py::arg("segments") = std::vector<uintptr_t>{}, py::arg("eot") = 0)
      .def("start", &BatchLoader::Start, py::arg("first_step") = 0)
      .def("acquire", [](BatchLoader& l) {
        uint64_t step = 0;
        int slot;
        {
          py::gil_scoped_release nogil;      // blocks until a worker thread has finished the batch
          slot = l.Acquire(&step);
        }
        return py::make_tuple(slot, step);
      })
      .def("release", &BatchLoader::Release)
      .def("stop", &BatchLoader::Stop, py::call_guard<py::gil_scoped_release>())
      .def("num_slots", &BatchLoader::num_slots)
      .def("batches_filled", &BatchLoader::batches_filled);

  // ---- device mesh
  py::class_<DevGroup>(m, "DevGroup").def_readonly("ordinal", &DevGroup::ordinal).def_readonly("devices", &DevGroup::devices);
  py::class_<CommDevManager>(m, "CommDevManager")
      .def(py::init<>())
      .def("build", &CommDevManager::Build, py::arg("split_nums"), py::arg("share_dev"), py::arg("placement_layout") = std::vector<int>(),
           py::arg("num_workers") = 1, py::arg("devs_per_worker") = 0)
      .def("total_devices", &CommDevManager::total_devices)
      .def("global_device", [](const CommDevManager& c, const std::vector<int>& ids) { return c.GlobalDevice(SplitId{ids}); })
      .def("worker_of", &CommDevManager::WorkerOf).def("local_device", &CommDevManager::LocalDevice)
      .def("coords", &CommDevManager::Coords).def("group_of", &CommDevManager::GroupOf)
      .def("rank_in_group", &CommDevManager::RankInGroup).def("all_groups", &CommDevManager::AllGroups)
      .def("group_spans_workers", &CommDevManager::GroupSpansWorkers).def("describe", &CommDevManager::Describe);

  // ---- task graph / scheduler
  py::enum_<TaskType>(m, "TaskType")
      .value("Split", TaskType::kSplit).value("Input", TaskType::kInput).value("Compute", TaskType::kCompute)
      .value("Output", TaskType::kOutput).value("Send", TaskType::kSend).value("Recv", TaskType::kRecv)
      .value("GAInit", TaskType::kGAInit).value("GA", TaskType::kGA).value("AG", TaskType::kAG).value("Merge", TaskType::kMerge);
  py::class_<TaskNode>(m, "TaskNode")
      .def_readonly("id", &TaskNode::id).def_readonly("type", &TaskNode::type).def_readonly("name", &TaskNode::name)
      .def_readonly("stage", &TaskNode::stage).def_readonly("micro", &TaskNode::micro).def_readonly("backward", &TaskNode::backward)
      .def_readonly("device", &TaskNode::device).def_readonly("peer_device", &TaskNode::peer_device)
      .def_readonly("cost", &TaskNode::cost).def_readonly("out_bytes", &TaskNode::out_bytes)
      .def_readonly("parents", &TaskNode::parents).def_readonly("children", &TaskNode::children)
      .def_readonly("mem_to_release", &TaskNode::mem_to_release).def_readonly("buffer_id", &TaskNode::buffer_id)
      .def_readonly("buffer_reused", &TaskNode::buffer_reused).def_readonly("def_ctx", &TaskNode::def_ctx);
  py::class_<TaskDAG>(m, "TaskDAG")
      .def(py::init<>())
      .def_readonly("nodes", &TaskDAG::nodes).def_readonly("source", &TaskDAG::source).def_readonly("sink", &TaskDAG::sink)
      .def("add_node", &TaskDAG::AddNode).def("add_edge", &TaskDAG::AddEdge)
      .def("topo_order", &TaskDAG::TopoOrder).def("dominance_tree", &TaskDAG::BuildDominanceTree).def("to_dot", &TaskDAG::ToDot);
  py::class_<PipelineSpec>(m, "PipelineSpec")
      .def(py::init<>())
      .def_readwrite("num_stages", &PipelineSpec::num_stages).def_readwrite("num_micro", &PipelineSpec::num_micro)
      .def_readwrite("spmd", &PipelineSpec::spmd).def_readwrite("fwd_seconds", &PipelineSpec::fwd_seconds)
      .def_readwrite("bwd_seconds", &PipelineSpec::bwd_seconds).def_readwrite("ag_seconds", &PipelineSpec::ag_seconds)
      .def_readwrite("act_bytes", &PipelineSpec::act_bytes).def_readwrite("boundary_bytes", &PipelineSpec::boundary_bytes)
      .def_readwrite("p2p_bw", &PipelineSpec::p2p_bw).def_readwrite("p2p_latency", &PipelineSpec::p2p_latency)
      .def_readwrite("mem_limit", &PipelineSpec::mem_limit);
  m.def("build_pipeline_task_dag", &BuildPipelineTaskDAG);
  py::class_<ScheduleOptions>(m, "ScheduleOptions")
      .def(py::init<>())
      .def_readwrite("micro_num_limit", &ScheduleOptions::micro_num_limit).def_readwrite("early_ga", &ScheduleOptions::early_ga)
      .def_readwrite("reorder_send", &ScheduleOptions::reorder_send).def_readwrite("buffer_save", &ScheduleOptions::buffer_save)
      .def_readwrite("group_sched_count", &ScheduleOptions::group_sched_count)
      .def_readwrite("recv_ring", &ScheduleOptions::recv_ring);
  py::class_<Schedule>(m, "Schedule")
      .def_readonly("device_tasks", &Schedule::device_tasks).def_readonly("start", &Schedule::start)
      .def_readonly("finish", &Schedule::finish).def_readonly("makespan", &Schedule::makespan)
      .def_readonly("peak_bytes", &Schedule::peak_bytes).def_readonly("oom", &Schedule::oom)
      .def_readonly("bubble_ratio", &Schedule::bubble_ratio).def("dump", &Schedule::Dump);
  m.def("schedule_tasks", [](TaskDAG& d, const PipelineSpec& s, const ScheduleOptions& o) { return ScheduleTasks(&d, s, o); });
  m.def("compute_release_plan", &ComputeReleasePlan);

  // ---- slicing + philox
  m.def("slice_runs", &SliceRuns);
  m.def("shard_shape", &ShardShape);
  m.def("slice_copy", [](py::array_t<float, py::array::c_style | py::array::forcecast> src, const std::vector<int64_t>& shape,
                         const std::vector<DimStrategy>& levels, const std::vector<int>& ids) {
    auto ss = ShardShape(shape, levels);
    int64_t n = 1;
    for (auto d : ss) n *= d;
    py::array_t<float> out(n);
    SliceCopy(reinterpret_cast<const uint8_t*>(src.data()), reinterpret_cast<uint8_t*>(out.mutable_data()), 4, shape, levels, ids);
    out.resize(ss);
    return out;
  });
  m.def("philox_fill", [](const std::string& kind, uint64_t seed, int64_t offset, int64_t n, float mean, float stddev, float lo, float hi) {
    py::array_t<float> out(n);
    PhiloxFill(kind, seed, offset, n, mean, stddev, lo, hi, out.mutable_data());
    return out;
  });
  m.def("philox_fill_shard", [](const std::string& kind, uint64_t seed, const std::vector<int64_t>& shape,
                                const std::vector<DimStrategy>& levels, const std::vector<int>& ids, float mean, float stddev, float lo, float hi) {
    auto v = PhiloxFillShard(kind, seed, shape, levels, ids, mean, stddev, lo, hi);
    py::array_t<float> out(v.size());
    std::copy(v.begin(), v.end(), out.mutable_data());
    out.resize(ShardShape(shape, levels));
    return out;
  });

  // ---- ServiceEnv
  py::class_<ServiceEnv>(m, "ServiceEnv")
      .def_static("instance", &ServiceEnv::Instance, py::return_value_policy::reference)
      .def("load", &ServiceEnv::Load, py::arg("config_file") = "")
      .def("get", &ServiceEnv::Get).def("get_int", &ServiceEnv::GetInt).def("get_double", &ServiceEnv::GetDouble)
      .def("get_bool", &ServiceEnv::GetBool).def("set", &ServiceEnv::Set).def("dump", &ServiceEnv::Dump)
      .def("keys", &ServiceEnv::Keys);
}
