// CUDA-graph capture, replay and the n-update graph cache, shared by the agents and the prioritised-replay draw.
//
// Launch accounting (gcrl_kernel_launches): the kernels a capture records are not executed by it, so they leave the
// launch counter when the capture ends and come back with every replay.
#pragma once
#include <functional>
#include <map>
#include <set>
#include <utility>

#include "common.cuh"

namespace gcrl {

struct GraphRec {
  cudaGraphExec_t exec;
  uint64_t kernels;   // launches recorded into the graph
};

// false when GCRL_B200_NO_GRAPH=1: every update is issued eagerly.  Read when a handle is created and kept per handle.
bool graphs_enabled();

void begin_capture(cudaStream_t cap);
// End the capture on `cap` and instantiate it; `kernels` launches were recorded since it began (or since the last cut).
GraphRec end_capture(cudaStream_t cap, uint64_t kernels);
// End a capture that failed part-way, if it is still open, and drop what it recorded.
void abort_capture(cudaStream_t cap);

// Record `body` on the capture stream `cap` into an instantiated graph.
GraphRec capture_graph(cudaStream_t cap, const std::function<void(cudaStream_t)> &body);
void launch_graph(const GraphRec &g, cudaStream_t st);

// The n-update graphs of one agent (gcrl_agent_update_many*, gcrl_sac_update_many*).
template <typename Key>
struct ManyGraphs {
  static constexpr size_t kCap = 8;   // graphs kept per agent (one flag pattern per run is typical)
  std::map<Key, GraphRec> graphs;
  std::set<Key> seen;                 // keys issued eagerly once (capture_new false: captured when one repeats)

  // Replay the graph of `key`, capturing it on `cap` first when it is new -- or, with capture_new false, only when
  // the key was issued before (a key seen for the first time is issued eagerly: a prioritised buffer that is still
  // filling draws from a new length every call, and its graphs would never be replayed).  Without graphs, eager.
  void launch(Key key, bool capture_new, const std::function<void(cudaStream_t)> &body, cudaStream_t st,
              bool use_graphs, cudaStream_t cap) {
    if (!use_graphs) {
      body(st);
      return;
    }
    auto it = graphs.find(key);
    if (it == graphs.end() && !capture_new && seen.count(key) == 0) {
      if (seen.size() >= 2 * kCap) seen.clear();
      seen.insert(std::move(key));
      body(st);
      return;
    }
    if (it == graphs.end()) {
      const GraphRec g = capture_graph(cap, body);
      if (graphs.size() >= kCap) clear();     // a replay still in flight is released when it completes
      it = graphs.emplace(std::move(key), g).first;
    }
    launch_graph(it->second, st);
  }

  // drop every graph (the `seen` keys stay)
  void clear() {
    for (auto &kv : graphs) cudaGraphExecDestroy(kv.second.exec);
    graphs.clear();
  }
};

}  // namespace gcrl
