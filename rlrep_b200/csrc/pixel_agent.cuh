// What the pixel agents (DrQ-v2, muLV-Rep DrQ-v2, latent Diff-SR DrQ-v2) share around their update: the stream, the
// pinned staging and metrics buffers, the timing and profiling aids, target sync, and the end of update() (see
// pixel_agent.cu).  Each agent keeps its own config, inputs and launch sequence.
#pragma once
#include <memory>
#include <string>
#include <vector>

#include "agent.cuh"
#include "conv.cuh"
#include "pixel_act.cuh"

namespace rlrep {

class PixelAgent {
 public:
  explicit PixelAgent(cudaStream_t s) : stream_(s) {}
  virtual ~PixelAgent();
  PixelAgent(const PixelAgent&) = delete;
  PixelAgent& operator=(const PixelAgent&) = delete;

  // The optimiser groups, in the order their tensors are exported.
  virtual std::vector<ParamGroup*> groups() = 0;
  // Reference state_dict name of tensor `t` of group `g`.  The conv stacks name their tensors relative to their module
  // ("convnet.0.weight"); the agent places them.  A group's target copy is exported under this name with the group's
  // target_prefix_from replaced by target_prefix_to.
  virtual std::string tensor_name(const ParamGroup& g, const std::string& t) const { return t; }

  // Benchmark aids on the batch uploaded by the last update(): n_steps updates back to back, CUDA-event time of the loop
  // in milliseconds; one update with an event behind every launch.
  float update_resident(int n_steps, float stddev);
  std::vector<ProfileEntry> profile_update(float stddev);
  // target <- params of every group that has a Polyak target (after loading weights)
  void sync_targets_from_params();
  cudaStream_t stream() const { return stream_; }
  // The Adam step counters (t_feat, t_critic, t_actor) are the optimiser state that is not a tensor: the tick at the head
  // of every update derives that update's bias corrections from them, so writing them is all a resume needs.
  Control* control() const { return ctl_; }
  int last_launches = 0;

 protected:
  static constexpr int kMetrics = 8;  // floats of metrics_dev_
  // Every launch of one update on the batch currently resident in the device buffers.
  virtual void launch_update(float stddev) = 0;
  // Pinned host memory: stage_bytes for update()'s inputs (stage_h2d) and the metrics block.
  void alloc_host(size_t stage_bytes);
  // The end of update(), once its inputs are staged: launch_update (its launches counted into last_launches), then the
  // first n_metrics floats of metrics_dev_ -> metrics_out.
  void finish_update(float stddev, float* metrics_out, int n_metrics);

  cudaStream_t stream_;
  Control* ctl_ = nullptr;        // in the agent's arena
  float* metrics_dev_ = nullptr;  // [kMetrics], in the agent's arena
  unsigned char* stage_host_ = nullptr;
  float* metrics_host_ = nullptr;
};

// The small-batch policy's view of a DrQ-v2 actor: the encoder's four conv layers, then actor.trunk.0 (`trunk`),
// actor.trunk.1 (LayerNorm at ln_w / ln_b) and actor.policy.0 / .2 / .4 (`p0`, `p1`, `p2`), all in the group `actor`.
PixelPolicyWeights actor_policy_weights(const ConvEncoder& enc, const ParamGroup& actor, const LinearSlot& trunk,
                                        size_t ln_w, size_t ln_b, const LinearSlot& p0, const LinearSlot& p1,
                                        const LinearSlot& p2);

}  // namespace rlrep
