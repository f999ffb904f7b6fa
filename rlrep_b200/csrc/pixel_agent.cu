// Shared host side of the pixel agents (pixel_agent.cuh).
#include <cstring>

#include "pixel_agent.cuh"

namespace rlrep {

PixelAgent::~PixelAgent() {
  if (stage_host_) cudaFreeHost(stage_host_);
  if (metrics_host_) cudaFreeHost(metrics_host_);
}

void PixelAgent::alloc_host(size_t stage_bytes) {
  RLREP_CUDA(cudaMallocHost(&stage_host_, stage_bytes));
  RLREP_CUDA(cudaMallocHost(&metrics_host_, kMetrics * sizeof(float)));
}

void PixelAgent::finish_update(float stddev, float* metrics_out, int n_metrics) {
  const long long before = launch_count();
  launch_update(stddev);
  last_launches = (int)(launch_count() - before);
  RLREP_CUDA(cudaMemcpyAsync(metrics_host_, metrics_dev_, kMetrics * sizeof(float), cudaMemcpyDeviceToHost, stream_));
  RLREP_CUDA(cudaStreamSynchronize(stream_));
  std::memcpy(metrics_out, metrics_host_, n_metrics * sizeof(float));
}

float PixelAgent::update_resident(int n_steps, float stddev) {
  RLREP_CHECK(n_steps > 0, "bad step count");
  cudaEvent_t e0, e1;
  RLREP_CUDA(cudaEventCreate(&e0));
  RLREP_CUDA(cudaEventCreate(&e1));
  RLREP_CUDA(cudaStreamSynchronize(stream_));
  RLREP_CUDA(cudaEventRecord(e0, stream_));
  for (int i = 0; i < n_steps; ++i) launch_update(stddev);
  RLREP_CUDA(cudaEventRecord(e1, stream_));
  RLREP_CUDA(cudaEventSynchronize(e1));
  float ms = 0.f;
  RLREP_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  return ms;
}

std::vector<ProfileEntry> PixelAgent::profile_update(float stddev) {
  RLREP_CUDA(cudaStreamSynchronize(stream_));
  profile_begin(stream_);
  launch_update(stddev);
  return profile_end(stream_);
}

void PixelAgent::sync_targets_from_params() {
  for (ParamGroup* g : groups())
    if (g->n_target) RLREP_CUDA(cudaMemcpyAsync(g->target, g->p, g->n_target * 4, cudaMemcpyDeviceToDevice, stream_));
  RLREP_CUDA(cudaStreamSynchronize(stream_));
}

PixelPolicyWeights actor_policy_weights(const ConvEncoder& enc, const ParamGroup& actor, const LinearSlot& trunk,
                                        size_t ln_w, size_t ln_b, const LinearSlot& p0, const LinearSlot& p1,
                                        const LinearSlot& p2) {
  PixelPolicyWeights w;
  for (int l = 0; l < 4; ++l) w.conv[l] = enc.layer(l);
  w.trunk = trunk.view(actor);
  w.ln_w = actor.p + ln_w;
  w.ln_b = actor.p + ln_b;
  w.policy[0] = p0.view(actor);
  w.policy[1] = p1.view(actor);
  w.policy[2] = p2.view(actor);
  return w;
}

}  // namespace rlrep
