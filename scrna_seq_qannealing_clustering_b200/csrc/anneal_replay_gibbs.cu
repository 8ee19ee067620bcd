// anneal_replay_gibbs.cu -- the Gibbs-acceptance instances of k_anneal_replay (replay.cuh), in a translation unit of their own
// so that anneal_replay.cu's module holds exactly the Metropolis instances and the two compile in parallel.
#include "device_common.cuh"

using namespace qa;

namespace {

#include "replay.cuh"

}  // namespace

namespace qa {

const void *replay_gibbs_kernel(const qa_model *M, GroupKind gk) { return replay_instance<PROP_GIBBS>(M, gk); }

}  // namespace qa
