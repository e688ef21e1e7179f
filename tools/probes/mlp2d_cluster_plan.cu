// Probe: the shared-memory plan of the 2-D cluster kernels (csrc/mlp2d_cluster.cu) for one (nhidden, nlayers), and
// how many of their clusters the current device holds at once -- the answer of the same cudaOccupancyMaxActiveClusters
// query the library asks before its first launch.  tools/profile_2d.py builds and runs it.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -I collaborative-gan-sampling_b200/csrc -I include \
//             -o /tmp/mlp2d_cluster_plan tools/probes/mlp2d_cluster_plan.cu
// Run:   /tmp/mlp2d_cluster_plan <nhidden> <nlayers>
#include <cstdio>
#include <cstdlib>

#include "mlp2d_cluster.cu"

namespace cgs {   // the few library helpers the included file calls (api.cu)
char* error_buffer() {
  static char b[512];
  return b;
}
int current_device() {
  int d = -1;
  return cudaGetDevice(&d) == cudaSuccess ? d : -1;
}
void count_launch(int) {}
}  // namespace cgs

int main(int argc, char** argv) {
  if (argc != 3) {
    fprintf(stderr, "usage: %s nhidden nlayers\n", argv[0]);
    return 2;
  }
  cgs_mlp_desc d = {};
  d.nhidden = atoi(argv[1]);
  d.nlayers = atoi(argv[2]);
  cgs::ClusterLaunch L;
  // a batch large enough that every resident cluster gets points: L.clusters is then the resident count
  if (cgs::plan_launch(cgs::mlp2d_cluster_refine_kernel, d, (int64_t)1 << 40, L)) {
    printf("error: %s\n", cgs::error_buffer());
    return 1;
  }
  printf("cluster_ctas %d points_per_round %d smem_bytes %zu resident_clusters %d\n", L.C, L.P, L.smem, L.clusters);
  return 0;
}
