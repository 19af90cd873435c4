// Explicit instantiation of engine A for mlp_units=64, n_invariant_feat_hidden=32, exact divergence off, saving the path (SaveAt(ts)).
#include "ecnf_solve_impl.cuh"
namespace ecnf_solve_detail {
template int launch_t<64, 32, false, true>(const ecnf_model*, KernelArgs&, int, cudaStream_t);
}
