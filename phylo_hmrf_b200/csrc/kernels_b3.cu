// Phase B, bulk-copy pipeline: dispatch (the kernel lives in estep_bulk.cuh) and the instantiations
// for 1..4 features.
#define PHMRF_B3_ENTRY launch_estep_bulk_d14
#define PHMRF_B3_D0 1
#include "estep_bulk.cuh"

namespace phmrf {

int launch_estep_bulk_d58(const EstepArgs &a, int sm_count, cudaStream_t s);
int launch_estep_bulk_d9c(const EstepArgs &a, int sm_count, cudaStream_t s);

bool estep_bulk_supported(const EstepArgs &a) {
    const int nk8 = (a.K + 7) / 8;
    return a.n > 0 && a.pp_soa == nullptr && a.potts && a.W >= 1 && a.W <= estep::kFastSlots &&
           fabs(a.s_bound) < 100.0 &&  // exp(S) * exp(600) must stay finite without range checks
           a.K <= 40 && bulk_acc_fits(a.D, nk8) && bulk_smem_fits(a.D, nk8);
}

int launch_estep_bulk(const EstepArgs &a, int sm_count, cudaStream_t s) {
    if (a.D >= 1 && a.D <= 4) return launch_estep_bulk_d14(a, sm_count, s);
    if (a.D >= 5 && a.D <= 8) return launch_estep_bulk_d58(a, sm_count, s);
    if (a.D >= 9 && a.D <= 12) return launch_estep_bulk_d9c(a, sm_count, s);
    return bulk_unsupported(a);
}

}  // namespace phmrf
