// perm_bound_on_host.cpp -- TEST HARNESS, not part of the product.
//
// Compiles dm_perm_inv_lo and det_pow of samsim_b200/csrc/detmath.h for the host (g++ -ffp-contract=off, the same
// arithmetic the GPU build gets from -fmad=false), so that tests/test_perm_bound_cpu.py can check the bound against
// the permeability fl_grav_drain computes.
#include <stdint.h>

#include "../../samsim_b200/csrc/detmath.h"

extern "C" {

// perm[q] = 1e-17 * det_pow(1000|psi_l|, 3.10) as grav_drain evaluates it, inv[q] = dm_perm_inv_lo(psi_l)
void pb_eval(int64_t n, const double* psi_l, double* perm, double* inv) {
  for (int64_t q = 0; q < n; q++) {
    perm[q] = 1e-17 * det_pow(1000.0 * fabs(psi_l[q]), 3.10);
    inv[q] = dm_perm_inv_lo(psi_l[q]);
  }
}

double pb_slack(void) { return DM_PERM_SLACK; }

}
