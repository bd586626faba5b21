/*
 * TEST INFRASTRUCTURE — NOT PART OF THE PRODUCT.  The oracle's SCF of an electron configuration (dftatom_oracle_config.c).
 */
#ifndef DFTATOM_ORACLE_CONFIG_H
#define DFTATOM_ORACLE_CONFIG_H

#include "dftatom_oracle.h"

#ifdef __cplusplus
extern "C" {
#endif

/* The SCF of an electron configuration (methods 0-3): entries (n 1-based, l, spin 0 / 1, occ a double), each spin solved in (n, l) order
 * (the records' orc_level.occ is the occupation rounded).  The start density is a uniform sphere of the configuration's electrons per
 * spin and the Hartree boundary value is their count Q; the nucleus keeps Z.  With the Aufbau configuration it is orc_scf_ex (methods
 * 0 / 1) or orc_scf_uniform (2 / 3) bit for bit.  V_out / rho_out as orc_scf_ex (may be NULL).  Returns -1 for a malformed configuration
 * (the full validation is the library's). */
typedef struct { int n, l, spin; double occ; } orc_orbital;
typedef struct { int n_orbitals; orc_orbital orb[2 * ORC_MAX_LEVELS]; } orc_config;
int orc_scf_config(const orc_options* opt, const orc_config* cfg, orc_result* res, orc_step_cb cb, void* user, int max_vcycles,
                   double* V_out, double* rho_out);

#ifdef __cplusplus
}
#endif
#endif
