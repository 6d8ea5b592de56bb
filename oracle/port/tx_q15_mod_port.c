/* ORACLE / TEST INFRASTRUCTURE ONLY. The port_ instantiation of ../tx_q15_mod.inc.c: every stage it calls (fir_q15, abs_q15, max_q15,
 * scale_q15, add_q15, and tx_fm_nco with its q31_to_float, scale_f32, cos_f32, sin_f32, float_to_q15) is restated elsewhere in this
 * directory and pinned bit-exact to the reference. */
#include "port_common.h"
#include "../slo_tx_q15_mod.h"

#include "../tx_q15_mod.inc.c"
