/* ORACLE / TEST INFRASTRUCTURE ONLY. The port_ instantiation of ../rx_q15.inc.c: every stage it calls (fir_q15, cmplx_mag_q15, add_q15,
 * sub_q15, abs_q15, max_q15, scale_q15) is restated elsewhere in this directory and pinned bit-exact to the reference. */
#include "port_common.h"
#include "../slo_rx_q15.h"

#include "../rx_q15.inc.c"
