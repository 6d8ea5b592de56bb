/* ORACLE / TEST INFRASTRUCTURE ONLY. The port_ instantiation of ../chan_q15.inc.c: every stage it calls (fir_q15, cfft_q15, cmplx_mag_q15,
 * abs_q15, max_q15, scale_q15) is restated elsewhere in this directory and pinned bit-exact (cfft_q15: to the Cortex-M4 branch). */
#include "port_common.h"
#include "../slo_chan_q15.h"

#include "../chan_q15.inc.c"
