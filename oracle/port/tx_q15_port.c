/* ORACLE / TEST INFRASTRUCTURE ONLY. The port_ instantiation of ../tx_q15.inc.c: every stage it calls (fir_q15, abs_q15, max_q15,
 * scale_q15) is restated elsewhere in this directory and pinned bit-exact to the reference. */
#include "port_common.h"
#include "../slo_tx_q15.h"

#include "../tx_q15.inc.c"
