/* ORACLE / TEST INFRASTRUCTURE ONLY. The port_ instantiation of ../tune.inc.c: every stage it calls is restated elsewhere in this
 * directory (q31_to_float in tx_mod_port.c). */
#include "port_common.h"
#include "../slo_tune.h"

#include "../tune.inc.c"
