// g++ harness of tests/test_mg_slabs_host.py: the plane reach of the class tables (csrc/mg_transfer.h: plane_reach) that
// mg_transfer_init uses to check the coarse halo and to build the restriction's transfer halo of a z-slab.
#include "mg_transfer.h"

extern "C" void mg_reach(int kind, int prolong, int64_t a, int64_t b, int64_t L_to, int64_t* lo, int64_t* hi) {
    const poromg::Table T = prolong ? poromg::prolong_table(kind, 3) : poromg::restrict_table(kind, 3);
    poromg::plane_reach(T, 3, prolong != 0, kind, a, b, L_to, *lo, *hi);
}
