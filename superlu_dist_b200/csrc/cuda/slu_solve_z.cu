// slu_solve_z.cu -- the doublecomplex build of the resident-factor solve and the device-side distribution (namespace sluz)
#define SLU_COMPLEX 1
#include "slu_solve.cu"
