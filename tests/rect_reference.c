/* TEST INFRASTRUCTURE ONLY -- CPU reference for stage 1 of a tall m x n matrix (m >= n) in the panel order.
 * It is the text of svdo_brd_p1_panel (the oracle's restatement of csc586::gpu::brd_p1, svd_cpu.h:370-425) with the
 * trailing rows of step k running to m instead of n; the storage stays row-major with ld = n.  It is compiled together
 * with the oracle's primitives (qr, lq, form_q, ...); only the loop order of the Q application differs, not its sums, so
 * at m == n it is the oracle's panel reduction to the bit (tests/test_rect_cpu.py checks that). */
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <stddef.h>
#include "svd_oracle.h"

#define T float
#define FN(name) name##_f32
#define SQRT_T sqrtf
#define FABS_T fabsf
#include "svd_oracle_impl.h"
#include "rect_reference_impl.h"
#undef T
#undef FN
#undef SQRT_T
#undef FABS_T

#define T double
#define FN(name) name##_f64
#define SQRT_T sqrt
#define FABS_T fabs
#include "svd_oracle_impl.h"
#include "rect_reference_impl.h"
#undef T
#undef FN
#undef SQRT_T
#undef FABS_T
