// float32 (tolerance) mode of every entry point.  FMA contraction allowed.
#define EMEI_REAL float
#define EMEI_FN(name) name##_f32
#include "impl.inc"
