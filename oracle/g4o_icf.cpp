// Integer-coded float elements (GvrsElementSpecificationIntCodedFloat / GvrsElementIntCodedFloat).
// The reference source is not in this tree.  These two functions restate the mapping as the ICF feature request gives it;
// no reference fixture pins it beyond exactly representable values (the reference's sample files hold integer values
// only).  Built with -ffp-contract=off: the float32 subtraction and multiplication must not be fused.
#include <cmath>
#include <cstdint>

namespace {

// Java's (int) cast of a double: NaN -> 0, saturating at the int range, truncating toward zero otherwise.
int32_t java_d2i(double d) {
  if (d != d) return 0;
  if (d >= 2147483647.0) return INT32_MAX;
  if (d <= -2147483648.0) return INT32_MIN;
  return int32_t(d);
}

}  // namespace

extern "C" {

// float -> code: NaN -> fillInt; else (int) Math.floor((double)((v - offset) * scale) + 0.5), the subtraction and the
// multiplication in float32, + 0.5 and floor in double.
void g4o_icf_to_int(const float* v, long n, float scale, float offset, int32_t fillInt, int32_t* out) {
  for (long i = 0; i < n; i++) {
    if (std::isnan(v[i])) {
      out[i] = fillInt;
      continue;
    }
    const float t = (v[i] - offset) * scale;
    out[i] = java_d2i(std::floor(double(t) + 0.5));
  }
}

// code -> float: fillInt -> fillValue; else (float) code / scale + offset in float32.
void g4o_icf_to_float(const int32_t* k, long n, float scale, float offset, int32_t fillInt, float fillValue, float* out) {
  for (long i = 0; i < n; i++) {
    if (k[i] == fillInt) {
      out[i] = fillValue;
      continue;
    }
    const float q = float(k[i]) / scale;
    out[i] = q + offset;
  }
}

}  // extern "C"
