// code8check.cpp - the factor-code -> FP8 operand mapping of csrc/numerics.cuh (fp8_operand_format, code_to_fp8)
// compiled for the HOST, for the CPU part of tests/test_code_gemm.py.
// TEST INFRASTRUCTURE: never linked into libadmmq.so.
// Build: g++ -O2 -ffp-contract=off -shared -fPIC (tests/test_code_gemm.py does it).
#include "../../admm-quantization_b200/csrc/numerics.cuh"

using namespace admmq;

extern "C" {
int hc_fp8_operand_format(int scheme, int bits) { return fp8_operand_format(scheme, bits); }
int hc_code_to_fp8(int scheme, int code) { return (int)code_to_fp8(scheme, code); }
}
