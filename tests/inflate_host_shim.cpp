// Host build of the device BGZF block decoder (alntools_b200/csrc/ecb_inflate.cuh) for
// tests/test_device_inflate_host.py: the same source, compiled by g++ with sanitizers and loaded with ctypes.
#include "../alntools_b200/csrc/ecb_inflate.cuh"

extern "C" int shim_inflate(const uint8_t* src, int64_t src_len, uint8_t* dst, int64_t dst_len) {
  ecbinf::Tables t;
  return ecbinf::inflate_block(src, (uint32_t)src_len, dst, (uint32_t)dst_len, t) ? 1 : 0;
}
