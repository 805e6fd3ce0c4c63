// CPU harness around trueconsense_b200/csrc/cuda/deflate_core.cuh (the same source bamwrite.cu's kernel compiles): one
// member compressed by running the kernel's phases on one thread, so the CPU test-suite can check the bytes against zlib
// and against the GPU's members.  Test infrastructure only.
#include <stdlib.h>
#include <string.h>

#include "deflate_core.cuh"

using namespace tcdef;

// raw DEFLATE of in[0 .. n) (n <= 0xff00) into out (room for n + 8 bytes); returns its length, -1 for a bad size
extern "C" int h_deflate(const uint8_t* in, int n, uint8_t* out, uint32_t* crc, int n_threads) {
    if (n < 0 || n > MEMBER_MAX || n_threads <= 0 || n_threads % 32) return -1;
    member_smem* s = (member_smem*)calloc(1, sizeof(member_smem));
    uint32_t* words = (uint32_t*)calloc((size_t)n / 4 + 16, 4);
    memcpy(s->in, in, (size_t)n);
    deflate_member(*s, n, words, n_threads, 0);
    const int len = s->t.out_bytes;
    memcpy(out, words, (size_t)len);
    *crc = s->t.crc;
    free(words);
    free(s);
    return len;
}
