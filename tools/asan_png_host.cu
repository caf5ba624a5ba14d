// AddressSanitizer / UBSan harness for the PNG decoder's routines (csrc/p2p_pngdec.cuh): every file named on the command
// line is read into an exact-size heap buffer and run through the serial host model of the device decoder - the same
// __host__ __device__ bit reader, header parser, table builder, block decoder, tail / resolution passes and filters the
// kernels execute.  No CUDA call is made, so it runs without a GPU.
//   nvcc -O1 -g -Xcompiler -fsanitize=address,-fsanitize=undefined,-fno-omit-frame-pointer \
//        -gencode arch=compute_100a,code=sm_100a -o /tmp/asan_png_host tools/asan_png_host.cu -lasan -lubsan
//   ASAN_OPTIONS=detect_leaks=0 /tmp/asan_png_host [--formats 1] damaged/*.png
// (--formats: the decoder's subset, P2P_OPT_PNG_FORMATS; tests/test_png_decode_oracle.py and
// tests/test_png_decode_formats_oracle.py build and run it on seeded damaged files)
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../360-to-planer-images_b200/csrc/p2p_pngdec.cuh"

int main(int argc, char **argv) {
    int decoded = 0, declined = 0, formats = 0, first = 1;
    if (argc > 2 && strcmp(argv[1], "--formats") == 0) {
        formats = atoi(argv[2]);
        first = 3;
    }
    for (int a = first; a < argc; ++a) {
        FILE *f = fopen(argv[a], "rb");
        if (!f) return 2;
        fseek(f, 0, SEEK_END);
        const long n = ftell(f);
        fseek(f, 0, SEEK_SET);
        uint8_t *buf = static_cast<uint8_t *>(malloc(n ? (size_t)n : 1));
        if (fread(buf, 1, (size_t)n, f) != (size_t)n) return 2;
        fclose(f);
        p2ppdec::Parsed P;
        if (p2ppdec::parse_png(buf, (size_t)n, P, formats) == 0) {
            std::vector<uint8_t> bgr((size_t)P.info.W * P.info.H * 3);
            if (p2ppdec::decode_host_model(buf, (size_t)n, bgr.data(), (size_t)P.info.W * 3, nullptr, formats) == 0) ++decoded;
            else ++declined;
        } else {
            ++declined;
        }
        free(buf);
    }
    printf("decoded %d declined %d\n", decoded, declined);
    return 0;
}
