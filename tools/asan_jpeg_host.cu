// AddressSanitizer / UBSan harness for the HOST half of the JPEG decoder (header parser, device table builder and Huffman
// decoder of csrc/p2p_jpegdec.cuh): every file named on the command line is read into an exact-size heap buffer and decoded.
// No CUDA call is made, so it runs without a GPU.
//   nvcc -O1 -g -Xcompiler -fsanitize=address,-fsanitize=undefined,-fno-omit-frame-pointer \
//        -gencode arch=compute_100a,code=sm_100a -o /tmp/asan_jpeg_host tools/asan_jpeg_host.cu -lasan -lubsan
//   ASAN_OPTIONS=detect_leaks=0 /tmp/asan_jpeg_host damaged/*.jpg
// (tests/test_jpeg_oracle.py::test_host_decoder_under_address_sanitizer builds and runs it on seeded damaged files,
// tests/test_jpeg_progressive_scripts_oracle.py on progressive files of every scan script and damaged copies of them)
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../360-to-planer-images_b200/csrc/p2p_jpegdec.cuh"

int main(int argc, char **argv) {
    int decoded = 0, declined = 0;
    for (int a = 1; a < argc; ++a) {
        FILE *f = fopen(argv[a], "rb");
        if (!f) return 2;
        fseek(f, 0, SEEK_END);
        const long n = ftell(f);
        fseek(f, 0, SEEK_SET);
        uint8_t *buf = static_cast<uint8_t *>(malloc(n ? (size_t)n : 1));
        if (fread(buf, 1, (size_t)n, f) != (size_t)n) return 2;
        fclose(f);
        p2pjdec::Parsed P;
        if (p2pjdec::parse_headers(buf, (size_t)n, P) == 0) {
            if (!P.progressive) {   // the tables the device stage would upload
                std::vector<unsigned char> mem(sizeof(p2pjdec::DevTables));
                p2pjdec::build_device_tables(P, *reinterpret_cast<p2pjdec::DevTables *>(mem.data()));
            }
            std::vector<int16_t> coef(P.info.n_coef);
            if (p2pjdec::decode_scan(buf, (size_t)n, P, coef.data()) == 0) ++decoded;
            else ++declined;
        } else {
            ++declined;
        }
        free(buf);
    }
    printf("decoded %d declined %d\n", decoded, declined);
    return 0;
}
