// build_ref_check.cpp -- host builds of the index build's own key and node functions, for tests/test_build_ref_cpu.py to compare
// with the numpy restatement of the build (tests/build_ref.py).
//   build_ref_check keys  cells.bin out.bin : uint32 (x, y, z) cells -> uint32 lh_hilbert30 keys (10 bits per axis)
//   build_ref_check nodes keys.bin out.bin  : n sorted uint64 keys -> for every inner node i < n - 1 the int64 row
//                                             (first, last, split, ref0, cnt0, ref1, cnt1) of pc_lbvh_node / pc_lbvh_children
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "lbvh_host_build.hpp"

template <typename T>
static std::vector<T> read_all(const char *path)
{
    FILE *f = fopen(path, "rb");
    if (!f) { perror(path); exit(2); }
    fseek(f, 0, SEEK_END);
    const long bytes = ftell(f);
    fseek(f, 0, SEEK_SET);
    std::vector<T> v((size_t)bytes / sizeof(T));
    if (fread(v.data(), sizeof(T), v.size(), f) != v.size()) { perror(path); exit(2); }
    fclose(f);
    return v;
}

template <typename T>
static void write_all(const char *path, const std::vector<T> &v)
{
    FILE *f = fopen(path, "wb");
    if (!f || fwrite(v.data(), sizeof(T), v.size(), f) != v.size()) { perror(path); exit(2); }
    fclose(f);
}

int main(int argc, char **argv)
{
    if (argc != 4) { fprintf(stderr, "usage: %s keys|nodes in.bin out.bin\n", argv[0]); return 2; }
    if (!strcmp(argv[1], "keys")) {
        const std::vector<uint32_t> c = read_all<uint32_t>(argv[2]);
        std::vector<uint32_t> k(c.size() / 3);
        for (size_t i = 0; i < k.size(); i++) k[i] = lh_hilbert30(c[3 * i], c[3 * i + 1], c[3 * i + 2]);
        write_all(argv[3], k);
    } else if (!strcmp(argv[1], "nodes")) {
        const std::vector<uint64_t> keys = read_all<uint64_t>(argv[2]);
        const int64_t n = (int64_t)keys.size();
        std::vector<int64_t> out;
        for (int64_t i = 0; i + 1 < n; i++) {
            int64_t f, l, s;
            uint32_t r0, c0, r1, c1;
            pc_lbvh_node(keys.data(), n, i, &f, &l, &s);
            pc_lbvh_children(f, l, s, &r0, &c0, &r1, &c1);
            const int64_t row[7] = { f, l, s, r0, c0, r1, c1 };
            out.insert(out.end(), row, row + 7);
        }
        write_all(argv[3], out);
    } else {
        return 2;
    }
    printf("ok\n");
    return 0;
}
