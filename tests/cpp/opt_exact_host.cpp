// Solves QPs through wbc_b200::OPT (include/wbc_dogctrl.hpp) with exact_qp = true.  Usage:
//   opt_exact_host IN.bin OUT.bin -> IN: m, nrows (86 or 82), neq (int32), then per QP Q 900, c 30, L nrows*31 (doubles);
//                                     OUT: per QP x 30 and the status word (doubles)
#include <cstdio>
#include <vector>

#include "wbc_dogctrl.hpp"

struct Dense {
    const double* a;
    int cols;
    double operator()(int i, int j) const { return a[i * cols + j]; }
    double operator()(int i) const { return a[i]; }
};
struct Vec30 {
    double a[30];
    double& operator()(int i) { return a[i]; }
};

int main(int argc, char** argv)
{
    if (argc < 3) return 2;
    FILE* fi = fopen(argv[1], "rb");
    FILE* fo = fopen(argv[2], "wb");
    if (!fi || !fo) return 3;
    int hdr[3];
    if (fread(hdr, 4, 3, fi) != 3) return 3;
    const int m = hdr[0], nrows = hdr[1], neq = hdr[2];
    if ((nrows != 86 || neq != 18) && (nrows != 82 || neq != 12)) return 4;
    try {
        wbc_b200::OPT opt(30, 86, 82);
        opt.exact_qp = true;
        std::vector<double> buf(900 + 30 + (size_t)nrows * 31);
        for (int k = 0; k < m; k++) {
            if (fread(buf.data(), 8, buf.size(), fi) != buf.size()) return 3;
            opt.setQ(Dense{buf.data(), 30});
            opt.setc(Dense{buf.data() + 900, 1});
            Vec30 x;
            for (int i = 0; i < 30; i++) x.a[i] = 0.0;
            if (nrows == 86) {
                opt.setL_stance(Dense{buf.data() + 930, 31});
                opt.opt_stance(x);
            } else {
                opt.setL_swing(Dense{buf.data() + 930, 31});
                opt.opt_swing(x);
            }
            double rec[31];
            for (int i = 0; i < 30; i++) rec[i] = x.a[i];
            rec[30] = opt.last_status;
            if (fwrite(rec, 8, 31, fo) != 31) return 3;
        }
    } catch (const wbc_b200::Error& e) {
        fprintf(stderr, "%s\n", e.what());
        return 5;
    }
    fclose(fi);
    fclose(fo);
    return 0;
}
