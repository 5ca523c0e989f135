// Solves QPs twice through one wbc_b200::OPT (include/wbc_dogctrl.hpp) with exact_qp and warm_start: the first pass starts
// each QP from the previous QP's final active set, the second from the first pass's last one.  Usage:
//   opt_warm_host IN.bin OUT.bin -> IN: m, nrows (86 or 82), neq (int32), then per QP Q 900, c 30, L nrows*31 (doubles);
//                                   OUT: per pass and QP x 30, the status word and the warm rows added (last_info[6]) (doubles)
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
    const size_t per = 900 + 30 + (size_t)nrows * 31;
    std::vector<double> all(per * m);
    if (fread(all.data(), 8, all.size(), fi) != all.size()) return 3;
    try {
        wbc_b200::OPT opt(30, 86, 82);
        opt.exact_qp = true;
        opt.warm_start = true;
        for (int pass = 0; pass < 2; pass++) {
            for (int k = 0; k < m; k++) {
                const double* buf = all.data() + per * k;
                opt.setQ(Dense{buf, 30});
                opt.setc(Dense{buf + 900, 1});
                Vec30 x;
                for (int i = 0; i < 30; i++) x.a[i] = 0.0;
                if (nrows == 86) {
                    opt.setL_stance(Dense{buf + 930, 31});
                    opt.opt_stance(x);
                } else {
                    opt.setL_swing(Dense{buf + 930, 31});
                    opt.opt_swing(x);
                }
                double rec[32];
                for (int i = 0; i < 30; i++) rec[i] = x.a[i];
                rec[30] = opt.last_status;
                rec[31] = opt.last_info[6];
                if (fwrite(rec, 8, 32, fo) != 32) return 3;
            }
        }
    } catch (const wbc_b200::Error& e) {
        fprintf(stderr, "%s\n", e.what());
        return 5;
    }
    fclose(fi);
    fclose(fo);
    return 0;
}
