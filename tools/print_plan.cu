// Prints the launch plans of the peak kernel (host only): nvcc -o /tmp/print_plan tools/print_plan.cu && /tmp/print_plan
// `print_plan` prints a few bench-like shapes; `print_plan table` prints one row per shape of a grid that covers both sides
// of every eligibility edge of the planner, in the format of tests/golden/launch_plans.txt.gz; `print_plan shape H W esize
// maps C K fused` prints the row of one shape in the same format (tests/test_gpu_multiwave.py sizes its batches by it).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "../object_keypoints_b200/csrc/okp_peaks_stream.cuh"

static void print_row(int H, int W, int esize, int maps, int C, int K, int fused) {
    // the fused form's grouping scratch per frame, as okp_decode_* sizes it (max_objects 16)
    const int frame_bytes = fused ? (int)okp_group_smem_bytes(C, K, 16) : 0;
    printf("%d %d %d %d %d %d %d:", H, W, esize, maps, C, K, fused);
    OkpStreamPlan sp;
    if (!okp_stream_plan(maps, C, H, W, K, esize, frame_bytes, 0, &sp)) { printf(" -\n"); return; }
    const OkpStripPlan& p = sp.s;
    printf(" %d %d %d %d %d %d %d %d %d %d %d %d %d\n", p.M, p.strips, p.halves, p.BW, p.lead[1], p.NS, p.nb,
           sp.EW, p.threads, sp.threads, sp.smem_bytes, sp.groups, sp.F);
}

static const char* kHeader = "H W esize maps C K fused: M strips halves BW lead1 NS nb EW threads total smem groups F\n";

static void print_table() {
    const int Hs[] = {1, 2, 5, 64, 65, 180, 720};
    const int Ws[] = {4, 6, 8, 12, 60, 64, 68, 252, 256, 260, 320, 496, 500, 504};
    const int maps_list[] = {1, 3, 7, 12288, 98304};
    const int Cs[] = {1, 3, 4};
    const int Ks[] = {1, 32, 256};
    printf("%s", kHeader);
    for (int H : Hs)
        for (int W : Ws)
            for (int esize = 4; esize >= 2; esize -= 2)
                for (int maps : maps_list)
                    for (int C : Cs)
                        for (int K : Ks)
                            for (int fused = 0; fused < 2; ++fused) print_row(H, W, esize, maps, C, K, fused);
}

int main(int argc, char** argv) {
    if (argc > 1 && strcmp(argv[1], "table") == 0) {
        print_table();
        return 0;
    }
    if (argc > 1 && strcmp(argv[1], "shape") == 0) {
        if (argc != 9) {
            fprintf(stderr, "usage: print_plan shape H W esize maps C K fused\n");
            return 2;
        }
        int v[7];
        for (int i = 0; i < 7; ++i) v[i] = atoi(argv[2 + i]);
        printf("%s", kHeader);
        print_row(v[0], v[1], v[2], v[3], v[4], v[5], v[6]);
        return 0;
    }
    const int shapes[][3] = {{180, 320, 4096 * 3}, {64, 64, 32768 * 3}, {64, 64, 256 * 3}, {128, 128, 3000}, {360, 480, 300}};
    for (auto& sh : shapes)
        for (int esize = 4; esize >= 2; esize -= 2)
            for (int fused = 0; fused < 2; ++fused) {
                OkpStreamPlan sp;
                const int frame_bytes = fused ? (int)okp_group_smem_bytes(3, 32, 16) : 0;
                if (!okp_stream_plan(sh[2], 3, sh[0], sh[1], 32, esize, frame_bytes, 0, &sp)) { printf("%dx%d esize %d: no plan\n", sh[0], sh[1], esize); continue; }
                printf("%3dx%3d esize %d fused %d: M %2d strips %2d compute threads %3d EW %d total threads %3d smem %6d NS %d nb %d groups %d F %d\n",
                       sh[0], sh[1], esize, fused, sp.s.M, sp.s.strips, sp.s.threads, sp.EW, sp.threads, sp.smem_bytes, sp.s.NS, sp.s.nb, sp.groups, sp.F);
            }
    return 0;
}
