// Compiled and run by tests/test_gpu_gray.py: the facade on 8UC1 input.  Frame::set with a gray image must give exactly what
// it gives for the same image replicated to 8UC3 (points and distance transforms at every level), SolveEA must solve the two
// to the same pose, and an image of any other type must be refused.
#include <cstdio>
#include <cstdlib>
#include <stdexcept>
#include <vector>

#include "edge_alignment/SolveEA.h"

static std::vector<unsigned char> read_file(const char* path, size_t n) {
  std::vector<unsigned char> b(n);
  FILE* f = fopen(path, "rb");
  if (!f || fread(b.data(), 1, n, f) != n) { fprintf(stderr, "cannot read %s\n", path); exit(2); }
  fclose(f);
  return b;
}

static std::vector<unsigned char> replicate3(const std::vector<unsigned char>& g) {
  std::vector<unsigned char> b(g.size() * 3);
  for (size_t i = 0; i < g.size(); ++i) b[3 * i] = b[3 * i + 1] = b[3 * i + 2] = g[i];
  return b;
}

int main(int argc, char** argv) {
  if (argc < 6) { fprintf(stderr, "usage: gray_facade_test ref.gray ref.depth16 now.gray W H\n"); return 2; }
  const int W = atoi(argv[4]), H = atoi(argv[5]);
  auto ref_g = read_file(argv[1], size_t(W) * H);
  auto ref_d = read_file(argv[2], size_t(W) * H * 2);
  auto now_g = read_file(argv[3], size_t(W) * H);
  auto ref_b = replicate3(ref_g), now_b = replicate3(now_g);
  ea::Mat ref_gray(H, W, ea::U8C1, ref_g.data()), ref_bgr(H, W, ea::U8C3, ref_b.data()), ref_depth(H, W, ea::U16C1, ref_d.data());
  ea::Mat now_gray(H, W, ea::U8C1, now_g.data()), now_bgr(H, W, ea::U8C3, now_b.data()), none;
  try {
    // Frame::set, three pyramid levels, both roles
    ea_frame_params fp;
    ea_frame_params_default(&fp);
    fp.width = W; fp.height = H; fp.n_levels = 3;
    Frame fg(fp), fb(fp);
    fg.set(ref_gray, &ref_depth, EA_ROLE_BOTH);
    fb.set(ref_bgr, &ref_depth, EA_ROLE_BOTH);
    for (int l = 0; l < fp.n_levels; ++l) {
      const bool same = fg.edgePoints(l) == fb.edgePoints(l) && fg.distanceTransform(l) == fb.distanceTransform(l);
      printf("frame%d %d %d\n", l, int(same), fg.numEdgePoints(l));
    }
    // SolveEA (reference defaults: Canny on the colour image, exact DT) and its standalone pipeline
    for (int standalone = 0; standalone < 2; ++standalone) {
      double pose[2][7];
      for (int k = 0; k < 2; ++k) {
        SolveEA s;
        s.setK(525.0, 525.0, 319.5, 239.5);
        if (standalone) s.useStandalonePipeline();
        s.setRefFrame(k ? ref_bgr : ref_gray, ref_depth);
        s.setNowFrame(k ? now_bgr : now_gray, none);
        s.setAsCERESProblem();
        s.getPose(pose[k], pose[k] + 4);
      }
      bool same = true;
      for (int i = 0; i < 7; ++i) same = same && pose[0][i] == pose[1][i];
      printf("solve%d %d %.9f %.9f %.9f\n", standalone, int(same), pose[0][4], pose[0][5], pose[0][6]);
    }
    // an image of another type is refused instead of being read as BGR
    std::vector<uint16_t> wide(size_t(W) * H, 0);
    ea::Mat u16(H, W, ea::U16C1, wide.data());
    bool threw = false;
    try { fg.set(u16, &ref_depth, EA_ROLE_BOTH); } catch (const std::runtime_error&) { threw = true; }
    printf("u16 %d\n", int(threw));
  } catch (const std::exception& e) { fprintf(stderr, "exception: %s\n", e.what()); return 1; }
  return 0;
}
