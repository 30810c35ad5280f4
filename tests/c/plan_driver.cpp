// Runs the kernel planners (csic_plan.cpp) without a GPU.  One case per input line, one result line per case:
//   F W H a b f ops fmt in pool n row0 rows compact family stages tile_bytes block_threads ctas_per_sm
//     -> family grid stages ctas_per_sm tile_rows nsplit tile_px n_tiles block_threads smem_bytes Ho n_frames tall_ho
//   D W H a b f n to_rgb tile_px
//     -> ok tile_px stages threads grid smem
// `ops` is the stage order as three digits of csic_step (e.g. 312 = chroma, spatial, colour).  Buffers are dense and
// 4 KiB aligned.  Device limits: argv[1] SMs, argv[2] opt-in shared memory per block.  A line that fails parameter
// validation or build_plan prints "error <code>".
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <sstream>
#include <string>

#include "../../chroma-subsampling-image-compressor_b200/csrc/csic_internal.h"

namespace {

int make_params(std::istringstream& in, csic_params& p) {
  int W, H, a, b, f;
  in >> W >> H >> a >> b >> f;
  csic_params_default(W, H, &p);
  p.chroma_a = a; p.chroma_b = b; p.factor = f;
  p.y_bits = p.cb_bits = p.cr_bits = 8;
  return csic_validate(&p, nullptr, 0);
}

}  // namespace

int main(int argc, char** argv) {
  if (argc != 3) {
    std::fprintf(stderr, "usage: plan_driver SMS MAX_SMEM_OPTIN < cases\n");
    return 2;
  }
  const csic::DeviceLimits dev{std::atoi(argv[1]), (size_t)std::atoll(argv[2])};
  void* const in_buf = reinterpret_cast<void*>(uintptr_t(1) << 32);
  void* const out_buf = reinterpret_cast<void*>(uintptr_t(2) << 32);
  std::string line;
  while (std::getline(std::cin, line)) {
    std::istringstream in(line);
    std::string kind;
    if (!(in >> kind)) continue;
    csic_params p;
    int rc = make_params(in, p);
    if (kind == "F") {
      int ops, fmt, in_fmt, pool, row0, rows, compact;
      size_t n;
      csic::PlanOptions opt;
      in >> ops >> fmt >> in_fmt >> pool >> n >> row0 >> rows >> compact >> opt.family >> opt.stages >> opt.tile_bytes >>
          opt.block_threads >> opt.ctas_per_sm;
      p.op[0] = ops / 100; p.op[1] = ops / 10 % 10; p.op[2] = ops % 10;
      p.out_format = fmt; p.in_format = in_fmt; p.pool_mode = pool;
      if (rc == CSIC_OK) rc = csic_validate(&p, nullptr, 0);
      csic::KPlan base;
      if (rc == CSIC_OK)
        rc = csic::build_plan(p, in_buf, out_buf, n, row0, rows < 0 ? csic::geometry(p).out_h : rows, compact != 0,
                              csic::Layout(), base);
      if (rc != CSIC_OK) { std::printf("error %d\n", rc); continue; }
      const csic::KernelChoice c = csic::select_kernel(base, dev, opt);
      const csic::KPlan& k = c.k;
      std::printf("%d %u %d %d %d %d %d %u %d %u %d %u %d\n", c.family, c.grid, k.stages, k.ctas_per_sm, k.tile_rows, k.nsplit,
                  k.tile_px, k.n_tiles, k.block_threads, k.smem_bytes, k.Ho, k.n_frames, k.tall_ho);
    } else if (kind == "D") {
      size_t n;
      int to_rgb;
      uint32_t tile_px;
      in >> n >> to_rgb >> tile_px;
      p.op[0] = CSIC_STEP_CHROMA; p.op[1] = CSIC_STEP_SPATIAL; p.op[2] = CSIC_STEP_COLOR;
      p.out_format = CSIC_OUT_PLANAR;
      if (rc == CSIC_OK) rc = csic_validate(&p, nullptr, 0);
      csic::KPlan k;
      if (rc == CSIC_OK) rc = csic::build_plan(p, in_buf, out_buf, n, 0, csic::geometry(p).out_h, false, csic::Layout(), k);
      if (rc != CSIC_OK) { std::printf("error %d\n", rc); continue; }
      csic::DecodeLaunch d;
      if (!csic::plan_decode(k, to_rgb, dev, tile_px, d)) {
        std::printf("0\n");
        continue;
      }
      std::printf("1 %u %u %u %u %zu\n", d.P.tile_px, d.P.stages, d.threads, d.grid, d.smem);
    } else {
      std::printf("error bad-line\n");
    }
  }
  return 0;
}
