// Runs the kernel planners (csic_plan.cpp) without a GPU.  One case per input line, one result line per case:
//   F W H a b f ops fmt in pool n row0 rows compact family stages tile_bytes block_threads ctas_per_sm
//     [in_pitch in_frame out_pitch out_frame [y_bits cb_bits cr_bits]]
//     -> family grid stages ctas_per_sm tile_rows nsplit tile_px n_tiles block_threads smem_bytes Ho n_frames tall_ho
//        slots_per_row in_dense out_dense
//   D W H a b f n to_rgb tile_px [walk]
//     -> ok tile_px stages threads grid smem
//        [tiles_per_frame n_tiles A cw hs_sh vhold last_c y_slot c_slot frame_bytes cb_off cr_off]
//        (with any trailing token: what the decoder's producer reads from DecPlan; "0" when plan_decode declines)
//   H W H a b f ops fmt in pool n row0 rows full_frames chunk_bytes share_gpus
//     -> one JSON object: the host plan (plan_host) and, per chunk, the copies (frame_copies) of the direct path
//        (h2d: caller -> staging, d2h: staging -> caller) and of the bounce path (gather: caller -> bounce, b2d, d2b,
//        scatter: bounce -> caller), each [dst offset, dst pitch, src offset, src pitch, width, height]
//   B W H a b f ops G
//     -> r0 r1 of each of G GPUs (band_split)
// `ops` is the stage order as three digits of csic_step (e.g. 312 = chroma, spatial, colour); rows -1: all.  Buffers
// are 4 KiB aligned and dense, except that an F line may end in a layout (row pitches and frame strides in bytes, 0 =
// dense, as csic_process_device_pitched takes them) and then in the bit depths of Y, Cb and Cr (default 8 each: they
// set the slot width of the bundle formats).  Device limits: argv[1] SMs, argv[2] opt-in shared memory per block.  A
// line that fails parameter validation, build_plan or plan_host prints "error <code>".
#include <algorithm>
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

void set_ops(csic_params& p, int ops) { p.op[0] = ops / 100; p.op[1] = ops / 10 % 10; p.op[2] = ops % 10; }

void print_copies(const char* name, const std::vector<csic::Copy>& cs) {
  std::printf(", \"%s\": [", name);
  for (size_t i = 0; i < cs.size(); ++i)
    std::printf("%s[%zu, %zu, %zu, %zu, %zu, %zu]", i ? ", " : "", cs[i].dst, cs[i].dst_pitch, cs[i].src, cs[i].src_pitch,
                cs[i].width, cs[i].height);
  std::printf("]");
}

void print_side(const char* name, const csic::CopySide& s) {
  std::printf(", \"%s\": [%zu, %zu, %zu]", name, s.off, s.pitch, s.frame);
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
      csic::Layout lay;
      for (size_t* v : {&lay.in_pitch, &lay.in_frame, &lay.out_pitch, &lay.out_frame})
        if (!(in >> *v)) *v = 0;
      int bits[3] = {8, 8, 8};
      for (int& b : bits)
        if (!(in >> b)) b = 8;
      p.y_bits = bits[0]; p.cb_bits = bits[1]; p.cr_bits = bits[2];
      set_ops(p, ops);
      p.out_format = fmt; p.in_format = in_fmt; p.pool_mode = pool;
      if (rc == CSIC_OK) rc = csic_validate(&p, nullptr, 0);
      csic::KPlan base;
      if (rc == CSIC_OK)
        rc = csic::build_plan(p, in_buf, out_buf, n, row0, rows < 0 ? csic::geometry(p).out_h : rows, compact != 0,
                              lay, base);
      if (rc != CSIC_OK) { std::printf("error %d\n", rc); continue; }
      const csic::KernelChoice c = csic::select_kernel(base, dev, opt);
      const csic::KPlan& k = c.k;
      std::printf("%d %u %d %d %d %d %d %u %d %u %d %u %d %d %d %d\n", c.family, c.grid, k.stages, k.ctas_per_sm, k.tile_rows,
                  k.nsplit, k.tile_px, k.n_tiles, k.block_threads, k.smem_bytes, k.Ho, k.n_frames, k.tall_ho, k.slots_per_row,
                  k.in_dense, k.out_dense);
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
      std::printf("1 %u %u %u %u %zu", d.P.tile_px, d.P.stages, d.threads, d.grid, d.smem);
      std::string more;
      if (in >> more)
        std::printf(" %u %u %u %u %u %u %u %u %u %llu %llu %llu", d.P.tiles_per_frame, d.P.n_tiles, d.P.A, d.P.cw, d.P.hs_sh,
                    d.P.vhold, d.P.last_c, d.P.y_slot, d.P.c_slot, (unsigned long long)d.P.frame_bytes,
                    (unsigned long long)d.P.cb_off, (unsigned long long)d.P.cr_off);
      std::printf("\n");
    } else if (kind == "H") {
      int ops, fmt, in_fmt, pool, row0, rows, full;
      size_t n, chunk, gpus;
      in >> ops >> fmt >> in_fmt >> pool >> n >> row0 >> rows >> full >> chunk >> gpus;
      set_ops(p, ops);
      p.out_format = fmt; p.in_format = in_fmt; p.pool_mode = pool;
      if (rc == CSIC_OK) rc = csic_validate(&p, nullptr, 0);
      if (rc == CSIC_OK && rows < 0) rows = csic::geometry(p).out_h;
      int32_t in_row0 = 0, in_rows = p.height;
      if (rc == CSIC_OK) rc = csic_band_input_rows(&p, row0, rows, &in_row0, &in_rows);
      csic::HostPlan h;
      if (rc == CSIC_OK) rc = csic::plan_host(p, row0, rows, n, dev, csic::PlanOptions(), chunk, full != 0, gpus, h);
      if (rc != CSIC_OK) { std::printf("error %d\n", rc); continue; }
      const csic::Layout& l = h.lay;
      std::printf("{\"compact\": %d, \"first_stored\": %zu, \"in_pitch\": %zu, \"out_pitch\": %zu, \"per\": %zu, "
                  "\"in_rows\": [%d, %d], \"lay\": [%zu, %zu, %zu, %zu, %d], \"in_shape\": [%zu, %zu], \"out_shape\": [%zu, %zu]",
                  h.compact ? 1 : 0, h.first_stored, h.in_pitch, h.out_pitch, h.frames_per_chunk, in_row0, in_rows,
                  l.in_pitch, l.in_frame, l.out_pitch, l.out_frame, l.short_frames ? 1 : 0, h.in.width, h.in.rows,
                  h.out.width, h.out.rows);
      print_side("in_caller", h.in.caller); print_side("in_bounce", h.in.bounce); print_side("in_staging", h.in.staging);
      print_side("out_caller", h.out.caller); print_side("out_bounce", h.out.bounce); print_side("out_staging", h.out.staging);
      std::printf(", \"chunks\": [");
      for (size_t f0 = 0; f0 < n; f0 += h.frames_per_chunk) {
        const size_t nf = std::min(h.frames_per_chunk, n - f0);
        std::printf("%s{\"f0\": %zu, \"nf\": %zu", f0 ? ", " : "", f0, nf);
        print_copies("h2d", csic::frame_copies(h.in, h.in.staging, h.in.caller.at(f0), nf));
        print_copies("d2h", csic::frame_copies(h.out, h.out.caller.at(f0), h.out.staging, nf));
        print_copies("gather", csic::frame_copies(h.in, h.in.bounce, h.in.caller.at(f0), nf));
        print_copies("b2d", csic::frame_copies(h.in, h.in.staging, h.in.bounce, nf));
        print_copies("d2b", csic::frame_copies(h.out, h.out.bounce, h.out.staging, nf));
        print_copies("scatter", csic::frame_copies(h.out, h.out.caller.at(f0), h.out.bounce, nf));
        std::printf("}");
      }
      std::printf("]}\n");
    } else if (kind == "B") {
      int ops;
      size_t G;
      in >> ops >> G;
      set_ops(p, ops);
      if (rc == CSIC_OK) rc = csic_validate(&p, nullptr, 0);
      if (rc != CSIC_OK) { std::printf("error %d\n", rc); continue; }
      for (size_t i = 0; i < G; ++i) {
        int32_t r0, r1;
        csic::band_split(p, i, G, r0, r1);
        std::printf("%s%d %d", i ? " " : "", r0, r1);
      }
      std::printf("\n");
    } else {
      std::printf("error bad-line\n");
    }
  }
  return 0;
}
