// Headless counterpart of the reference's Source/main.cpp:9-21 — the same wiring (Evaluator -> Marching) without the
// GLUT/ImGui drawer: polygonise one equation, print counts and stage timings, optionally dump the mesh as the
// reference's ASCII PLY (marching.cpp:821-850) and/or a lossless binary dump.
//
//   mcb_headless [--eq "x^2+y^2+z^2-0.49" | --eq-file example_files/equation_1.txt] [--step 0.2 | --res 1024]
//                [--scale sx sy sz] [--iso c] [--constraint i "lhs" "op" rhs]... [--no-normals] [--soup]
//                [--ply out.ply] [--dump out.bin] [--repeat n] [--levels d]   (--levels: repeating-surface mode, distance d)
//                [--devices n]   (z-slabs over GPUs 0..n-1 of this box: Marching::set_devices)
//                [--functions]   (equations and constraints may use sin( cos( sqrt( abs( min( max(: Evaluator::set_function_grammar)
//                [--analytic-normals]   (normals from the equation's own gradient: Marching::set_analytic_normals)
//                [--dump-normals out.bin]   (the welded vertex normals, nv*3 f32, or the soup's 3 float4 per triangle)
//                [--refine-vertices]   (every vertex moved to the equation's root on its grid edge: Marching::set_refined_vertices)
//                [--dual-contouring]   (the dual-contoured mesh, sharp edges and corners kept: Marching::set_dual_contouring)
//
// Defaults are the reference GUI's (drawer.cpp:39-44): equation "x+y", grid 0.2, scale 1.1, iso 0.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "marching.h"

static int usage() {
    std::fprintf(stderr, "usage: mcb_headless [--eq S | --eq-file F] [--step h | --res n] [--scale sx sy sz] [--iso c]\n"
                         "                    [--constraint i lhs op rhs] [--no-normals] [--soup] [--ply F] [--dump F] [--repeat n] [--levels d] [--devices n]\n"
                         "                    [--functions] [--analytic-normals] [--dump-normals F] [--refine-vertices]\n"
                         "                    [--dual-contouring]\n");
    return 2;
}

int main(int argc, char** argv) {
    Evaluator evaluator;
    Marching march_maker;
    march_maker.set_evaluator(&evaluator);
    float step = 0.2f, sx = 1.1f, sy = 1.1f, sz = 1.1f, iso = 0.f;
    int res = 0, repeat = 1;
    std::string ply, dump, dump_normals;
    for (int a = 1; a < argc; a++) /* before any equation is parsed, wherever it stands */
        if (std::strcmp(argv[a], "--functions") == 0) evaluator.set_function_grammar(true);
    for (int a = 1; a < argc; a++) {
        const std::string o = argv[a];
        auto need = [&](int n) { return a + n < argc; };
        if (o == "--eq" && need(1)) {
            if (!evaluator.set_equation(argv[++a])) { std::fprintf(stderr, "equation rejected\n"); return 1; }
        } else if (o == "--eq-file" && need(1)) {
            setenv("MCB_EQUATION_FILE", argv[++a], 1);
            std::string s;
            if (!evaluator.get_equation_from_file(s)) { std::fprintf(stderr, "cannot read an equation from %s\n", argv[a]); return 1; }
        } else if (o == "--step" && need(1)) step = (float)std::atof(argv[++a]);
        else if (o == "--res" && need(1)) res = std::atoi(argv[++a]);
        else if (o == "--scale" && need(3)) { sx = (float)std::atof(argv[a + 1]); sy = (float)std::atof(argv[a + 2]); sz = (float)std::atof(argv[a + 3]); a += 3; }
        else if (o == "--iso" && need(1)) iso = (float)std::atof(argv[++a]);
        else if (o == "--constraint" && need(4)) {
            const int i = std::atoi(argv[a + 1]);
            if (!march_maker.set_constraint(i, argv[a + 2], argv[a + 3], (float)std::atof(argv[a + 4])) || !march_maker.use_constraint(i, true)) {
                std::fprintf(stderr, "constraint rejected\n");
                return 1;
            }
            a += 4;
        } else if (o == "--functions") continue;
        else if (o == "--no-normals") march_maker.set_normals(false);
        else if (o == "--analytic-normals") march_maker.set_analytic_normals(true);
        else if (o == "--refine-vertices") march_maker.set_refined_vertices(true);
        else if (o == "--dual-contouring") march_maker.set_dual_contouring(true);
        else if (o == "--soup") march_maker.set_weld(false);
        else if (o == "--ply" && need(1)) ply = argv[++a];
        else if (o == "--dump" && need(1)) dump = argv[++a];
        else if (o == "--dump-normals" && need(1)) dump_normals = argv[++a];
        else if (o == "--repeat" && need(1)) repeat = std::atoi(argv[++a]);
        else if (o == "--devices" && need(1)) { if (!march_maker.set_devices(std::atoi(argv[++a]))) { std::fprintf(stderr, "bad device count\n"); return 1; } }
        else if (o == "--levels" && need(1)) { /* Marching::set_surface_repeat_step_distance + repeating_surface_mode */
            if (!march_maker.set_surface_repeat_step_distance((float)std::atof(argv[++a]))) { std::fprintf(stderr, "the level distance must be positive\n"); return 1; }
            march_maker.repeating_surface_mode(true);
        }
        else return usage();
    }
    if (res > 0 ? !march_maker.set_grid_resolution(res) : !march_maker.set_grid_step_size(step)) {
        std::fprintf(stderr, "grid step rejected (the reference accepts [0.001, 0.5]; use --res n for finer grids)\n");
        return 1;
    }
    march_maker.set_scaling_x(sx); march_maker.set_scaling_y(sy); march_maker.set_scaling_z(sz);
    march_maker.set_surface_constant(iso);
    const Poly_Data* pData = march_maker.get_poly_data();
    double best_ms = 1e30, first_ms = 0, steady_sum = 0;
    int steady_n = 0;
    for (int r = 0; r < repeat; r++) {
        const auto t0 = std::chrono::steady_clock::now();
        if (!march_maker.recalculate()) {
            std::fprintf(stderr, "recalculate failed: %s (is there a CUDA device? there is no CPU fallback)\n", march_maker.last_error());
            return 1;
        }
        const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (ms < best_ms) best_ms = ms;
        if (r == 0) {                                   /* context creation, buffer growth; NVRTC works in the background */
            first_ms = ms;
            if (repeat > 1) march_maker.wait_for_compiled_kernels(); /* the steady state is what the other calls measure */
        }
        if (r >= 3 || repeat < 6) { steady_sum += ms; steady_n++; } /* the first calls size and page-lock the Poly_Data vectors */
    }
    const mcb_counts& c = march_maker.last_counts();
    std::printf("{\"equation\": \"%s\", \"M\": %d, \"cubes\": %llu, \"active\": %llu, \"triangles\": %llu, \"vertices\": %zu, "
                "\"ambiguous\": %llu, \"redirected\": %llu, \"ms_eval\": %.4f, \"ms_classify\": %.4f, \"ms_emit\": %.4f, \"ms_weld\": %.4f, "
                "\"ms_device\": %.4f, \"ms_recalculate_wall\": %.3f, \"ms_recalculate_mean\": %.3f, \"ms_recalculate_first\": %.3f, \"calls\": %d}\n",
                evaluator.equation().c_str(), c.M, (unsigned long long)c.cubes, (unsigned long long)c.active,
                (unsigned long long)c.triangles, pData->vertex_list.size() / 3, (unsigned long long)c.ambiguous,
                (unsigned long long)c.redirected, c.ms_eval, c.ms_classify, c.ms_emit, c.ms_weld, c.ms_total, best_ms,
                steady_n ? steady_sum / steady_n : best_ms, first_ms, repeat);
    {
        const Marching::DeviceTiming& dt = march_maker.last_device_timing();
        if (dt.polygonise > 0)
            std::fprintf(stderr, "devices: polygonise+exchange %.3f ms, size+page-lock Poly_Data %.3f ms, copies+index fix-up %.3f ms (last call)\n",
                         dt.polygonise, dt.prepare, dt.fetch);
    }
    if (!ply.empty()) {
        setenv("MCB_MESH_FILE", ply.c_str(), 1);
        if (!march_maker.save_poly_to_file()) { std::fprintf(stderr, "nothing to save / cannot write %s\n", ply.c_str()); return 1; }
    }
    if (!dump.empty()) { /* lossless: u64 nv, u64 nt, nv*3 f32, nt*3 u32 */
        FILE* fp = std::fopen(dump.c_str(), "wb");
        if (!fp) return 1;
        const unsigned long long nv = pData->vertex_list.size() / 3, nt = pData->tri_list.size() / 3;
        std::fwrite(&nv, 8, 1, fp); std::fwrite(&nt, 8, 1, fp);
        std::fwrite(pData->vertex_list.data(), 4, pData->vertex_list.size(), fp);
        std::fwrite(pData->tri_list.data(), 4, pData->tri_list.size(), fp);
        std::fclose(fp);
    }
    if (!dump_normals.empty()) {
        const std::vector<float>& n = march_maker.get_vertex_normals().empty() ? march_maker.get_normals() : march_maker.get_vertex_normals();
        FILE* fp = std::fopen(dump_normals.c_str(), "wb");
        if (!fp) return 1;
        std::fwrite(n.data(), 4, n.size(), fp);
        std::fclose(fp);
    }
    return 0;
}
