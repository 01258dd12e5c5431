/* Drop-in for the reference's Source/marching.h (class Marching, marching.h:72-157) on top of the C ABI (mcb.h).
 *
 * The public surface — Step_Data, Poly_Data, xyz, Constraint's comparison names, and every public method of Marching —
 * keeps the reference's names, signatures and bool-return conventions, so main.cpp:11-20, drawer.cpp:785-942 and
 * normal.h compile against this header.  recalculate() (marching.cpp:308-433, full-grid branch :368-384) runs on the
 * GPU: field + sign planes -> classify/scan/compact -> emit; the triangle soup comes back in the reference's emission
 * order and fills Poly_Data.
 *
 * Poly_Data::vertex_list / tri_list: by default the GPU produces them directly in the reference's layout — vertices
 * welded and numbered the way add_step_to_poly_data / add_point do it (marching.cpp:599-654; tolerance comparator of
 * marching.h:38-54, first-inserted coordinates win) — because that is what the GL drawer and normal.h expect; see
 * the weld kernels in csrc/mcb_kernels.cuh and DESIGN.md for the one documented deviation.  set_weld(false) hands
 * out the unwelded float4 soup with a trivial index list instead.
 *
 * Seed mode (seed_mode / set_seed, marching.cpp:42-137, 310-331) runs on the GPU too: the same cubes and triangles as
 * the reference's BFS from the seed cube, emitted in the full-grid loop order instead of BFS order (get_seed_queue()
 * stays empty).  Step-by-step mode (marching.cpp:386-428) advances one cube per recalculate() like the reference: the
 * cube is computed on the GPU (mcb_inspect_cube = calculate_step) and appended on the host.  Not carried over: the
 * step-by-step inside seed mode and the repeating-surface mode combined with seed mode.
 * load/save of .ply use plain files ("mesh.ply" or $MCB_MESH_FILE) instead of Win32 dialogs.
 *
 * Extensions: set_grid_resolution(n) (step 2/n without the 0.001 floor, SURVEY.md D4), set_slab(k0,k1) for z-slab
 * sharding, set_normals(bool), get_normals() (central-difference gradient normals per soup vertex), last_counts().
 */
#pragma once

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <deque>
#include <set>
#include <string>
#include <chrono>
#include <thread>
#include <vector>

#include "evaluator.h"
#include "mcb.h"

struct Step_Data {
    int step_i;                         /* -2 not started, -1 finished (step-by-step mode is not carried over) */
    std::vector<float> corner_coords;   /* 24 */
    std::vector<float> corner_values;   /* 8 */
    std::vector<float> intersect_coord;
    std::vector<int> tri_vlist;
    std::vector<int> edge_list;
    float surf_constant;
};

struct Poly_Data {
    std::vector<float> vertex_list;       /* xyz per vertex */
    std::vector<unsigned int> tri_list;   /* 3 indices per triangle */
    Step_Data step_data;
};

/* point with the reference's tolerance ordering (marching.h:33-55): |d| < 1e-6 per axis counts as equal */
struct xyz {
    float x, y, z;
    int idx;
    xyz() : x(NAN), y(NAN), z(NAN), idx(-1) {}
    xyz(float a, float b, float c, int i) : x(a), y(b), z(c), idx(i) {}
    xyz(float a, float b, float c) : x(a), y(b), z(c), idx(-1) {}
    bool close_enough(float a, float b) const { return std::fabs(a - b) < 0.000001; }
    bool operator<(const xyz& r) const {
        if (!close_enough(x, r.x)) return x < r.x;
        if (!close_enough(y, r.y)) return y < r.y;
        if (!close_enough(z, r.z)) return z < r.z;
        return false;
    }
};

enum Comp_Op { GT, LT, GE, LE, NAO };

class Marching {
public:
    Marching()
        : ctx_(nullptr), evaluator_(nullptr), step_(0.25f), iso_(0.f), sx_(1.f), sy_(1.f), sz_(1.f), weld_(true),
          normals_(true), seed_mode_(false), step_mode_(false), repeat_(false), repeat_step_(0.f) {
        seed_[0] = seed_[1] = seed_[2] = 0.f;
        poly_data.step_data.corner_coords.resize(24);
        poly_data.step_data.corner_values.resize(8);
        poly_data.step_data.step_i = -2;
        poly_data.step_data.surf_constant = 0.f;
        for (int i = 0; i < 3; i++) { cons_valid_[i] = cons_use_[i] = false; cons_op_[i] = NAO; cons_rhs_[i] = 0.f; }
        counts_ = mcb_counts();
    }
    ~Marching() {
        unpin_all();
        release_devices();
        if (ctx_) mcb_destroy(ctx_);
    }
    Marching(const Marching&) = delete;
    Marching& operator=(const Marching&) = delete;

    bool set_evaluator(Evaluator* e) { if (!e) return false; evaluator_ = e; return true; } /* borrowed, marching.cpp:140-147 */
    Poly_Data const* get_poly_data() { return &poly_data; }
    std::deque<xyz> const* get_seed_queue() { return &seed_queue_; }

    bool recalculate() {
        if (!ensure_ctx()) return false;
        if (step_mode_ && !seed_mode_) { unpin_all(); return step_once(); } /* marching.cpp:386-428 */
        if (devices_ > 1 && weld_ && !seed_mode_ && !(repeat_ && !(repeat_step_ > 0.f))) return recalculate_on_devices();
        /* reset_all_data() of the reference (marching.cpp:293-305), except that vertex_list / tri_list keep their storage
         * AND their size until the new mesh is in: the GPU streams the new Poly_Data straight into them (below) */
        reset_step_data();
        if (!evaluator_) { poly_data.vertex_list.clear(); poly_data.tri_list.clear(); return true; } /* Marching::evaluate returns 0 without an evaluator */
        if (!push_parameters()) return false;
        /* welded: the GPU builds Poly_Data's own layout (vertex_list + tri_list, numbered and welded like
         * add_step_to_poly_data, marching.cpp:599-654); unwelded: the float4 triangle soup */
        mcb_set_seed(ctx_, seed_mode_ ? 1 : 0, seed_[0], seed_[1], seed_[2]); /* marching.cpp:310-331, as a set (loop order) */
        mcb_set_mesh_mode(ctx_, weld_ ? MCB_MESH_INDEXED : MCB_MESH_SOUP);
        if (repeat_ && !(repeat_step_ > 0.f)) { /* distance 0: NaN iso levels, no cube is active */
            poly_data.vertex_list.clear(); poly_data.tri_list.clear();
            soup_.clear(); normals_soup_.clear(); vertex_normals_.clear();
            poly_data.step_data.step_i = -1;
            return true;
        }
        if (weld_) {
            /* Poly_Data's vectors, page-locked where they are, are the destination of the device's copy engine: while the
             * later parts of the mesh are still being welded the earlier ones are already crossing PCIe, and the call
             * returns with Poly_Data filled (drawer.cpp:795-801 reads it next).  That needs the vectors to be large
             * enough before the mesh size is known: they are whenever the mesh did not grow since the last call — a
             * repeated or shrinking configuration; a growing one takes the plain copy below once, then streams again. */
            const size_t cv = poly_data.vertex_list.size() / 3, ct = poly_data.tri_list.size() / 3;
            const bool with_n = normals_mode() == 1;
            bool stream = cv > 0 && ct > 0 && normals_mode() <= 1 && (!with_n || vertex_normals_.size() / 3 >= cv);
            if (stream) stream = pin(pin_v_, poly_data.vertex_list) && pin(pin_t_, poly_data.tri_list) && (!with_n || pin(pin_n_, vertex_normals_));
            mcb_set_host_output(ctx_, stream ? poly_data.vertex_list.data() : nullptr, stream ? poly_data.tri_list.data() : nullptr,
                                stream && with_n ? vertex_normals_.data() : nullptr, stream ? cv : 0, stream ? ct : 0);
            if (mcb_polygonise(ctx_, &counts_) != MCB_OK) return false;
            const size_t T = (size_t)counts_.triangles, nv = (size_t)counts_.vertices;
            const bool filled = stream && mcb_host_output_filled(ctx_) != 0;
            if (nv * 3 > poly_data.vertex_list.capacity() || T * 3 > poly_data.tri_list.capacity() ||
                (normals_ && nv * 3 > vertex_normals_.capacity()))
                unpin_all(); /* a vector is about to move: its old storage must not stay page-locked */
            poly_data.vertex_list.resize(nv * 3); /* shrinks (free) when the mesh was streamed, grows otherwise */
            poly_data.tri_list.resize(T * 3);
            if (normals_) vertex_normals_.resize(nv * 3); else vertex_normals_.clear();
            soup_.clear(); normals_soup_.clear();
            if (!filled && T && mcb_get_indexed_mesh(ctx_, poly_data.vertex_list.data(), poly_data.tri_list.data(),
                                                     normals_ ? vertex_normals_.data() : nullptr, nv, T) != MCB_OK) return false;
        } else {
            unpin_all();
            mcb_set_host_output(ctx_, nullptr, nullptr, nullptr, 0, 0);
            if (mcb_polygonise(ctx_, &counts_) != MCB_OK) return false;
            const size_t T = (size_t)counts_.triangles;
            soup_.resize(T * 12);
            if (normals_) normals_soup_.resize(T * 12); else normals_soup_.clear();
            vertex_normals_.clear();
            if (T && mcb_get_mesh(ctx_, soup_.data(), normals_ ? normals_soup_.data() : nullptr, T) != MCB_OK) return false;
            fill_poly_data_from_soup();
        }
        poly_data.step_data.step_i = -1;
        return true;
    }

    void reset_all_data() { /* marching.cpp:293-305 */
        poly_data.tri_list.clear(); poly_data.vertex_list.clear();
        reset_step_data();
    }

    bool set_grid_step_size(float v) { /* [0.001, 0.5], marching.cpp:226-238 */
        if (v >= 0.001 && v <= .5) {
            if (v != step_) { step_ = v; reset_step(); }
            return true;
        }
        return false;
    }
    bool set_grid_resolution(int n) { if (n < 2 || n > 4094) return false; step_ = 2.0f / (float)n; reset_step(); return true; }
    float get_grid_size() { return step_; }

    void step_by_step_mode(bool b) { step_mode_ = b; reset_step(); }
    void reset_step() { poly_data.step_data.step_i = -2; }
    void set_surface_constant(float c) { if (iso_ != c) { iso_ = c; reset_step(); } }

    void seed_mode(bool b) { seed_mode_ = b; reset_step(); }
    bool set_seed(float x, float y, float z) {
        if (x <= 1 && x >= -1 && y >= -1 && y <= 1 && z >= -1 && z <= 1) { seed_[0] = x; seed_[1] = y; seed_[2] = z; reset_step(); return true; }
        return false;
    }
    void get_seed(float* x, float* y, float* z) { *x = seed_[0]; *y = seed_[1]; *z = seed_[2]; }

    bool set_surface_repeat_step_distance(float l) { if (l <= 0) return false; repeat_step_ = l; reset_step(); return true; }
    bool repeating_surface_mode(bool b) { /* marching.cpp:164-170 */
        if (repeat_step_ < 0) return repeat_ = false;
        repeat_ = b; reset_step(); return true;
    }

    bool set_constraint0(std::string lhs, std::string op, float rhs) { return set_constraint(0, lhs, op, rhs); }
    bool set_constraint1(std::string lhs, std::string op, float rhs) { return set_constraint(1, lhs, op, rhs); }
    bool set_constraint2(std::string lhs, std::string op, float rhs) { return set_constraint(2, lhs, op, rhs); }
    bool set_constraint(int i, std::string lhs, std::string op, float rhs) { /* marching.cpp:173-200 (with the missing `return true`) */
        if (i < 0 || i > 2) return false;
        Comp_Op o;
        if (op == "<=") o = LE; else if (op == ">=") o = GE; else if (op == "<") o = LT; else if (op == ">") o = GT; else return false;
        if (!ensure_ctx()) return false;
        /* the left-hand side parses in the grammar of the evaluator set at this time (the reference's without one) */
        mcb_set_grammar(ctx_, evaluator_ ? evaluator_->grammar() : MCB_GRAMMAR_REFERENCE);
        if (mcb_set_equation(ctx_, i + 1, lhs.c_str()) != MCB_OK) return false;
        cons_valid_[i] = true; cons_op_[i] = o; cons_rhs_[i] = rhs;
        reset_step();
        return true;
    }
    bool use_constraint0(bool b) { return use_constraint(0, b); }
    bool use_constraint1(bool b) { return use_constraint(1, b); }
    bool use_constraint2(bool b) { return use_constraint(2, b); }
    bool use_constraint(int i, bool use) { if (i < 0 || i > 2) return false; reset_step(); return cons_use_[i] = use; } /* marching.cpp:202-207 */

    void set_scaling_x(float s) { sx_ = s; reset_step(); }
    void set_scaling_y(float s) { sy_ = s; reset_step(); }
    void set_scaling_z(float s) { sz_ = s; reset_step(); }

    /* ASCII PLY in the reference's format (marching.cpp:821-850: "element face %d " keeps its trailing blank, %f coordinates) */
    bool save_poly_to_file() {
        if (poly_data.vertex_list.empty()) return false;
        FILE* fp = std::fopen(mesh_file(), "w");
        if (!fp) return false;
        const int nv = (int)(poly_data.vertex_list.size() / 3), nt = (int)(poly_data.tri_list.size() / 3);
        std::fprintf(fp, "ply\nformat ascii 1.0\nelement vertex %d\nproperty float x\nproperty float y\nproperty float z\n", nv);
        std::fprintf(fp, "element face %d \nproperty list uchar int vertex_indices\nend_header\n", nt);
        for (int i = 0; i < nv; i++)
            std::fprintf(fp, "%f %f %f\n", poly_data.vertex_list[3 * i], poly_data.vertex_list[3 * i + 1], poly_data.vertex_list[3 * i + 2]);
        for (int i = 0; i < nt; i++)
            std::fprintf(fp, "%u %u %u %u\n", 3u, poly_data.tri_list[3 * i], poly_data.tri_list[3 * i + 1], poly_data.tri_list[3 * i + 2]);
        std::fclose(fp);
        return true;
    }
    bool load_poly_from_file() {
        unpin_all();
        reset_all_data();
        FILE* fp = std::fopen(mesh_file(), "r");
        if (!fp) return false;
        int nv = 0, nt = 0;
        char line[256];
        bool header_done = false;
        while (!header_done && std::fgets(line, sizeof line, fp)) {
            std::sscanf(line, "element vertex %d", &nv);
            std::sscanf(line, "element face %d", &nt);
            if (std::string(line).rfind("end_header", 0) == 0) header_done = true;
        }
        bool ok = header_done;
        for (int i = 0; ok && i < nv; i++) {
            float x, y, z;
            ok = std::fscanf(fp, "%f %f %f", &x, &y, &z) == 3;
            if (ok) { poly_data.vertex_list.push_back(x); poly_data.vertex_list.push_back(y); poly_data.vertex_list.push_back(z); }
        }
        for (int i = 0; ok && i < nt; i++) {
            unsigned n, a, b, c;
            ok = std::fscanf(fp, "%u %u %u %u", &n, &a, &b, &c) == 4 && n == 3;
            if (ok) { poly_data.tri_list.push_back(a); poly_data.tri_list.push_back(b); poly_data.tri_list.push_back(c); }
        }
        std::fclose(fp);
        return ok;
    }

    /* ---- extensions ---- */
    /* Several GPUs of one box: the grid is cut into z-slabs (SURVEY.md §8e), one mcb context and one host thread per
     * device 0..n-1.  The slabs' triangle counts are all-gathered over NCCL (mcb_comm_exchange) into global offsets; the
     * first recalculate() of a configuration also measures the triangles per layer and re-cuts the slabs to equal cost
     * (mcb_comm_balance, refined once by measured time: mcb_comm_rebalance).  Poly_Data is the slabs' welded meshes one after the other — triangles in the reference's order,
     * vertices on a plane shared by two slabs present once per slab.  Seed mode and step mode stay on device 0. */
    bool set_devices(int n) {
        if (n < 1 || n > 64) return false;
        if (n != devices_) { release_devices(); devices_ = n; }
        return true;
    }
    /* The kernels NVRTC compiles for a new equation are built on a background thread while recalculate() already
     * delivers meshes through the bytecode interpreter (same results): this blocks until they are in place (benchmarks). */
    bool wait_for_compiled_kernels() {
        bool ok = ctx_ && mcb_jit_wait(ctx_) >= 0;
        for (size_t r = 1; r < dev_ctx_.size(); r++) if (dev_ctx_[r]) ok = mcb_jit_wait(dev_ctx_[r]) >= 0 && ok;
        return ok;
    }
    void set_weld(bool b) { weld_ = b; }
    void set_normals(bool b) { normals_ = b; }
    /* true: get_vertex_normals() returns what CalculateNormal(get_poly_data()) would (normal.h:3-42), computed on the GPU,
     * bit for bit; false (default): central-difference gradient normals */
    void set_reference_normals(bool b) { reference_normals_ = b; }
    /* true: the equation's own gradient at every vertex, soup or welded (mcb_set_normals mode 3, DESIGN.md §12); takes
     * precedence over set_reference_normals.  false (default): as set_reference_normals says */
    void set_analytic_normals(bool b) { analytic_normals_ = b; }
    bool set_slab(int k_begin, int k_end) { slab_[0] = k_begin; slab_[1] = k_end; have_slab_ = true; return true; }
    const mcb_counts& last_counts() const { return counts_; }
    /* set_devices(n > 1): wall time of the phases of the last recalculate(), ms: the slabs' polygonisation (+ exchange),
     * sizing and page-locking Poly_Data, the copies from the devices, the index fix-up (inside the copy threads) */
    struct DeviceTiming { double polygonise = 0, prepare = 0, fetch = 0; };
    const DeviceTiming& last_device_timing() const { return dev_timing_; }
    /* set_weld(false): triangle soup of the last recalculate(), 3 float4 per triangle, (x,y,z,1) and (nx,ny,nz,0) */
    const std::vector<float>& get_soup() const { return soup_; }
    const std::vector<float>& get_normals() const { return normals_soup_; }
    /* set_weld(true), set_normals(true): gradient normal (x,y,z) of every vertex of Poly_Data::vertex_list */
    const std::vector<float>& get_vertex_normals() const { return vertex_normals_; }

private:
    void reset_step_data() {
        poly_data.step_data.intersect_coord.clear(); poly_data.step_data.tri_vlist.clear(); poly_data.step_data.edge_list.clear();
        seed_queue_.clear();
        vertex_set_.clear();
        reset_step();
    }
    /* a vector's storage, page-locked in place (mcb_host_register = cudaHostRegister) for as long as it stays where it is */
    struct Pinned { void* ptr = nullptr; size_t bytes = 0; };
    static void unpin(Pinned& p) { if (p.ptr) mcb_host_unregister(p.ptr); p.ptr = nullptr; p.bytes = 0; }
    void unpin_all() { unpin(pin_v_); unpin(pin_t_); unpin(pin_n_); }
    template <class T>
    static bool pin(Pinned& p, std::vector<T>& v) {
        void* ptr = v.data();
        const size_t bytes = v.capacity() * sizeof(T);
        if (p.ptr == ptr && p.bytes == bytes) return true;
        unpin(p);
        if (!ptr || !bytes || mcb_host_register(ptr, bytes) != MCB_OK) return false;
        p.ptr = ptr; p.bytes = bytes;
        return true;
    }
    bool ensure_ctx() {
        if (!ctx_) {
            const char* d = std::getenv("MCB_DEVICE");
            if (mcb_create(d ? std::atoi(d) : 0, &ctx_) != MCB_OK) { ctx_ = nullptr; return false; }
        }
        if (mcb_set_grid_step(ctx_, step_) < 0) return false;
        if (have_slab_ && mcb_set_slab(ctx_, slab_[0], slab_[1]) != MCB_OK) return false;
        return true;
    }
    int normals_mode() const { return normals_ ? (analytic_normals_ ? 3 : weld_ && reference_normals_ ? 2 : 1) : 0; }
    bool push_parameters() { return push_parameters(ctx_); }
    bool push_parameters(mcb_ctx* c) {
        mcb_set_grammar(c, evaluator_->grammar()); /* Evaluator::set_function_grammar */
        if (mcb_set_equation(c, 0, evaluator_->equation().c_str()) != MCB_OK) return false;
        mcb_set_surface_constant(c, iso_);
        mcb_set_scaling(c, sx_, sy_, sz_);
        mcb_set_normals(c, normals_mode());
        /* marching.cpp:156-170, 481-494.  The reference accepts the mode with its initial distance 0: every cube's iso is
         * then NaN and nothing is drawn; recalculate() short-cuts that case, the GPU only sees positive distances */
        mcb_set_repeat(c, repeat_ && repeat_step_ > 0.f ? 1 : 0, repeat_step_);
        mcb_set_field_mode(c, MCB_FIELD_AUTO); /* nothing here reads the field back: only the blocks around the surface are evaluated */
        for (int i = 0; i < 3; i++)
            mcb_set_constraint(c, i, cons_op_[i] == NAO ? 0 : (int)cons_op_[i], cons_rhs_[i], cons_valid_[i] && cons_use_[i]);
        return true;
    }

    /* ---- several GPUs: one context + one host thread per device ---- */
    void release_devices() {
        for (size_t r = 1; r < dev_ctx_.size(); r++) if (dev_ctx_[r]) mcb_destroy(dev_ctx_[r]);
        if (!dev_ctx_.empty() && dev_ctx_[0]) mcb_comm_finalize(dev_ctx_[0]);
        dev_ctx_.clear();
        comm_ready_ = false;
        balanced_key_.clear();
    }
    std::string configuration_key() const {
        char b[256];
        std::snprintf(b, sizeof b, "|%a|%a|%a|%a|%a|%d|%a", (double)step_, (double)iso_, (double)sx_, (double)sy_, (double)sz_, (int)repeat_, (double)repeat_step_);
        std::string k = evaluator_->equation() + b;
        for (int i = 0; i < 3; i++) { std::snprintf(b, sizeof b, "|%d%d%d%a", (int)cons_valid_[i], (int)cons_use_[i], (int)cons_op_[i], (double)cons_rhs_[i]); k += b; }
        return k;
    }
    bool recalculate_on_devices() {
        reset_step_data();
        if (!evaluator_) { poly_data.vertex_list.clear(); poly_data.tri_list.clear(); return true; }
        const int n = devices_;
        dev_ctx_.resize((size_t)n, nullptr);
        dev_ctx_[0] = ctx_; /* ensure_ctx() made it */
        char id[128];
        if (!comm_ready_ && mcb_comm_unique_id(id) != MCB_OK) return false; /* libnccl.so.2 is needed for more than one device */
        const std::string key = configuration_key();
        const bool rebalance = key != balanced_key_;
        std::vector<mcb_counts> cnt((size_t)n);
        std::vector<uint64_t> tri_off((size_t)n, 0);
        std::vector<int> ok((size_t)n, 1);
        auto per_device = [&](int r) {
            mcb_ctx*& c = dev_ctx_[(size_t)r];
            if (!c && mcb_create(r, &c) != MCB_OK) { c = nullptr; ok[(size_t)r] = 0; }
            /* every thread keeps going through the collectives below even after a local failure would deadlock the
             * others: creation failures are therefore checked before the first collective */
        };
        {
            std::vector<std::thread> th;
            for (int r = 1; r < n; r++) th.emplace_back(per_device, r);
            for (auto& t : th) t.join();
            for (int r = 0; r < n; r++) if (!ok[(size_t)r]) return false;
        }
        auto run = [&](int r) {
            mcb_ctx* c = dev_ctx_[(size_t)r];
            bool good = mcb_set_grid_step(c, step_) >= 0 && push_parameters(c);
            mcb_set_seed(c, 0, 0.f, 0.f, 0.f);
            mcb_set_mesh_mode(c, MCB_MESH_INDEXED);
            mcb_set_host_output(c, nullptr, nullptr, nullptr, 0, 0);
            if (!comm_ready_) good = mcb_comm_init(c, id, r, n) == MCB_OK && good;          /* collective; sets the uniform slab */
            else if (rebalance) { int k0, k1; good = mcb_slab_range(cnt_M(c), r, n, &k0, &k1) == MCB_OK && mcb_set_slab(c, k0, k1) == MCB_OK && good; }
            else good = mcb_set_slab(c, cuts_[(size_t)r], cuts_[(size_t)r + 1]) == MCB_OK && good;
            good = mcb_polygonise(c, &cnt[(size_t)r]) == MCB_OK && good;
            if (rebalance) { /* measured triangles per layer -> slabs of equal cost, then the real run */
                int k0 = 0, k1 = 0;
                good = mcb_comm_balance(c, -1.0, &k0, &k1) == MCB_OK && good;                   /* collective */
                good = mcb_polygonise(c, &cnt[(size_t)r]) == MCB_OK && good;
                /* one refinement by the measured device time of the balanced slabs (a failed run still takes part) */
                good = mcb_comm_rebalance(c, good && cnt[(size_t)r].ms_total > 0.f ? (double)cnt[(size_t)r].ms_total : 1.0, &k0, &k1) == MCB_OK && good;
                cuts_r_[(size_t)r] = k0; cuts_end_ = r == n - 1 ? k1 : cuts_end_;
                good = mcb_polygonise(c, &cnt[(size_t)r]) == MCB_OK && good;
            }
            good = mcb_comm_exchange(c) == MCB_OK && good;                                      /* collective: NCCL all-gather */
            good = mcb_comm_offsets(c, &tri_off[(size_t)r], nullptr, nullptr) == MCB_OK && good;
            ok[(size_t)r] = good ? 1 : 0;
        };
        cuts_r_.assign((size_t)n, 0);
        const auto tp0 = std::chrono::steady_clock::now();
        {
            std::vector<std::thread> th;
            for (int r = 1; r < n; r++) th.emplace_back(run, r);
            run(0);
            for (auto& t : th) t.join();
        }
        const auto tp1 = std::chrono::steady_clock::now();
        comm_ready_ = true;
        for (int r = 0; r < n; r++) if (!ok[(size_t)r]) return false;
        if (rebalance) {
            cuts_.assign(cuts_r_.begin(), cuts_r_.end());
            cuts_.push_back(cuts_end_);
            balanced_key_ = key;
        }
        /* Poly_Data: the slabs one after the other */
        std::vector<size_t> v_off((size_t)n + 1, 0);
        size_t T = 0;
        for (int r = 0; r < n; r++) { v_off[(size_t)r + 1] = v_off[(size_t)r] + (size_t)cnt[(size_t)r].vertices; T += (size_t)cnt[(size_t)r].triangles; }
        if (v_off[(size_t)n] * 3 > poly_data.vertex_list.capacity() || T * 3 > poly_data.tri_list.capacity() ||
            (normals_ && v_off[(size_t)n] * 3 > vertex_normals_.capacity()))
            unpin_all(); /* a vector is about to move: its old storage must not stay page-locked */
        poly_data.vertex_list.resize(v_off[(size_t)n] * 3);
        poly_data.tri_list.resize(T * 3);
        if (normals_) vertex_normals_.resize(v_off[(size_t)n] * 3); else vertex_normals_.clear();
        soup_.clear(); normals_soup_.clear();
        /* page-locked destinations: every device copies its part at full PCIe speed, all of them at once */
        pin(pin_v_, poly_data.vertex_list); pin(pin_t_, poly_data.tri_list);
        if (normals_) pin(pin_n_, vertex_normals_);
        const auto tp2 = std::chrono::steady_clock::now();
        auto fetch = [&](int r) {
            const mcb_counts& c = cnt[(size_t)r];
            if (!c.triangles) return;
            unsigned* tl = poly_data.tri_list.data() + 3 * (size_t)tri_off[(size_t)r];
            mcb_set_index_base(dev_ctx_[(size_t)r], (uint32_t)v_off[(size_t)r]); /* the slab's indices are shifted on the device */
            if (mcb_get_indexed_mesh(dev_ctx_[(size_t)r], poly_data.vertex_list.data() + 3 * v_off[(size_t)r], tl,
                                     normals_ ? vertex_normals_.data() + 3 * v_off[(size_t)r] : nullptr, c.vertices, c.triangles) != MCB_OK) { ok[(size_t)r] = 0; return; }
        };
        {
            std::vector<std::thread> th;
            for (int r = 1; r < n; r++) th.emplace_back(fetch, r);
            fetch(0);
            for (auto& t : th) t.join();
        }
        const auto tp3 = std::chrono::steady_clock::now();
        dev_timing_.polygonise = std::chrono::duration<double, std::milli>(tp1 - tp0).count();
        dev_timing_.prepare = std::chrono::duration<double, std::milli>(tp2 - tp1).count();
        dev_timing_.fetch = std::chrono::duration<double, std::milli>(tp3 - tp2).count();
        counts_ = cnt[0];
        for (int r = 1; r < n; r++) {
            counts_.cubes += cnt[(size_t)r].cubes; counts_.active += cnt[(size_t)r].active; counts_.triangles += cnt[(size_t)r].triangles;
            counts_.ambiguous += cnt[(size_t)r].ambiguous; counts_.redirected += cnt[(size_t)r].redirected; counts_.vertices += cnt[(size_t)r].vertices;
            if (cnt[(size_t)r].ms_total > counts_.ms_total) counts_.ms_total = cnt[(size_t)r].ms_total;
            counts_.k_end = cnt[(size_t)r].k_end;
        }
        poly_data.step_data.step_i = -1;
        for (int r = 0; r < n; r++) if (!ok[(size_t)r]) return false;
        return true;
    }
    int cnt_M(mcb_ctx*) const { return mcb_grid_axis(step_, nullptr, 0); }

    /* Step-by-step mode (marching.cpp:386-428): one cube per recalculate() call, in the reference's own traversal
     * (x fastest, coordinates carried over from the previous cube's corners, `< 1.0` bounds).  The cube itself is
     * computed on the GPU (mcb_inspect_cube = calculate_step); appending it to Poly_Data is the reference's
     * add_step_to_poly_data / add_point with its std::set — a handful of points per call, host side like the GUI. */
    bool step_once() {
        Step_Data& sd = poly_data.step_data;
        if (sd.step_i == 0) { add_step_to_poly_data(); sd.step_i = -1; return true; } /* last step */
        if (sd.step_i == -1) return false;                                                /* finished already */
        float x_0, y_0, z_0;
        if (sd.step_i == -2) { /* first step */
            reset_all_data();
            x_0 = y_0 = z_0 = -1;
            sd.step_i = 0;
            for (float x0 = -1.0; x0 < 1.0; x0 += step_) sd.step_i++;
            sd.step_i *= sd.step_i * sd.step_i;
            sd.step_i--;
        } else {
            x_0 = sd.corner_coords[3]; y_0 = sd.corner_coords[4]; z_0 = sd.corner_coords[5];
            if (x_0 >= 1.0) { x_0 = -1; y_0 += step_; }
            if (y_0 >= 1.0) { y_0 = -1; z_0 += step_; }
            sd.step_i--;
        }
        add_step_to_poly_data();
        return calculate_step(x_0, y_0, z_0);
    }
    bool calculate_step(float x_0, float y_0, float z_0) { /* marching.cpp:456-595, on the GPU */
        Step_Data& sd = poly_data.step_data;
        sd.intersect_coord.clear(); sd.tri_vlist.clear(); sd.edge_list.clear();
        if (!evaluator_ || !push_parameters()) return false;
        mcb_step_data o;
        if (mcb_inspect_cube(ctx_, x_0, y_0, z_0, &o) != MCB_OK) return false;
        sd.corner_coords.assign(o.corner_coords, o.corner_coords + 24);
        sd.corner_values.assign(o.corner_values, o.corner_values + 8);
        sd.edge_list.assign(o.edge_list, o.edge_list + o.n_edges);
        sd.intersect_coord.assign(o.intersect_coord, o.intersect_coord + 3 * o.n_edges);
        sd.tri_vlist.assign(o.tri_vlist, o.tri_vlist + o.n_tri_idx);
        if (repeat_) sd.surf_constant = o.surf_constant; /* marching.cpp:493: only written in repeating-surface mode */
        return true;
    }
    void add_step_to_poly_data() { /* marching.cpp:599-654 */
        const Step_Data& sd = poly_data.step_data;
        int v_i_list[12];
        for (int i = 0; i < 12; i++) v_i_list[i] = -1;
        for (size_t i = 0; i < sd.intersect_coord.size(); i += 3) {
            const float x = sd.intersect_coord[i], y = sd.intersect_coord[i + 1], z = sd.intersect_coord[i + 2];
            if (std::isnan(x)) continue;
            const int new_i = (int)(poly_data.vertex_list.size() / 3);
            const int found = vertex_set_.insert(xyz(x, y, z, new_i)).first->idx;
            if (found == new_i) { poly_data.vertex_list.push_back(x); poly_data.vertex_list.push_back(y); poly_data.vertex_list.push_back(z); }
            v_i_list[i / 3] = found;
        }
        for (size_t i = 0; i + 2 < sd.tri_vlist.size(); i += 3)
            for (int q = 0; q < 3; q++) poly_data.tri_list.push_back((unsigned)v_i_list[sd.tri_vlist[i + q]]);
    }

    void fill_poly_data_from_soup() { /* set_weld(false): every triangle corner is its own vertex */
        const size_t nv = soup_.size() / 4;
        poly_data.vertex_list.resize(nv * 3);
        poly_data.tri_list.resize(nv);
        for (size_t v = 0; v < nv; v++) {
            for (int a = 0; a < 3; a++) poly_data.vertex_list[3 * v + a] = soup_[4 * v + a];
            poly_data.tri_list[v] = (unsigned)v;
        }
    }
    static const char* mesh_file() { const char* f = std::getenv("MCB_MESH_FILE"); return f ? f : "mesh.ply"; }

    mcb_ctx* ctx_;
    Evaluator* evaluator_;
    float step_, iso_, sx_, sy_, sz_;
    bool weld_, normals_, seed_mode_, step_mode_, repeat_;
    bool reference_normals_ = false;
    bool analytic_normals_ = false;
    float repeat_step_;
    float seed_[3];
    bool cons_valid_[3], cons_use_[3];
    Comp_Op cons_op_[3];
    float cons_rhs_[3];
    int slab_[2] = {0, 0};
    bool have_slab_ = false;
    Poly_Data poly_data;
    std::deque<xyz> seed_queue_;
    std::set<xyz> vertex_set_; /* step-by-step mode only (marching.h:149) */
    std::vector<float> soup_, normals_soup_, vertex_normals_;
    Pinned pin_v_, pin_t_, pin_n_;
    DeviceTiming dev_timing_;
    int devices_ = 1;
    std::vector<mcb_ctx*> dev_ctx_;       /* [devices_]; [0] = ctx_ */
    bool comm_ready_ = false;
    std::string balanced_key_;            /* configuration the slab cuts below were measured for */
    std::vector<int> cuts_, cuts_r_;
    int cuts_end_ = 0;
    mcb_counts counts_;
};


