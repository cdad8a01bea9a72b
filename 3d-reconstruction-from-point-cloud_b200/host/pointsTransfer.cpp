// pointsTransfer -- command-line front end of the B200 detail-transfer path.
//
// Keeps the reference CLI's contract (/root/reference src/pointsTransfer.cpp:109-125, 587-625):
//   pointsTransfer <input-point-cloud> <input-mesh>
// * fewer than two arguments: prints the (sic) usage string to stdout and exits 0 (:112-120);
// * unreadable file: message on stderr, exit 0 (:137-141, :269-273);
// * ASCII PLY only; cloud rows `x y z nx ny nz r g b` (:204-250), mesh vertex rows
//   `x y z nx ny nz u v r g b` (:340-396), face rows `3 i j k` (:425-451); only the header tokens
//   `vertex N`, `face N`, `end_header` are interpreted (:160-170, :289-301);
// * the same stdout labels, so log scrapers keep working.
// What changes: the kd-tree build (:259) and the per-face-corner k-NN loop (:465-479) are
// replaced by one pt_index_build + one pt_transfer call over the unique mesh vertices (K = 20 as
// at :128), executed by the CUDA library through its C ABI.  The projection / Delaunay /
// rasteriser stages (:484-615) are out of scope of this build (SURVEY.md section 8 rows N1-N4):
// instead of texture.png the tool writes `transferred.ply`, the input mesh in the same 11-column
// ASCII format with the transferred colour and normal per vertex.  Extra options (all default to
// the reference's behaviour): -k N, -r RADIUS, -o FILE, -d DEVICE.  -b FILE / -n FILE also bake the
// cloud's colour / object-space normal onto every texel of the mesh's UV atlas (pt_texture_bake_height,
// same -R, -k, -r) and write them as PNG; -t FILE writes the tangent-space normal map as PNG and
// -T FILE the input mesh as PLY with the per-vertex tangents (tx ty tz tw) that map is expressed
// in, -H FILE the height map as a 16-bit greyscale PNG over the heights' own range (printed as
// "Height range: lo hi").  All of them come from one bake.  -e K first estimates the cloud's normals
// by PCA over each point's K nearest neighbours (pt_index_estimate_normals) and stores them in the
// index, so the transfer and the bake blend them: for scans whose nx ny nz columns are zero or noisy.
// -O K then orients the index's normals consistently along the minimum spanning forest of the
// K-NN graph (pt_index_orient_normals) and stores them: for normals whose signs are arbitrary.
#include <algorithm>
#include <charconv>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <iterator>
#include <string>
#include <thread>
#include <vector>

#include "points_transfer.h"
#include "pt_png.h"
#include "pt_point.h"

using ptb::Point;

namespace {

struct Timer {
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    double time() const
    {
        return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    }
    void reset() { t0 = std::chrono::steady_clock::now(); }
};

// whole-file tokenizer over spaces / tabs / newlines (the reference reads char by char, :149-252)
struct Tokens {
    std::string buf;
    size_t pos = 0;
    bool load(const std::string &path)
    {
        FILE *f = fopen(path.c_str(), "rb");
        if (!f) return false;
        fseek(f, 0, SEEK_END);
        long size = ftell(f);
        fseek(f, 0, SEEK_SET);
        buf.resize(size > 0 ? (size_t)size : 0);
        size_t got = size > 0 ? fread(&buf[0], 1, (size_t)size, f) : 0;
        fclose(f);
        buf.resize(got);
        return true;
    }
    bool next(const char *&b, const char *&e)
    {
        const size_t n = buf.size();
        while (pos < n && (buf[pos] == ' ' || buf[pos] == '\t' || buf[pos] == '\n' || buf[pos] == '\r')) ++pos;
        if (pos >= n) return false;
        size_t s = pos;
        while (pos < n && !(buf[pos] == ' ' || buf[pos] == '\t' || buf[pos] == '\n' || buf[pos] == '\r')) ++pos;
        b = buf.data() + s;
        e = buf.data() + pos;
        return true;
    }
    bool next_is(const char *b, const char *e, const char *word)
    {
        size_t len = strlen(word);
        return (size_t)(e - b) == len && memcmp(b, word, len) == 0;
    }
    bool next_double(double &v)
    {
        const char *b, *e;
        if (!next(b, e)) return false;
        v = strtod(std::string(b, e).c_str(), nullptr);   // atof semantics (:207 etc.)
        return true;
    }
};

struct Header { long vertex = -1, face = -1; };

bool read_header(Tokens &t, Header &h)
{
    const char *b, *e;
    while (t.next(b, e)) {
        if (t.next_is(b, e, "vertex")) { double v; if (!t.next_double(v)) return false; h.vertex = (long)v; }
        else if (t.next_is(b, e, "face")) { double v; if (!t.next_double(v)) return false; h.face = (long)v; }
        else if (t.next_is(b, e, "end_header")) return true;
    }
    return false;
}

bool read_rows(Tokens &t, long count, int columns, std::vector<Point> &out)
{
    out.reserve(count > 0 ? count : 0);
    std::vector<double> row(columns);
    for (long i = 0; i < count; ++i) {
        for (int c = 0; c < columns; ++c)
            if (!t.next_double(row[c])) return i > 0;   // truncated file: keep what was read
        Point p;
        p.ver[0] = row[0]; p.ver[1] = row[1]; p.ver[2] = row[2];
        p.normal[0] = row[3]; p.normal[1] = row[4]; p.normal[2] = row[5];
        int c0 = 6;
        if (columns == 11) { p.U = row[6]; p.V = row[7]; c0 = 8; }
        p.color[0] = (int)row[c0]; p.color[1] = (int)row[c0 + 1]; p.color[2] = (int)row[c0 + 2];
        out.push_back(p);
    }
    return true;
}

// ---- fast path (SURVEY.md section 8 row N2): line-parallel body parser ---------------------------
// Standard ASCII PLY puts one element per line.  The body is cut into byte ranges at line
// boundaries, every thread counts its non-empty lines, a prefix sum gives each thread its first
// record number, then the threads parse their lines straight into the output arrays with
// std::from_chars (correctly rounded, i.e. the same doubles atof produces at :207 etc.).
// Returns false (caller falls back to the sequential token parser, which accepts any
// whitespace layout like the reference does) if the file is not one-record-per-line.
inline const char *skip_ws(const char *p, const char *e)
{
    while (p < e && (*p == ' ' || *p == '\t' || *p == '\r')) ++p;
    return p;
}

inline bool parse_num(const char *&p, const char *e, double &v)
{
    p = skip_ws(p, e);
    if (p < e && *p == '+') ++p;          // from_chars rejects a leading '+', atof accepts it
    auto r = std::from_chars(p, e, v);
    if (r.ec != std::errc()) return false;
    p = r.ptr;
    return true;
}

bool parse_body_parallel(const std::string &buf, size_t body, long n_vertex, int columns, long n_face,
                         std::vector<Point> &vertices, std::vector<int> *faces)
{
    const char *b = buf.data() + body, *e = buf.data() + buf.size();
    const long want = n_vertex + (faces ? n_face : 0);
    if (n_vertex < 0 || want <= 0) return false;
    unsigned nt = std::max(1u, std::min(std::thread::hardware_concurrency(), 64u));
    if ((size_t)(e - b) < (size_t)nt * 65536) nt = 1;
    std::vector<const char *> lo(nt + 1);
    for (unsigned t = 0; t <= nt; ++t) {
        const char *p = b + (size_t)(e - b) * t / nt;
        if (t > 0 && t < nt) {               // advance to the start of the next line
            while (p < e && p[-1] != '\n') ++p;
        }
        lo[t] = t == nt ? e : p;
    }
    auto non_empty = [](const char *p, const char *q) {
        for (; p < q; ++p) if (*p != ' ' && *p != '\t' && *p != '\r') return true;
        return false;
    };
    std::vector<long> first(nt + 1, 0);
    {
        std::vector<std::thread> th;
        for (unsigned t = 0; t < nt; ++t)
            th.emplace_back([&, t] {
                long c = 0;
                for (const char *p = lo[t]; p < lo[t + 1];) {
                    const char *nl = (const char *)memchr(p, '\n', lo[t + 1] - p);
                    const char *q = nl ? nl : lo[t + 1];
                    if (non_empty(p, q)) ++c;
                    p = q + 1;
                }
                first[t + 1] = c;
            });
        for (auto &x : th) x.join();
    }
    for (unsigned t = 0; t < nt; ++t) first[t + 1] += first[t];
    if (first[nt] < want) return false;       // fewer lines than records: not line-structured
    vertices.assign((size_t)n_vertex, Point());
    if (faces) faces->assign((size_t)n_face * 3, 0);
    std::vector<char> ok(nt, 1);
    {
        std::vector<std::thread> th;
        for (unsigned t = 0; t < nt; ++t)
            th.emplace_back([&, t] {
                long rec = first[t];
                for (const char *p = lo[t]; p < lo[t + 1] && rec < want;) {
                    const char *nl = (const char *)memchr(p, '\n', lo[t + 1] - p);
                    const char *q = nl ? nl : lo[t + 1];
                    if (non_empty(p, q)) {
                        const char *c = p;
                        double row[11];
                        if (rec < n_vertex) {
                            for (int k = 0; k < columns; ++k)
                                if (!parse_num(c, q, row[k])) { ok[t] = 0; return; }
                            Point &v = vertices[(size_t)rec];
                            v.ver[0] = row[0]; v.ver[1] = row[1]; v.ver[2] = row[2];
                            v.normal[0] = row[3]; v.normal[1] = row[4]; v.normal[2] = row[5];
                            int c0 = 6;
                            if (columns == 11) { v.U = row[6]; v.V = row[7]; c0 = 8; }
                            v.color[0] = (int)row[c0]; v.color[1] = (int)row[c0 + 1]; v.color[2] = (int)row[c0 + 2];
                        } else {
                            for (int k = 0; k < 4; ++k)
                                if (!parse_num(c, q, row[k])) { ok[t] = 0; return; }
                            int *f = faces->data() + 3 * (size_t)(rec - n_vertex);
                            f[0] = (int)row[1]; f[1] = (int)row[2]; f[2] = (int)row[3];
                        }
                        ++rec;
                    }
                    p = q + 1;
                }
            });
        for (auto &x : th) x.join();
    }
    for (char c : ok) if (!c) return false;
    return true;
}

void memory_report()
{
    long virt = 0, res = 0;
    if (FILE *f = fopen("/proc/self/statm", "r")) {
        if (fscanf(f, "%ld %ld", &virt, &res) != 2) virt = res = 0;
        fclose(f);
    }
    const long page = 4096;
    std::cout << "VIRT: " << ((virt * page) >> 20) << " MiB" << std::endl;
    std::cout << "RES:  " << ((res * page) >> 20) << " MiB" << std::endl;
}

}  // namespace

static int run(int argc, char **argv)
{
    std::string usage_str = "Usage: ./pointTransfer <input-point-cloud> <input-mesh>";
    std::vector<std::string> pos_args;
    int K = 20;             // src/pointsTransfer.cpp:128
    double radius = -1.0;   // unbounded, as the reference
    int device = -1;
    int n_gpus = 1;         // -g N: the cloud sharded into N x-slabs (pt_sharded_*), slab r on GPU r mod #GPUs
    int resolution = 8192;  // src/pointsTransfer.cpp:129
    std::string out_name = "texture.png";          // src/pointsTransfer.cpp:613
    std::string ply_name;                          // optional extra: the per-vertex blend as a PLY
    std::string bake_name, normal_name;            // optional extras: the per-texel colour / normal maps
    std::string tangent_name, tangent_ply_name;    // ... the tangent-space normal map, the mesh with tangents
    std::string height_name;                       // ... the height map
    bool estimate = false;                         // -e K: estimate the cloud's normals first
    int estimate_k = 0;
    bool orient = false;                           // -O K: orient the cloud's normals (after -e)
    int orient_k = 0;
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        if (a == "-k" && i + 1 < argc) K = atoi(argv[++i]);
        else if (a == "-r" && i + 1 < argc) radius = atof(argv[++i]);
        else if (a == "-o" && i + 1 < argc) out_name = argv[++i];
        else if (a == "-p" && i + 1 < argc) ply_name = argv[++i];
        else if (a == "-R" && i + 1 < argc) resolution = atoi(argv[++i]);
        else if (a == "-d" && i + 1 < argc) device = atoi(argv[++i]);
        else if (a == "-g" && i + 1 < argc) n_gpus = atoi(argv[++i]);
        else if (a == "-b" && i + 1 < argc) bake_name = argv[++i];
        else if (a == "-n" && i + 1 < argc) normal_name = argv[++i];
        else if (a == "-t" && i + 1 < argc) tangent_name = argv[++i];
        else if (a == "-T" && i + 1 < argc) tangent_ply_name = argv[++i];
        else if (a == "-H" && i + 1 < argc) height_name = argv[++i];
        else if (a == "-e" && i + 1 < argc) { estimate = true; estimate_k = atoi(argv[++i]); }
        else if (a == "-O" && i + 1 < argc) { orient = true; orient_k = atoi(argv[++i]); }
        else pos_args.push_back(a);
    }
    if (pos_args.size() < 2) {
        std::cout << usage_str << std::endl;
        return 0;
    }
    if (K < 1 || K > PT_MAX_K || resolution < 1 || resolution > 32768 || n_gpus < 1 || n_gpus > 64) {
        // like every error path of the reference: a message, exit code 0
        std::cerr << "-k must be 1.." << PT_MAX_K << ", -R 1..32768 and -g 1..64" << std::endl;
        return 0;
    }
    if (estimate && (estimate_k < 3 || estimate_k > PT_MAX_K || n_gpus > 1)) {
        std::cerr << "-e must be 3.." << PT_MAX_K << " and estimates normals on one GPU (no -g)" << std::endl;
        return 0;
    }
    if (orient && (orient_k < 2 || orient_k > PT_MAX_K || n_gpus > 1)) {
        std::cerr << "-O must be 2.." << PT_MAX_K << " and orients normals on one GPU (no -g)" << std::endl;
        return 0;
    }
    const bool bake = !bake_name.empty() || !normal_name.empty() || !tangent_name.empty() || !tangent_ply_name.empty() ||
                      !height_name.empty();
    if (bake && (n_gpus > 1 || resolution > 16384)) {
        std::cerr << "-b / -n / -t / -T / -H bake on one GPU (no -g) at -R 1..16384" << std::endl;
        return 0;
    }
    const std::string pc_file_name = pos_args[0], mesh_file_name = pos_args[1];

    Timer task_timer, real_total_timer;

    Tokens pc;
    if (!pc.load(pc_file_name)) {
        std::cerr << "Cannot read or find point cloud file: " << pc_file_name << std::endl;
        return 0;
    }
    Header ph;
    read_header(pc, ph);
    std::cout << "PC Point count: " << ph.vertex << std::endl;
    std::vector<Point> points;
    if (!parse_body_parallel(pc.buf, pc.pos, ph.vertex, 9, 0, points, nullptr)) {
        points.clear();
        read_rows(pc, ph.vertex, 9, points);      // any-whitespace layout, like the reference
    }
    std::cout << "Read point set in: " << task_timer.time() << " seconds" << std::endl;
    task_timer.reset();

    pt_index *index = nullptr;
    pt_sharded *sharded = nullptr;
    int rc;
    if (n_gpus > 1) {
        pt_sharded_opts so;
        memset(&so, 0, sizeof so);
        so.n_devices = n_gpus;
        so.k_hint = K;
        so.coord_mode = PT_COORD_AUTO;
        rc = pt_sharded_build(points.data(), points.size(), &so, &sharded);
    } else {
        pt_build_opts opts;
        memset(&opts, 0, sizeof opts);
        opts.device = device;
        opts.coord_mode = PT_COORD_AUTO;
        rc = pt_index_build(points.data(), points.size(), &opts, &index);
    }
    if (rc != PT_OK) {
        std::cerr << "index build failed: " << pt_status_string(rc) << std::endl;
        return 0;
    }
    std::cout << "Built Kd tree in: " << task_timer.time() << " seconds" << std::endl;
    task_timer.reset();
    if (estimate) {
        pt_normals_stats ns;
        rc = pt_index_estimate_normals(index, estimate_k, radius, nullptr, 1, nullptr, nullptr, &ns);
        if (rc != PT_OK) {
            std::cerr << "pt_index_estimate_normals failed: " << pt_status_string(rc) << std::endl;
            pt_index_free(index);
            return 0;
        }
        std::cout << "Estimated normals: " << ns.estimated << " of " << points.size() << " points in "
                  << task_timer.time() << " seconds" << std::endl;
        task_timer.reset();
    }
    if (orient) {
        pt_orient_stats os;
        rc = pt_index_orient_normals(index, orient_k, radius, nullptr, 1, nullptr, nullptr, &os);
        if (rc != PT_OK) {
            std::cerr << "pt_index_orient_normals failed: " << pt_status_string(rc) << std::endl;
            pt_index_free(index);
            return 0;
        }
        std::cout << "Oriented normals: " << os.oriented << " of " << points.size() << " points, " << os.flipped
                  << " flipped, " << os.components << " components in " << task_timer.time() << " seconds" << std::endl;
        task_timer.reset();
    }

    Tokens mesh;
    if (!mesh.load(mesh_file_name)) {
        std::cerr << "Cannot read or find mesh file: " << mesh_file_name << std::endl;
        pt_index_free(index);
        pt_sharded_free(sharded);
        return 0;
    }
    Header mh;
    read_header(mesh, mh);
    std::cout << "Mesh vertex count: " << mh.vertex << std::endl;
    std::cout << "Mesh face count: " << mh.face << std::endl;
    std::vector<Point> vertices;
    std::vector<int> faces;   // heap, not the reference's stack VLA (:406)
    if (!parse_body_parallel(mesh.buf, mesh.pos, mh.vertex, 11, mh.face < 0 ? 0 : mh.face, vertices, &faces)) {
        vertices.clear();
        faces.clear();
        read_rows(mesh, mh.vertex, 11, vertices);
        faces.reserve(mh.face > 0 ? 3 * mh.face : 0);
        for (long f = 0; f < mh.face; ++f) {
            double cnt, a, b, c;
            if (!mesh.next_double(cnt) || !mesh.next_double(a) || !mesh.next_double(b) || !mesh.next_double(c)) break;
            faces.push_back((int)a); faces.push_back((int)b); faces.push_back((int)c);
        }
    }
    std::cout << "Read mesh faces: " << task_timer.time() << " seconds" << std::endl;
    task_timer.reset();

    // The face loop (:462-585) and the texture post-process (:593-611) in one call: ONE batched
    // search over the unique vertices replaces the 3*F per-corner searches (:465-479), then the
    // per-face projection / Delaunay / rasterisation kernels and the dilate + gutter.
    const size_t m = vertices.size();
    std::vector<uint8_t> texture((size_t)resolution * resolution * 4);
    pt_texture_stats ts;
    memset(&ts, 0, sizeof ts);
    if (sharded) {
        // sharded search (one host thread and one index per slab), then the face / texture stage on
        // one GPU from the lists
        std::vector<int32_t> nn(m * (size_t)K);
        Timer knn_timer;
        rc = pt_sharded_knn(sharded, vertices.data(), m, K, radius, nn.data(), nullptr);
        const double knn_s = knn_timer.time();
        if (rc == PT_OK)
            rc = pt_texture_render_lists(points.data(), points.size(), vertices.data(), m, faces.data(), faces.size() / 3,
                                         nn.data(), K, resolution, 1, device, texture.data(), &ts);
        ts.knn_ms = (float)(knn_s * 1e3);
    } else {
        rc = pt_texture_render(index, vertices.data(), m, faces.data(), faces.size() / 3, K, radius, resolution, 1,
                               texture.data(), &ts);
    }
    if (rc != PT_OK) {
        std::cerr << "pt_texture_render failed: " << pt_status_string(rc) << std::endl;
        pt_index_free(index);
        pt_sharded_free(sharded);
        return 0;
    }
    task_timer.reset();
    std::cout << "Neighbor search total time: " << ts.knn_ms * 1e-3 << " seconds" << std::endl;
    std::cout << "Draw triangles total time: " << (ts.draw_ms + ts.pad_ms) * 1e-3 << " seconds" << std::endl;

    // extra (not in the reference): per-texel colour, normal and tangent-space normal maps and the
    // 16-bit height map, padded like the texture, and the per-vertex tangents
    std::vector<uint8_t> baked, baked_normal, baked_tangent;
    std::vector<float> vertex_tangents;
    std::vector<uint16_t> baked_height;
    if (bake) {
        const size_t n_bytes = (size_t)resolution * resolution * 4;
        if (!bake_name.empty()) baked.resize(n_bytes);
        if (!normal_name.empty()) baked_normal.resize(n_bytes);
        if (!tangent_name.empty()) baked_tangent.resize(n_bytes);
        if (!tangent_ply_name.empty()) vertex_tangents.resize(4 * m);
        pt_bake_outputs bo;
        memset(&bo, 0, sizeof bo);
        bo.bgra = baked.empty() ? nullptr : baked.data();
        bo.normal_bgra = baked_normal.empty() ? nullptr : baked_normal.data();
        bo.tangent_bgra = baked_tangent.empty() ? nullptr : baked_tangent.data();
        bo.vertex_tangents = tangent_ply_name.empty() ? nullptr : vertex_tangents.data();
        pt_bake_height hb;
        memset(&hb, 0, sizeof hb);                 // range (0, 0): the heights' own min and max
        if (!height_name.empty()) {
            baked_height.resize((size_t)resolution * resolution);
            hb.height_u16 = baked_height.data();
        }
        pt_bake_stats bs;
        rc = pt_texture_bake_height(index, vertices.data(), m, faces.data(), faces.size() / 3, K, radius, resolution, 1,
                                    &bo, height_name.empty() ? nullptr : &hb, &bs);
        if (rc != PT_OK) {
            std::cerr << "pt_texture_bake_height failed: " << pt_status_string(rc) << std::endl;
            pt_index_free(index);
            return 0;
        }
        if (!height_name.empty()) {
            char line[96];
            snprintf(line, sizeof line, "Height range: %.9g %.9g", hb.range_used[0], hb.range_used[1]);
            std::cout << line << std::endl;
        }
        std::cout << "Bake total time: " << task_timer.time() << " seconds" << std::endl;
        task_timer.reset();
    }

    if (!ptb::write_png_bgra(out_name.c_str(), texture.data(), resolution, resolution))
        std::cerr << "Cannot write " << out_name << std::endl;
    if (!baked.empty() && !ptb::write_png_bgra(bake_name.c_str(), baked.data(), resolution, resolution))
        std::cerr << "Cannot write " << bake_name << std::endl;
    if (!baked_normal.empty() && !ptb::write_png_bgra(normal_name.c_str(), baked_normal.data(), resolution, resolution))
        std::cerr << "Cannot write " << normal_name << std::endl;
    if (!baked_tangent.empty() && !ptb::write_png_bgra(tangent_name.c_str(), baked_tangent.data(), resolution, resolution))
        std::cerr << "Cannot write " << tangent_name << std::endl;
    if (!baked_height.empty() && !ptb::write_png_gray16(height_name.c_str(), baked_height.data(), resolution, resolution))
        std::cerr << "Cannot write " << height_name << std::endl;
    if (!tangent_ply_name.empty()) {
        // the input mesh with the tangent frame of the tangent-space map: tx ty tz tw per vertex
        // (%.9g round-trips the fp32 values)
        std::ofstream out(tangent_ply_name);
        out << "ply\nformat ascii 1.0\nelement vertex " << m << "\n"
            << "property double x\nproperty double y\nproperty double z\n"
            << "property double nx\nproperty double ny\nproperty double nz\n"
            << "property double s\nproperty double t\n"
            << "property uchar red\nproperty uchar green\nproperty uchar blue\n"
            << "property float tx\nproperty float ty\nproperty float tz\nproperty float tw\n"
            << "element face " << faces.size() / 3 << "\nproperty list uchar int vertex_indices\nend_header\n";
        char line[640];
        for (size_t i = 0; i < m; ++i) {
            const Point &v = vertices[i];
            const float *t = vertex_tangents.data() + 4 * i;
            snprintf(line, sizeof line, "%.17g %.17g %.17g %.17g %.17g %.17g %.17g %.17g %d %d %d %.9g %.9g %.9g %.9g\n",
                     v.ver[0], v.ver[1], v.ver[2], v.normal[0], v.normal[1], v.normal[2], v.U, v.V, v.color[0],
                     v.color[1], v.color[2], t[0], t[1], t[2], t[3]);
            out << line;
        }
        for (size_t f = 0; f + 2 < faces.size(); f += 3)
            out << "3 " << faces[f] << ' ' << faces[f + 1] << ' ' << faces[f + 2] << '\n';
        if (!out) std::cerr << "Cannot write " << tangent_ply_name << std::endl;
    }
    if (!ply_name.empty()) {
        // extra (not in the reference): the fused per-vertex colour / normal blend of pt_transfer
        std::vector<uint8_t> rgba(m * 4);
        std::vector<float> normal(m * 3);
        rc = sharded ? pt_sharded_transfer(sharded, vertices.data(), m, K, radius, nullptr, nullptr, rgba.data(), normal.data())
                     : pt_transfer(index, vertices.data(), m, K, radius, nullptr, nullptr, rgba.data(), normal.data());
        if (rc != PT_OK) {
            std::cerr << "pt_transfer failed: " << pt_status_string(rc) << std::endl;
            pt_index_free(index);
            pt_sharded_free(sharded);
            return 0;
        }
        std::ofstream out(ply_name);
        out << "ply\nformat ascii 1.0\nelement vertex " << m << "\n"
            << "property float x\nproperty float y\nproperty float z\n"
            << "property float nx\nproperty float ny\nproperty float nz\n"
            << "property float s\nproperty float t\n"
            << "property uchar red\nproperty uchar green\nproperty uchar blue\n"
            << "element face " << faces.size() / 3 << "\nproperty list uchar int vertex_indices\nend_header\n";
        char line[512];
        for (size_t i = 0; i < m; ++i) {
            const Point &v = vertices[i];
            snprintf(line, sizeof line, "%.17g %.17g %.17g %.9g %.9g %.9g %.17g %.17g %d %d %d\n", v.ver[0],
                     v.ver[1], v.ver[2], normal[3 * i], normal[3 * i + 1], normal[3 * i + 2], v.U, v.V,
                     (int)rgba[4 * i], (int)rgba[4 * i + 1], (int)rgba[4 * i + 2]);
            out << line;
        }
        for (size_t f = 0; f + 2 < faces.size(); f += 3)
            out << "3 " << faces[f] << ' ' << faces[f + 1] << ' ' << faces[f + 2] << '\n';
    }
    std::cout << "Output time: " << task_timer.time() << " seconds" << std::endl;
    std::cout << "Total real time: " << real_total_timer.time() << " seconds" << std::endl;
    memory_report();
    pt_index_free(index);
    pt_sharded_free(sharded);
    return 0;
}

int main(int argc, char **argv)
{
    // like every error path of the reference: a message, exit code 0 (a header announcing more
    // records than memory holds ends here instead of in std::terminate)
    try {
        return run(argc, argv);
    } catch (const std::exception &e) {
        std::cerr << "pointsTransfer: " << e.what() << std::endl;
    } catch (...) {
        std::cerr << "pointsTransfer: unexpected error" << std::endl;
    }
    return 0;
}
