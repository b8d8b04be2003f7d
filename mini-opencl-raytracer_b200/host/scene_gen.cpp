// scene_gen.cpp -- seeded synthetic scenes of the shapes BASELINE.json names, written as OBJ + MTL text in
// the dialect CLOBJloader accepts (v/vt/vn triplets, sibling .mtl, `usemtl`), so that they enter the system
// through the same loader + BVH builder as cornell.obj:
//   * displaced geodesic icosphere: 20*f^2 faces (f = 224 -> 1 003 520 faces -> 2 007 040 CLTriangle after
//     the loader's duplication), radius R, smooth seeded radial displacement, analytic smooth normals;
//   * scattered triangles: n small randomly oriented triangles with centres uniform in a cube.
// Generated on the machine that uses them (a 1 M-face OBJ is ~110 MB of text); never committed.
#include <charconv>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <map>
#include <string>
#include <vector>

namespace
{
    struct Rng   // splitmix64: identical streams on every platform
    {
        uint64_t s;
        explicit Rng(uint64_t seed) : s(seed) {}
        uint64_t next() { uint64_t z = (s += 0x9e3779b97f4a7c15ull); z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull; z = (z ^ (z >> 27)) * 0x94d049bb133111ebull; return z ^ (z >> 31); }
        double uniform() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }
        double normal() { double u = uniform(), v = uniform(); if (u < 1e-300) u = 1e-300; return std::sqrt(-2.0 * std::log(u)) * std::cos(6.283185307179586 * v); }
    };
    struct D3 { double x, y, z; };
    inline D3 operator+(D3 a, D3 b) { return { a.x + b.x, a.y + b.y, a.z + b.z }; }
    inline D3 operator-(D3 a, D3 b) { return { a.x - b.x, a.y - b.y, a.z - b.z }; }
    inline D3 operator*(D3 a, double s) { return { a.x * s, a.y * s, a.z * s }; }
    inline double dot(D3 a, D3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
    inline D3 cross(D3 a, D3 b) { return { a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x }; }
    inline D3 unit(D3 a) { double l = std::sqrt(dot(a, a)); return a * (1.0 / l); }

    struct Writer
    {
        FILE* f;
        std::vector<char> buf;
        explicit Writer(FILE* file) : f(file) { buf.reserve(1 << 22); }
        void put(const char* s, int n) { buf.insert(buf.end(), s, s + n); if (buf.size() > (1u << 22) - 512) flush(); }
        void flush() { if (!buf.empty()) std::fwrite(buf.data(), 1, buf.size(), f); buf.clear(); }
        // Numbers are printed with std::to_chars: the shortest decimal that reads back as the same float (strtof / scanf
        // "%f"), an order of magnitude faster than printf("%.9g") -- a 10 M-face scene is 50 M lines.
        char* num(char* p, float v) { return std::to_chars(p, p + 32, v).ptr; }
        char* num(char* p, long long v) { return std::to_chars(p, p + 24, v).ptr; }
        void v3(const char* tag, D3 p)
        {
            char line[128], *q = line;
            while (*tag) *q++ = *tag++;
            *q++ = ' '; q = num(q, (float)p.x); *q++ = ' '; q = num(q, (float)p.y); *q++ = ' '; q = num(q, (float)p.z); *q++ = '\n';
            put(line, (int)(q - line));
        }
        void faceN(long long a, long long b, long long c, long long na, long long nb, long long nc)
        {
            char line[192], *q = line;
            *q++ = 'f';
            const long long v[3] = { a, b, c }, n[3] = { na, nb, nc };
            for (int k = 0; k < 3; ++k) { *q++ = ' '; q = num(q, v[k]); *q++ = '/'; *q++ = (char)('1' + k); *q++ = '/'; q = num(q, n[k]); }
            *q++ = '\n';
            put(line, (int)(q - line));
        }
        void face(long a, long b, long c) { faceN(a, b, c, a, b, c); }
        void faceN(long long a, long long b, long long c, long long nrm) { faceN(a, b, c, nrm, nrm, nrm); }
        void text(const std::string& s) { put(s.data(), (int)s.size()); }
    };

    bool writeMtl(const std::string& objPath)
    {
        std::string p = objPath.substr(0, objPath.size() - 4) + ".mtl";
        FILE* f = std::fopen(p.c_str(), "w");
        if (!f) return false;
        std::fputs("newmtl surface\nNs 9999.0\nKd 0.7 0.7 0.7\nKs 0 0 0\nKe 0 0 0\nNi 1.0\n"
                   "newmtl lamp\nNs 9999.0\nKd 0.8 0.8 0.8\nKs 0 0 0\nKe 1 1 1\nNi 1.0\n", f);
        std::fclose(f);
        return true;
    }
    std::string mtllibLine(const std::string& objPath)
    {
        size_t slash = objPath.find_last_of('/');
        std::string base = objPath.substr(slash == std::string::npos ? 0 : slash + 1);
        return "mtllib " + base.substr(0, base.size() - 4) + ".mtl\n";
    }
}

namespace
{
    // Geodesic icosphere of frequency f: unit directions of the 10 f^2 + 2 vertices and the 20 f^2 faces (0-based vertex
    // ids, counter-clockwise seen from outside). The topology is shared by every sphere a scene contains.
    struct Geodesic { std::vector<D3> dir; std::vector<long> faces; };

    void buildGeodesic(int f, Geodesic& g)
    {
        const double t = (1.0 + std::sqrt(5.0)) / 2.0;
        const D3 corner[12] = { unit({ -1, t, 0 }), unit({ 1, t, 0 }), unit({ -1, -t, 0 }), unit({ 1, -t, 0 }), unit({ 0, -1, t }), unit({ 0, 1, t }),
                                unit({ 0, -1, -t }), unit({ 0, 1, -t }), unit({ t, 0, -1 }), unit({ t, 0, 1 }), unit({ -t, 0, -1 }), unit({ -t, 0, 1 }) };
        const int faces[20][3] = { { 0, 11, 5 }, { 0, 5, 1 }, { 0, 1, 7 }, { 0, 7, 10 }, { 0, 10, 11 }, { 1, 5, 9 }, { 5, 11, 4 }, { 11, 10, 2 }, { 10, 7, 6 }, { 7, 1, 8 },
                                   { 3, 9, 4 }, { 3, 4, 2 }, { 3, 2, 6 }, { 3, 6, 8 }, { 3, 8, 9 }, { 4, 9, 5 }, { 2, 4, 11 }, { 6, 2, 10 }, { 8, 6, 7 }, { 9, 8, 1 } };
        std::map<std::pair<int, int>, int> edgeIndex;
        for (auto& fc : faces)
            for (int e = 0; e < 3; ++e)
            {
                int a = fc[e], b = fc[(e + 1) % 3];
                std::pair<int, int> key(a < b ? a : b, a < b ? b : a);
                if (!edgeIndex.count(key)) { int idx = (int)edgeIndex.size(); edgeIndex[key] = idx; }
            }
        const long perEdge = f - 1, perFace = (long)(f - 1) * (f - 2) / 2;
        const long nVerts = 12 + 30 * perEdge + 20 * perFace;
        g.dir.assign((size_t)nVerts, D3{ 0, 0, 0 });
        for (int c = 0; c < 12; ++c) g.dir[c] = corner[c];
        for (auto& kv : edgeIndex)
            for (int s = 1; s < f; ++s)
                g.dir[12 + (long)kv.second * perEdge + (s - 1)] = unit(corner[kv.first.first] * (double)(f - s) + corner[kv.first.second] * (double)s);
        // vertex id of barycentric (i,j,k) on face fi: i weighs corner A, j corner B, k corner C
        auto vid = [&](int fi, int i, int j, int k) -> long {
            const int A = faces[fi][0], B = faces[fi][1], C = faces[fi][2];
            if (i == f) return A;
            if (j == f) return B;
            if (k == f) return C;
            auto onEdge = [&](int a, int b, int towardsB) -> long {   // towardsB = weight of corner b
                std::pair<int, int> key(a < b ? a : b, a < b ? b : a);
                int s = a < b ? towardsB : f - towardsB;
                return 12 + (long)edgeIndex[key] * perEdge + (s - 1);
            };
            if (k == 0) return onEdge(A, B, j);
            if (i == 0) return onEdge(B, C, k);
            if (j == 0) return onEdge(C, A, i);
            long row = 0;                                             // interior: rows by j = 1..f-2, within a row k = 1..f-1-j
            for (int jj = 1; jj < j; ++jj) row += f - 1 - jj;
            return 12 + 30 * perEdge + (long)fi * perFace + row + (k - 1);
        };
        for (int fi = 0; fi < 20; ++fi)
            for (int j = 1; j <= f - 2; ++j)
                for (int k = 1; k <= f - 1 - j; ++k)
                {
                    int i = f - j - k;
                    g.dir[vid(fi, i, j, k)] = unit(corner[faces[fi][0]] * (double)i + corner[faces[fi][1]] * (double)j + corner[faces[fi][2]] * (double)k);
                }
        g.faces.clear();
        g.faces.reserve((size_t)60 * f * f);
        for (int fi = 0; fi < 20; ++fi)
            for (int j = 0; j < f; ++j)
                for (int k = 0; k < f - j; ++k)
                {
                    int i = f - j - k;   // i >= 1
                    // upright triangle (i,j,k) (i-1,j+1,k) (i-1,j,k+1): counter-clockwise seen from outside like (A,B,C)
                    g.faces.insert(g.faces.end(), { vid(fi, i, j, k), vid(fi, i - 1, j + 1, k), vid(fi, i - 1, j, k + 1) });
                    if (i >= 2)   // inverted triangle sharing the edge (i-1,j+1,k)-(i-1,j,k+1)
                        g.faces.insert(g.faces.end(), { vid(fi, i - 1, j + 1, k), vid(fi, i - 2, j + 1, k + 1), vid(fi, i - 1, j, k + 1) });
                }
    }

    // Radial displacement field r(d) = R * (1 + amplitude/3 * sum_k sin(w_k . d + phi_k)) with its analytic normal.
    struct Bumps
    {
        D3 wave[6];
        double phase[6];
        explicit Bumps(Rng& rng) { for (int k = 0; k < 6; ++k) { wave[k] = D3{ rng.normal(), rng.normal(), rng.normal() } * 4.0; phase[k] = rng.uniform() * 6.283185307179586; } }
        void eval(D3 d, double radius, double amplitude, D3& pos, D3& nrm) const
        {
            double s = 0;
            D3 grad{ 0, 0, 0 };
            for (int k = 0; k < 6; ++k) { double a = dot(wave[k], d) + phase[k]; s += std::sin(a); grad = grad + wave[k] * std::cos(a); }
            double r = radius * (1.0 + amplitude / 3.0 * s);
            grad = grad * (radius * amplitude / 3.0);
            D3 tangential = grad - d * dot(grad, d);
            nrm = unit(d * r - tangential);
            pos = d * r;
        }
    };

    // `count` displaced spheres (centres[i], same radius) as one OBJ.
    long long writeSpheres(const std::string& objPath, int frequency, const std::vector<D3>& centres, double radius, double amplitude, Rng& rng)
    {
        Geodesic g;
        buildGeodesic(frequency, g);
        const long nVerts = (long)g.dir.size();
        if (!writeMtl(objPath)) return -1;
        FILE* file = std::fopen(objPath.c_str(), "w");
        if (!file) return -1;
        Writer w(file);
        w.text(mtllibLine(objPath));
        std::vector<D3> nrm((size_t)nVerts * centres.size());
        for (size_t c = 0; c < centres.size(); ++c)
        {
            Bumps bumps(rng);
            for (long v = 0; v < nVerts; ++v)
            {
                D3 p;
                bumps.eval(g.dir[v], radius, amplitude, p, nrm[c * nVerts + v]);
                w.v3("v", centres[c] + p);
            }
        }
        w.text("vt 0 0\nvt 1 0\nvt 0 1\n");
        for (const D3& n : nrm) w.v3("vn", n);
        w.text("usemtl surface\n");
        long long nFaces = 0;
        for (size_t c = 0; c < centres.size(); ++c)
        {
            const long off = (long)(c * nVerts) + 1;
            for (size_t i = 0; i + 2 < g.faces.size(); i += 3, ++nFaces) w.face(g.faces[i] + off, g.faces[i + 1] + off, g.faces[i + 2] + off);
        }
        w.flush();
        bool ok = !std::ferror(file);
        std::fclose(file);
        return ok ? nFaces : -1;
    }
}

// Returns the number of OBJ faces written, or -1 on I/O error / bad arguments. Paths of any length are accepted, like
// CLOBJloader::LoadInto does (the reference's loader overflows an 80-byte buffer beyond ~75 characters).
extern "C" long long g3d_write_icosphere_obj(const char* path, int frequency, double radius, double amplitude, unsigned long long seed)
{
    std::string objPath(path ? path : "");
    if (objPath.size() < 5 || frequency < 1 || frequency > 2048) return -1;
    Rng rng(seed);
    return writeSpheres(objPath, frequency, { D3{ 0, 0, 0 } }, radius, amplitude, rng);
}

// `count` displaced icospheres of 20*f^2 faces each with centres uniform in [-extent, extent]^3 (they may overlap): a scene
// in which diffuse bounce rays leaving one surface meet another (BASELINE.json configs[2]'s incoherent batch).
extern "C" long long g3d_write_spheres_obj(const char* path, int count, int frequency, double extent, double radius, double amplitude, unsigned long long seed)
{
    std::string objPath(path ? path : "");
    if (objPath.size() < 5 || frequency < 1 || frequency > 2048 || count < 1 || count > 100000) return -1;
    Rng rng(seed);
    std::vector<D3> centres;
    for (int i = 0; i < count; ++i) centres.push_back(D3{ (rng.uniform() * 2 - 1) * extent, (rng.uniform() * 2 - 1) * extent, (rng.uniform() * 2 - 1) * extent });
    return writeSpheres(objPath, frequency, centres, radius, amplitude, rng);
}

extern "C" long long g3d_write_scattered_obj(const char* path, long long count, double extent, double edgeMin, double edgeMax, unsigned long long seed)
{
    std::string objPath(path ? path : "");
    if (objPath.size() < 5 || count < 1) return -1;
    if (!writeMtl(objPath)) return -1;
    FILE* file = std::fopen(objPath.c_str(), "w");
    if (!file) return -1;
    Writer w(file);
    w.text(mtllibLine(objPath));
    Rng rng(seed);
    std::vector<D3> normals((size_t)count);
    for (long long i = 0; i < count; ++i)
    {
        D3 c{ (rng.uniform() * 2 - 1) * extent, (rng.uniform() * 2 - 1) * extent, (rng.uniform() * 2 - 1) * extent };
        double e = edgeMin + (edgeMax - edgeMin) * rng.uniform();
        D3 p[3];
        for (int k = 0; k < 3; ++k) { p[k] = c + unit(D3{ rng.normal(), rng.normal(), rng.normal() }) * e; w.v3("v", p[k]); }
        D3 n = cross(p[1] - p[0], p[2] - p[0]);
        double l = std::sqrt(dot(n, n));
        normals[(size_t)i] = l > 0 ? n * (1.0 / l) : D3{ 0, 0, 1 };
    }
    w.text("vt 0 0\nvt 1 0\nvt 0 1\n");
    for (long long i = 0; i < count; ++i) w.v3("vn", normals[(size_t)i]);
    w.text("usemtl surface\n");
    for (long long i = 0; i < count; ++i) w.faceN(3 * i + 1, 3 * i + 2, 3 * i + 3, i + 1);
    w.flush();
    bool ok = !std::ferror(file);
    std::fclose(file);
    return ok ? count : -1;
}

#ifdef B2RT_SCENEGEN_MAIN
// Stand-alone scene generator (tools: bench.py's reference arm synthesises its workload with this executable so that it
// never loads the product's libraries):  scenegen icosphere <path.obj> <frequency> <radius> <amplitude> <seed>
//                                        scenegen scattered <path.obj> <count> <extent> <edge_min> <edge_max> <seed>
//                                        scenegen spheres <path.obj> <count> <frequency> <extent> <radius> <amplitude> <seed>
#include <cstdlib>
#include <cstring>
int main(int argc, char** argv)
{
    long long faces = -1;
    if (argc == 7 && !std::strcmp(argv[1], "icosphere"))
        faces = g3d_write_icosphere_obj(argv[2], std::atoi(argv[3]), std::atof(argv[4]), std::atof(argv[5]), std::strtoull(argv[6], nullptr, 10));
    else if (argc == 8 && !std::strcmp(argv[1], "scattered"))
        faces = g3d_write_scattered_obj(argv[2], std::atoll(argv[3]), std::atof(argv[4]), std::atof(argv[5]), std::atof(argv[6]), std::strtoull(argv[7], nullptr, 10));
    else if (argc == 9 && !std::strcmp(argv[1], "spheres"))
        faces = g3d_write_spheres_obj(argv[2], std::atoi(argv[3]), std::atoi(argv[4]), std::atof(argv[5]), std::atof(argv[6]), std::atof(argv[7]), std::strtoull(argv[8], nullptr, 10));
    else { std::fprintf(stderr, "usage: scenegen icosphere|scattered|spheres <path.obj> ...\n"); return 2; }
    if (faces < 0) { std::fprintf(stderr, "scenegen: failed to write %s\n", argv[2]); return 1; }
    std::printf("%lld\n", faces);
    return 0;
}
#endif
