// obj_scene.hpp — Wavefront OBJ/MTL -> std::vector<Triangle>, the job of loadTrianglesFromObj
// (common/loader.hpp:11-66) for the subset of the format the reference's assets use: v, f (v, v/vt, v//vn,
// v/vt/vn, negative indices), mtllib, usemtl; newmtl, Kd, Ke.
//
// Primitive ids and vertex bits are part of the parity contract (every kernel indexes the triangle array by
// primitive id and the intersector reads the vertex bits), so two behaviours of the reference's parser —
// tinyobjloader v1.0.6 (libs/tiny_obj_loader, MIT; a third-party dependency of the reference) — are restated:
//   * polygons become a triangle fan (f0, f[k-1], f[k]), faces in file order, one Triangle per fan triangle,
//     each with the material active at the face;
//   * decimal numbers are NOT correctly rounded: the parser accumulates the integer digits as m = m*10 + d in
//     double, adds each fraction digit as d * 10^-k (a table of the literals 0.1 ... 0.0000001 for k <= 7, pow(10,-k)
//     beyond), applies an exponent as ldexp(m * pow(5, e), e), and only then narrows to float.  parse_real() below
//     performs the same operations in the same order, so the floats match bit for bit
//     (tests/test_host_obj.py checks them against the reference loader's output).
#pragma once
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/cedecrt.h"
#include "crt_host.hpp"

namespace crt
{
namespace objdetail
{
inline bool is_digit(char c) { return c >= '0' && c <= '9'; }

// one whitespace-delimited token -> double by the accumulation scheme described above; false = not a number
inline bool parse_double(const char* s, const char* end, double* out)
{
    if (s >= end) return false;
    const char* p = s;
    bool negative = false;
    if (*p == '+' || *p == '-')
    {
        negative = *p == '-';
        ++p;
    }
    else if (!is_digit(*p)) return false;
    double m = 0.0;
    int n_read = 0;
    while (p != end && is_digit(*p))
    {
        m *= 10;
        m += (int)(*p - '0');
        ++p;
        ++n_read;
    }
    if (n_read == 0) return false;
    int exponent = 0;
    if (p != end && *p == '.')
    {
        static const double neg_pow10[] = {1.0, 0.1, 0.01, 0.001, 0.0001, 0.00001, 0.000001, 0.0000001};
        ++p;
        int k = 1;
        while (p != end && is_digit(*p))
        {
            m += (int)(*p - '0') * (k < 8 ? neg_pow10[k] : std::pow(10.0, -k));
            ++k;
            ++p;
        }
    }
    else if (p != end && !(*p == 'e' || *p == 'E')) p = end;  // trailing garbage: keep what was read
    if (p != end && (*p == 'e' || *p == 'E'))
    {
        ++p;
        bool exp_negative = false;
        if (p != end && (*p == '+' || *p == '-'))
        {
            exp_negative = *p == '-';
            ++p;
        }
        else if (p == end || !is_digit(*p)) return false;
        int digits = 0;
        while (p != end && is_digit(*p))
        {
            exponent = exponent * 10 + (int)(*p - '0');
            ++p;
            ++digits;
        }
        if (digits == 0) return false;
        if (exp_negative) exponent = -exponent;
    }
    const double v = exponent ? std::ldexp(m * std::pow(5.0, exponent), exponent) : m;
    *out = (negative ? -1 : 1) * v;
    return true;
}
inline float parse_real(const char** cursor, double fallback = 0.0)
{
    const char* t = *cursor + strspn(*cursor, " \t");
    const char* end = t + strcspn(t, " \t\r\n");
    double v = fallback;
    parse_double(t, end, &v);
    *cursor = end;
    return (float)v;
}
inline std::string rest_of_line(const char* p)
{
    p += strspn(p, " \t");
    std::string s(p);
    while (!s.empty() && (s.back() == '\n' || s.back() == '\r' || s.back() == ' ' || s.back() == '\t')) s.pop_back();
    return s;
}
struct Material
{
    crt_float3 kd{0.0f, 0.0f, 0.0f}, ke{0.0f, 0.0f, 0.0f};
};
inline void load_mtl(const std::string& path, std::vector<Material>& mats, std::map<std::string, int>& ids)
{
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) throw Error(CRT_EINVAL, "cannot open material library " + path);
    std::vector<char> line(1 << 16);
    int cur = -1;
    while (fgets(line.data(), (int)line.size(), f))
    {
        const char* p = line.data() + strspn(line.data(), " \t");
        if (!strncmp(p, "newmtl", 6) && (p[6] == ' ' || p[6] == '\t'))
        {
            const std::string name = rest_of_line(p + 7);
            mats.push_back(Material());
            cur = (int)mats.size() - 1;
            if (!ids.count(name)) ids[name] = cur;
        }
        else if (cur >= 0 && p[0] == 'K' && (p[1] == 'd' || p[1] == 'e') && (p[2] == ' ' || p[2] == '\t'))
        {
            const char* c = p + 3;
            crt_float3 v;
            v.x = parse_real(&c);
            v.y = parse_real(&c);
            v.z = parse_real(&c);
            (p[1] == 'd' ? mats[cur].kd : mats[cur].ke) = v;
        }
    }
    fclose(f);
}
}  // namespace objdetail

// loadTrianglesFromObj(filename, mtl_basedir) (common/loader.hpp:11-66); mtl_basedir defaults to the OBJ's directory
inline std::vector<crt_triangle> loadTrianglesFromObj(const std::string& filename, std::string mtl_basedir = "")
{
    using namespace objdetail;
    if (mtl_basedir.empty())
    {
        const size_t slash = filename.find_last_of('/');
        mtl_basedir = slash == std::string::npos ? "" : filename.substr(0, slash + 1);
    }
    else if (mtl_basedir.back() != '/') mtl_basedir += '/';
    FILE* f = fopen(filename.c_str(), "rb");
    if (!f) throw Error(CRT_EINVAL, "cannot open " + filename);
    std::vector<crt_float3> positions;
    std::vector<Material> mats;
    std::map<std::string, int> mat_ids;
    std::vector<crt_triangle> out;
    int cur_mat = -1;
    std::vector<char> line(1 << 20);  // 64-gons with v/vt/vn triples stay far below this
    std::vector<int> face;
    while (fgets(line.data(), (int)line.size(), f))
    {
        const char* p = line.data() + strspn(line.data(), " \t");
        if (p[0] == 'v' && (p[1] == ' ' || p[1] == '\t'))
        {
            const char* c = p + 2;
            crt_float3 v;
            v.x = parse_real(&c);
            v.y = parse_real(&c);
            v.z = parse_real(&c);
            positions.push_back(v);
        }
        else if (p[0] == 'f' && (p[1] == ' ' || p[1] == '\t'))
        {
            face.clear();
            const char* c = p + 2;
            for (;;)
            {
                c += strspn(c, " \t");
                if (*c == '\0' || *c == '\r' || *c == '\n') break;
                const int idx = atoi(c);  // the vertex index is the integer before the first '/'
                // 1-based; negative counts back from the vertices read so far
                face.push_back(idx > 0 ? idx - 1 : (int)positions.size() + idx);
                c += strcspn(c, " \t\r\n");
            }
            if (face.size() < 3) continue;
            if (cur_mat < 0) throw Error(CRT_EINVAL, filename + ": face without a material (the reference indexes materials[-1])");
            for (size_t k = 2; k < face.size(); k++)
            {
                const int id[3] = {face[0], face[k - 1], face[k]};
                crt_triangle t;
                for (int j = 0; j < 3; j++)
                {
                    if (id[j] < 0 || (size_t)id[j] >= positions.size()) throw Error(CRT_EINVAL, filename + ": vertex index out of range");
                    t.vertices[j] = positions[(size_t)id[j]];
                }
                t.color = mats[(size_t)cur_mat].kd;
                t.emissive = mats[(size_t)cur_mat].ke;
                out.push_back(t);
            }
        }
        else if (!strncmp(p, "usemtl", 6) && (p[6] == ' ' || p[6] == '\t'))
        {
            const std::string name = rest_of_line(p + 7);
            const auto it = mat_ids.find(name);
            cur_mat = it == mat_ids.end() ? -1 : it->second;
        }
        else if (!strncmp(p, "mtllib", 6) && (p[6] == ' ' || p[6] == '\t'))
            load_mtl(mtl_basedir + rest_of_line(p + 7), mats, mat_ids);
    }
    fclose(f);
    return out;
}
}  // namespace crt
