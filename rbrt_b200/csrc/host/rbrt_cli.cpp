// rbrt_cli.cpp — the `rbrt` command line (reference: src/main.rs:9-92) hosted in C++ over the C-ABI of
// include/rbrt_gpu.h.  The reference's host language is Rust and no Rust toolchain exists in the build image, so the
// compiled host side is C++: same flags and defaults (main.rs:14-50), same call sequence (main.rs:70-91)
//     load_blueprints_from_yaml_file -> Camera::new(height, width) -> create_scene_from_scene_blueprint -> render_scene -> save
// with the scene description of rbrt_lib/src/blueprints.rs:15-158 (YAML), the .obj loading and vertex transform of
// rbrt_lib/src/mesh.rs:78-121, and the reference's messages.  The hot path is entirely inside librbrt_gpu.so.
//
// Third-party pieces of the reference that are re-stated here, host-side and outside the hot path (parity unpinned by the
// reference's tests): serde_yaml 0.9 -> scene_yaml.hpp (block and flow YAML, anchors, serde's struct / Option / f32 rules);
// tobj 4 -> the library's rbrt_mesh_load_obj (csrc/obj_loader.cpp:
// `v` / `f` / `l` records, models per `o` / `g` / `usemtl`, faces consumed as index triples, no triangulation); image 0.25 -> an 8-bit RGB
// PNG written with zlib (lossless, so any conforming encoder stores the same pixels), binary PPM, 24-bit BMP, uncompressed TGA, baseline TIFF or QOI by extension.
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cctype>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <memory>
#include <sstream>
#include <string>
#include <system_error>
#include <thread>
#include <vector>

#include "../../../include/rbrt_gpu.h"
#include "scene_yaml.hpp"

namespace {

[[noreturn]] void die(const std::string& msg) {              // the reference panics; we exit(101) like a Rust panic does
    fprintf(stderr, "%s\n", msg.c_str());
    exit(101);
}

// ------------------------------------------------------------------ blueprints.rs:15-48,76-92 (scene_yaml.hpp)
using scene_yaml::MaterialBp;
using scene_yaml::SceneBp;

SceneBp load_blueprints_from_yaml_file(const std::string& path) {   // blueprints.rs:76-92
    std::ifstream f(path, std::ios::binary);
    if (!f) die("Failed to open " + path + " to load content.");
    std::stringstream buf; buf << f.rdbuf();
    try {
        return scene_yaml::parse_scene(buf.str());
    } catch (const scene_yaml::ParseError& e) {
        die("Unable to parse content of file \"" + path + "\" to scene blueprint: " + e.msg);
    }
}

std::string lower(std::string s) { for (auto& c : s) c = (char)tolower((unsigned char)c); return s; }

// blueprints.rs:50-74: first match of "metal", "lambert", "dielectric"; a missing required field is the reference's `expect` panic
bool create_material_from_description(const MaterialBp& m, rbrt_material* out) {
    std::string t = lower(m.type);
    if (t.find("metal") != std::string::npos) {
        if (!m.has_albedo) die("you forgot to specify an albedo vector for metal");
        if (!m.has_param) die("you forgot to specify a roughness (i.e. material_param: 0.1) for metal");
        *out = rbrt_material{RBRT_MAT_METAL, m.albedo, m.param};
        return true;
    }
    if (t.find("lambert") != std::string::npos) {
        if (!m.has_albedo) die("you forgot to specify an albedo vector for lambertian");
        *out = rbrt_material{RBRT_MAT_LAMBERTIAN, m.albedo, 0.0f};
        return true;
    }
    if (t.find("dielectric") != std::string::npos) {
        if (!m.has_param) die("you forgot to specify a refractory index vector (i.e. material_param: 1.8) dielectric");
        *out = rbrt_material{RBRT_MAT_DIELECTRIC, rbrt_vec3{0, 0, 0}, m.param};
        return true;
    }
    printf("Cannot figure out material_type from %s, material_type must be one of metal, lambertian or dielectric!\n", m.type.c_str());
    return false;
}

// ------------------------------------------------------------------ mesh.rs:78-121
// The .obj reader and the vertex transform are the library's (rbrt_mesh_load_obj, csrc/obj_loader.cpp): tobj's records and
// model boundaries, parsed on all host threads.  A load the reference would panic on (mesh.rs:89) ends the process the same way.
struct Soup {
    float* v = nullptr; uint64_t n = 0;
    Soup() = default;
    Soup(Soup&& o) noexcept : v(o.v), n(o.n) { o.v = nullptr; o.n = 0; }
    Soup(const Soup&) = delete;
    ~Soup() { rbrt_mesh_free(v); }
};
Soup load_mesh_vertices_from_file(const std::string& path, rbrt_vec3 translation, rbrt_vec3 rotation, float scale) {
    Soup s;
    if (rbrt_mesh_load_obj(path.c_str(), translation, rotation, scale, &s.v, &s.n) != RBRT_OK) die(std::string("assertion failed: loaded_mesh.is_ok() (") + rbrt_last_error() + ")");
    printf("Successfully loaded %llu triangles from file %s!\n", (unsigned long long)s.n, path.c_str());   // mesh.rs:115-119
    return s;
}

// ------------------------------------------------------------------ image save (main.rs:86)
void put_u32(std::vector<uint8_t>& v, uint32_t x) { for (int s = 24; s >= 0; s -= 8) v.push_back((uint8_t)(x >> s)); }
void chunk(std::vector<uint8_t>& out, const char* tag, const std::vector<uint8_t>& data) {
    put_u32(out, (uint32_t)data.size());
    out.insert(out.end(), tag, tag + 4);
    out.insert(out.end(), data.begin(), data.end());
    uLong crc = crc32(0L, (const Bytef*)tag, 4);                          // the CRC covers type + data
    for (size_t a = 0; a < data.size(); a += 1u << 30) crc = crc32(crc, data.data() + a, (uInt)std::min<size_t>(data.size() - a, 1u << 30));
    put_u32(out, (uint32_t)crc);
}
// One zlib stream from independently deflated 256 KB bands (the pigz construction): every band but the last ends with a sync flush — a byte
// boundary and no final block — so the raw-deflate pieces concatenate into one valid stream; zlib header and the Adler-32 of the whole input
// wrap it.  A noisy 1080p frame costs 280 ms of zlib on one core, nine times its 33 ms on the GPU; on 8 threads ~45 ms.
bool deflate_parallel(const std::vector<uint8_t>& raw, std::vector<uint8_t>& z) {
    const size_t band = 1u << 18, n_bands = raw.empty() ? 1 : (raw.size() + band - 1) / band;
    std::vector<std::vector<uint8_t>> parts(n_bands);
    std::vector<char> ok(n_bands, 0);
    auto one = [&](size_t k) {
        const size_t a = k * band, b = std::min(raw.size(), a + band);
        z_stream zs; memset(&zs, 0, sizeof(zs));
        if (deflateInit2(&zs, 6, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) return;
        parts[k].resize(deflateBound(&zs, (uLong)(b - a)) + 16);
        zs.next_in = const_cast<Bytef*>(raw.data() + a); zs.avail_in = (uInt)(b - a);
        zs.next_out = parts[k].data(); zs.avail_out = (uInt)parts[k].size();
        const bool last = k + 1 == n_bands;
        const int rc = deflate(&zs, last ? Z_FINISH : Z_SYNC_FLUSH);
        ok[k] = (last ? rc == Z_STREAM_END : rc == Z_OK) && zs.avail_in == 0;
        parts[k].resize(zs.total_out);
        deflateEnd(&zs);
    };
    unsigned threads = std::max(1u, std::min<unsigned>({std::thread::hardware_concurrency(), 16u, (unsigned)n_bands}));
    std::atomic<size_t> next{0};
    auto worker = [&] { for (size_t k; (k = next.fetch_add(1)) < n_bands;) one(k); };
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < threads; ++t) { try { pool.emplace_back(worker); } catch (const std::system_error&) { break; } }
    worker();
    for (auto& th : pool) th.join();
    z.clear(); z.push_back(0x78); z.push_back(0x9C);
    for (size_t k = 0; k < n_bands; ++k) { if (!ok[k]) return false; z.insert(z.end(), parts[k].begin(), parts[k].end()); }
    uLong ad = adler32(0L, Z_NULL, 0);
    for (size_t a = 0; a < raw.size(); a += 1u << 30) ad = adler32(ad, raw.data() + a, (uInt)std::min<size_t>(raw.size() - a, 1u << 30));
    for (int sft = 24; sft >= 0; sft -= 8) z.push_back((uint8_t)(ad >> sft));
    return true;
}

bool save_image(const std::string& path, const std::vector<uint8_t>& rgb, uint32_t w, uint32_t h) {
    std::string ext = path.size() >= 4 ? lower(path.substr(path.find_last_of('.') == std::string::npos ? path.size() : path.find_last_of('.'))) : "";
    std::vector<uint8_t> out;
    if (ext == ".png") {
        const uint8_t sig[8] = {0x89, 'P', 'N', 'G', '\r', '\n', 0x1a, '\n'};
        out.insert(out.end(), sig, sig + 8);
        std::vector<uint8_t> ihdr; put_u32(ihdr, w); put_u32(ihdr, h);
        const uint8_t tail[5] = {8, 2, 0, 0, 0};             // 8-bit, colour type 2 (RGB), deflate, filter 0, no interlace
        ihdr.insert(ihdr.end(), tail, tail + 5);
        chunk(out, "IHDR", ihdr);
        std::vector<uint8_t> raw; raw.reserve((size_t)h * (1 + 3 * (size_t)w));
        for (uint32_t y = 0; y < h; ++y) { raw.push_back(0); raw.insert(raw.end(), rgb.begin() + (size_t)y * w * 3, rgb.begin() + (size_t)(y + 1) * w * 3); }
        std::vector<uint8_t> z;
        if (!deflate_parallel(raw, z)) return false;
        chunk(out, "IDAT", z);
        chunk(out, "IEND", {});
    } else if (ext == ".ppm" || ext == ".pnm") {
        char hdr[64]; int n = snprintf(hdr, sizeof(hdr), "P6\n%u %u\n255\n", w, h);
        out.insert(out.end(), hdr, hdr + n);
        out.insert(out.end(), rgb.begin(), rgb.end());
    } else if (ext == ".bmp") {                                  // 24-bit BI_RGB, bottom-up rows of BGR padded to 4 bytes
        const uint32_t stride = (3 * w + 3) & ~3u, size = 54 + stride * h;
        auto le32 = [&](uint32_t x) { for (int s = 0; s < 32; s += 8) out.push_back((uint8_t)(x >> s)); };
        auto le16 = [&](uint32_t x) { out.push_back((uint8_t)x); out.push_back((uint8_t)(x >> 8)); };
        out.push_back('B'); out.push_back('M'); le32(size); le32(0); le32(54);
        le32(40); le32(w); le32(h); le16(1); le16(24); le32(0); le32(stride * h); le32(2835); le32(2835); le32(0); le32(0);
        for (uint32_t y = h; y-- > 0;) {
            for (uint32_t x = 0; x < w; ++x) { const uint8_t* p = &rgb[((size_t)y * w + x) * 3]; out.push_back(p[2]); out.push_back(p[1]); out.push_back(p[0]); }
            for (uint32_t k = 3 * w; k < stride; ++k) out.push_back(0);
        }
    } else if (ext == ".tga") {                                  // uncompressed true-colour, top-left origin, BGR
        const uint8_t hdr[18] = {0, 0, 2, 0, 0, 0, 0, 0, 0, 0, 0, 0, (uint8_t)w, (uint8_t)(w >> 8), (uint8_t)h, (uint8_t)(h >> 8), 24, 0x20};
        if (w > 65535 || h > 65535) return false;
        out.insert(out.end(), hdr, hdr + 18);
        for (size_t i = 0; i < (size_t)w * h; ++i) { out.push_back(rgb[3 * i + 2]); out.push_back(rgb[3 * i + 1]); out.push_back(rgb[3 * i]); }
    } else if (ext == ".tif" || ext == ".tiff") {                // baseline TIFF 6.0: little-endian, one uncompressed RGB strip, IFD after it
        const uint64_t n64 = 3ull * w * h;
        if (n64 > 0xFFFFF000ull) return false;
        const uint32_t n = (uint32_t)n64, ifd_at = 8 + n + (n & 1), bits_at = ifd_at + 2 + 10 * 12 + 4;
        auto le16 = [&](uint32_t x) { out.push_back((uint8_t)x); out.push_back((uint8_t)(x >> 8)); };
        auto le32 = [&](uint32_t x) { for (int s = 0; s < 32; s += 8) out.push_back((uint8_t)(x >> s)); };
        auto tag = [&](uint32_t t, uint32_t type, uint32_t count, uint32_t value) { le16(t); le16(type); le32(count); le32(value); };
        out.push_back('I'); out.push_back('I'); le16(42); le32(ifd_at);
        out.insert(out.end(), rgb.begin(), rgb.end());
        if (n & 1) out.push_back(0);
        le16(10);
        tag(256, 4, 1, w); tag(257, 4, 1, h); tag(258, 3, 3, bits_at); tag(259, 3, 1, 1); tag(262, 3, 1, 2); tag(273, 4, 1, 8); tag(277, 3, 1, 3);
        tag(278, 4, 1, h); tag(279, 4, 1, n); tag(284, 3, 1, 1);
        le32(0);
        le16(8); le16(8); le16(8);
    } else if (ext == ".qoi") {                                  // qoiformat.org, 3 channels: run / index / diff / luma / rgb
        const uint8_t hdr[14] = {'q', 'o', 'i', 'f', (uint8_t)(w >> 24), (uint8_t)(w >> 16), (uint8_t)(w >> 8), (uint8_t)w,
                                 (uint8_t)(h >> 24), (uint8_t)(h >> 16), (uint8_t)(h >> 8), (uint8_t)h, 3, 0};
        out.insert(out.end(), hdr, hdr + 14);
        uint8_t index[64][4] = {};                                 // RGBA, all zero at the start: an untouched slot (alpha 0) never equals a pixel (alpha 255)
        uint8_t pr = 0, pg = 0, pb = 0; int run = 0;
        const size_t px = (size_t)w * h;
        for (size_t i = 0; i < px; ++i) {
            const uint8_t r = rgb[3 * i], g = rgb[3 * i + 1], b = rgb[3 * i + 2];
            if (r == pr && g == pg && b == pb) {
                if (++run == 62 || i + 1 == px) { out.push_back((uint8_t)(0xC0 | (run - 1))); run = 0; }
                continue;
            }
            if (run) { out.push_back((uint8_t)(0xC0 | (run - 1))); run = 0; }
            const int k = (r * 3 + g * 5 + b * 7 + 255 * 11) % 64;
            if (index[k][0] == r && index[k][1] == g && index[k][2] == b && index[k][3] == 255) out.push_back((uint8_t)k);
            else {
                index[k][0] = r; index[k][1] = g; index[k][2] = b; index[k][3] = 255;
                const int dr = (int8_t)(r - pr), dg = (int8_t)(g - pg), db = (int8_t)(b - pb);
                if (dr >= -2 && dr <= 1 && dg >= -2 && dg <= 1 && db >= -2 && db <= 1) out.push_back((uint8_t)(0x40 | (dr + 2) << 4 | (dg + 2) << 2 | (db + 2)));
                else if (dg >= -32 && dg <= 31 && dr - dg >= -8 && dr - dg <= 7 && db - dg >= -8 && db - dg <= 7) { out.push_back((uint8_t)(0x80 | (dg + 32))); out.push_back((uint8_t)((dr - dg + 8) << 4 | (db - dg + 8))); }
                else { out.push_back(0xFE); out.push_back(r); out.push_back(g); out.push_back(b); }
            }
            pr = r; pg = g; pb = b;
        }
        for (int i = 0; i < 7; ++i) out.push_back(0);
        out.push_back(1);
    } else return false;                                         // lossy formats of the `image` crate (jpeg, ...) are not offered
    FILE* fp = fopen(path.c_str(), "wb");
    if (!fp) return false;
    bool ok = fwrite(out.data(), 1, out.size(), fp) == out.size();
    return fclose(fp) == 0 && ok;
}

// Portable float map (little-endian): "PF" (3 channels) or "Pf" (1), width height, scale -1 (negative = little-endian), rows bottom to top.
bool save_pfm(const std::string& path, const float* v, uint32_t w, uint32_t h, int channels) {
    FILE* fp = fopen(path.c_str(), "wb");
    if (!fp) return false;
    bool ok = fprintf(fp, "%s\n%u %u\n-1.0\n", channels == 3 ? "PF" : "Pf", w, h) > 0;
    const uint16_t probe = 1;
    const bool little = *(const uint8_t*)&probe == 1;
    std::vector<float> row((size_t)w * channels);
    for (uint32_t y = h; ok && y-- > 0;) {
        memcpy(row.data(), v + (size_t)y * w * channels, row.size() * 4);
        if (!little) for (float& f : row) { uint32_t u; memcpy(&u, &f, 4); u = __builtin_bswap32(u); memcpy(&f, &u, 4); }
        ok = fwrite(row.data(), 4, row.size(), fp) == row.size();
    }
    return fclose(fp) == 0 && ok;
}

void usage() {
    printf("a lighweight raytracer written in rust\n\nUsage: rbrt [OPTIONS]\n\nOptions:\n"
           "  -t, --target_file <target_file>  file that will be created witht he rendered output [default: dbg_out.png]\n"
           "      --height <height>            target image resolution height [default: 600]\n"
           "  -w, --width <width>              target image resolution width [default: 800]\n"
           "  -c, --config <config>            YAML file that specifies the scene layout and camera specification. [default: scenes/example_scene.yaml]\n"
           "  -s, --samples <samples>          number of rays per pixel [default: 5]\n"
           "      --seed <seed>                (extension) Philox seed; the reference is unseeded [default: 0]\n"
           "      --device <device>            (extension) CUDA device [default: 0]\n"
           "      --gpus <n>                   (extension) render on the first n GPUs of this box: tile-sharded inside the library [default: 1]\n"
           "      --transport <auto|nccl|peer> (extension) how the GPUs exchange the scene and the image [default: auto]\n"
           "      --check                      (extension) parse the scene, print a summary and exit without rendering\n"
           "      --dump                       (extension, with --check) also print every blueprint field as read (f32 bit patterns)\n"
           "      --from-ppm <file>            (extension) no rendering: read a binary PPM (P6) and save it as --target_file (format by extension)\n"
           "      --aov <prefix>               (extension) after the render also write first-hit AOVs of the same camera and --seed:\n"
           "                                   <prefix>.depth.pfm, <prefix>.normal.pfm, <prefix>.albedo.pfm, <prefix>.coverage.pfm\n"
           "      --aov-samples <n>            (extension) samples per pixel of the AOVs [default: --samples]\n"
           "      --denoise                    (extension) save the image denoised on the GPU, guided by AOVs of the same camera and --seed [--aov-samples default: min(--samples, 4)]\n"
           "      --denoise-splits <k>         (extension, with --denoise) render the image as k sample shards (2..16, dividing --samples) for its per-pixel\n"
           "                                   variance, and denoise with the variance-guided filter [--aov-samples default: min(--samples / k, 4)]\n"
           "  -h, --help                       Print help\n  -V, --version                    Print version\n");
}

uint32_t parse_u32(const char* s, const char* what) {
    char* end = nullptr;
    unsigned long v = strtoul(s, &end, 10);
    if (end == s || *end || v > 0xFFFFFFFFul) die(std::string("error: invalid value '") + s + "' for '" + what + "'");
    return (uint32_t)v;
}

}  // namespace

int main(int argc, char** argv) {
    std::string target = "dbg_out.png", config = "scenes/example_scene.yaml";      // main.rs:14-50
    uint32_t height = 600, width = 800, samples = 5;
    uint64_t seed = 0; int device = 0; bool check_only = false, dump = false, denoise = false;
    uint32_t gpus = 1; int transport = RBRT_TRANSPORT_AUTO;
    std::string from_ppm, aov;
    uint32_t aov_samples = 0, denoise_splits = 0;
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        auto value = [&](const char* name) -> const char* {
            size_t eq = a.find('=');
            if (eq != std::string::npos) return argv[i] + eq + 1;
            if (i + 1 >= argc) die(std::string("error: a value is required for '") + name + "' but none was supplied");
            return argv[++i];
        };
        std::string key = a.substr(0, a.find('='));
        if (key == "-t" || key == "--target_file") target = value("--target_file");
        else if (key == "--height") height = parse_u32(value("--height"), "--height");
        else if (key == "-w" || key == "--width") width = parse_u32(value("--width"), "--width");
        else if (key == "-c" || key == "--config") config = value("--config");
        else if (key == "-s" || key == "--samples") samples = parse_u32(value("--samples"), "--samples");
        else if (key == "--seed") seed = strtoull(value("--seed"), nullptr, 0);
        else if (key == "--device") device = (int)parse_u32(value("--device"), "--device");
        else if (key == "--gpus") gpus = parse_u32(value("--gpus"), "--gpus");
        else if (key == "--transport") {
            std::string t = value("--transport");
            if (t == "auto") transport = RBRT_TRANSPORT_AUTO; else if (t == "nccl") transport = RBRT_TRANSPORT_NCCL; else if (t == "peer") transport = RBRT_TRANSPORT_PEER;
            else die("error: invalid value '" + t + "' for '--transport' [possible values: auto, nccl, peer]");
        }
        else if (key == "--check") check_only = true;
        else if (key == "--dump") dump = true;
        else if (key == "--from-ppm") from_ppm = value("--from-ppm");
        else if (key == "--aov") aov = value("--aov");
        else if (key == "--aov-samples") aov_samples = parse_u32(value("--aov-samples"), "--aov-samples");
        else if (key == "--denoise") denoise = true;
        else if (key == "--denoise-splits") denoise_splits = parse_u32(value("--denoise-splits"), "--denoise-splits");
        else if (key == "-h" || key == "--help") { usage(); return 0; }
        else if (key == "-V" || key == "--version") { printf("rbrt 0.1 (%s)\n", rbrt_gpu_version()); return 0; }
        else { fprintf(stderr, "error: unexpected argument '%s' found\n", a.c_str()); return 2; }
    }

    if (denoise_splits) {
        if (!denoise) die("error: '--denoise-splits' needs '--denoise'");
        if (denoise_splits < 2 || denoise_splits > 16) die("error: '--denoise-splits' must be 2..16");
        if (!samples || samples % denoise_splits) die("error: '--denoise-splits' must divide '--samples'");
        if (aov_samples > samples / denoise_splits)
            die("error: '--aov-samples' must not exceed '--samples' / '--denoise-splits' with '--denoise-splits': the guides must be the first camera rays of shard 0");
        if (!aov_samples) aov_samples = std::min<uint32_t>(samples / denoise_splits, 4);
    }
    if (denoise) {
        if (!from_ppm.empty()) die("error: '--denoise' cannot be used with '--from-ppm' (there is no render to denoise)");
        if (aov_samples > samples) die("error: '--aov-samples' must not exceed '--samples' with '--denoise': the guides must be the image's first camera rays");
        if (!aov_samples) aov_samples = std::min<uint32_t>(samples, 4);
    }
    if (!from_ppm.empty()) {                                                        // the image writers on their own (main.rs:84-91)
        std::ifstream f(from_ppm, std::ios::binary);
        std::string magic; uint32_t w = 0, h = 0, maxv = 0;
        if (!(f >> magic >> w >> h >> maxv) || magic != "P6" || maxv != 255 || !w || !h) die("cannot read " + from_ppm + " as a binary PPM");
        f.get();
        std::vector<uint8_t> rgb((size_t)w * h * 3);
        if (!f.read((char*)rgb.data(), (std::streamsize)rgb.size())) die("cannot read " + from_ppm + " as a binary PPM");
        printf("Saving rendered image to %s\n", target.c_str());
        if (!save_image(target, rgb, w, h)) die("Unable to save target img to " + target + "! Maybe the directory does not exist?");
        return 0;
    }
    SceneBp bp = load_blueprints_from_yaml_file(config);
    if (check_only && dump) {                                                      // what serde would have put into SceneBlueprint
        auto bits = [](float f) { uint32_t u; memcpy(&u, &f, 4); return u; };
        auto v3 = [&](const char* name, rbrt_vec3 v) { printf("%s %08x %08x %08x\n", name, bits(v.x), bits(v.y), bits(v.z)); };
        auto mat = [&](const MaterialBp& m) {
            printf("material_type %zu:%s\n", m.type.size(), m.type.c_str());
            if (m.has_albedo) v3("albedo", m.albedo); else printf("albedo None\n");
            if (m.has_param) printf("material_param %08x\n", bits(m.param)); else printf("material_param None\n");
        };
        v3("camera_up", bp.up); v3("camera_look_at", bp.look_at); v3("camera_position", bp.position); printf("camera_focal_length_mm %08x\n", bits(bp.focal));
        for (auto& m : bp.meshes) { printf("mesh\nobj_filepath %zu:%s\nscale %08x\n", m.obj.size(), m.obj.c_str(), bits(m.scale)); v3("translation", m.translation); v3("rotation_rad", m.rotation); mat(m.mat); }
        for (auto& sp : bp.spheres) { printf("sphere\nradius %08x\n", bits(sp.radius)); v3("center", sp.center); mat(sp.mat); }
        return 0;
    }
    rbrt_camera cam;
    if (rbrt_camera_new(bp.position, bp.look_at, bp.up, height, width, bp.focal, &cam) != RBRT_OK) die("rbrt_camera_new failed");   // height BEFORE width (main.rs:71-78)

    // create_scene_from_scene_blueprint (blueprints.rs:132-158): meshes first, then spheres; unknown materials are skipped
    std::vector<Soup> soups;
    std::vector<rbrt_mesh_desc> meshes;
    for (auto& m : bp.meshes) {
        rbrt_material mat;
        if (!create_material_from_description(m.mat, &mat)) { printf("Failed to parse material info provided with mesh!\n"); continue; }
        soups.push_back(load_mesh_vertices_from_file(m.obj, m.translation, m.rotation, m.scale));
        meshes.push_back(rbrt_mesh_desc{soups.back().v, soups.back().n, mat});
    }
    std::vector<rbrt_sphere_desc> spheres;
    for (auto& s : bp.spheres) {
        rbrt_material mat;
        if (!create_material_from_description(s.mat, &mat)) continue;
        spheres.push_back(rbrt_sphere_desc{s.center, s.radius, mat});
    }
    if (check_only) {
        uint64_t nt = 0; for (auto& m : meshes) nt += m.num_triangles;
        printf("scene ok: %zu spheres, %zu meshes, %llu triangles, camera %ux%u focal %g mm\n", spheres.size(), meshes.size(), (unsigned long long)nt,
               cam.img_width_pix, cam.img_height_pix, cam.focal_len_mm);
        return 0;
    }

    // The reference's render_scene spreads over every core of the host (rayon, lib.rs:84-86); here --gpus spreads it over the
    // GPUs of the box: ONE process, the library replicates the scene and shards the image (csrc/multi.cu).
    if (gpus > 1) {
        std::vector<int> devs(gpus);
        for (uint32_t i = 0; i < gpus; ++i) devs[i] = device + (int)i;
        if (rbrt_gpu_init_multi(devs.data(), (int)gpus, transport) != RBRT_OK) die(std::string("rbrt_gpu: ") + rbrt_last_error());
    } else if (rbrt_gpu_init(device) != RBRT_OK) die(std::string("rbrt_gpu: ") + rbrt_last_error());
    rbrt_scene* scene = nullptr;
    if (rbrt_gpu_scene_create(spheres.data(), (uint32_t)spheres.size(), meshes.data(), (uint32_t)meshes.size(), nullptr, &scene) != RBRT_OK)
        die(std::string("rbrt_gpu: ") + rbrt_last_error());
    printf("Starting rendering...\n");                                             // lib.rs:80
    std::vector<uint8_t> rgb((size_t)width * height * 3);
    rbrt_render_opts opts; memset(&opts, 0, sizeof(opts)); opts.seed = seed;
    rbrt_stats st;
    std::vector<float> hdr, var;
    if (denoise_splits) {                                                          // the mean colour and its variance (on the first device)
        hdr.resize((size_t)width * height * 3); var.resize(hdr.size());
        if (rbrt_gpu_render_hdr_variance(scene, &cam, samples, denoise_splits, &opts, hdr.data(), var.data(), &st) != RBRT_OK)
            die(std::string("rbrt_gpu: ") + rbrt_last_error());
    } else if (denoise) {                                                          // the mean colour, denoised below into rgb
        hdr.resize((size_t)width * height * 3);
        if (rbrt_gpu_render_hdr(scene, &cam, samples, &opts, hdr.data(), &st) != RBRT_OK) die(std::string("rbrt_gpu: ") + rbrt_last_error());
    } else if (rbrt_gpu_render(scene, &cam, samples, &opts, rgb.data(), &st) != RBRT_OK) die(std::string("rbrt_gpu: ") + rbrt_last_error());
    printf("\rRendering 100%% complete!\n");                                        // lib.rs:114
    std::vector<float> depth, normal, albedo, coverage;
    if (!aov.empty() || denoise) {                                                 // first-hit AOVs of the same camera rays (include/rbrt_gpu.h)
        const size_t n = (size_t)width * height;
        depth.resize(n); normal.resize(3 * n); albedo.resize(3 * n); coverage.resize(n);
        rbrt_aov_out ao; memset(&ao, 0, sizeof(ao));
        ao.depth = depth.data(); ao.normal = normal.data(); ao.albedo = albedo.data(); ao.coverage = coverage.data();
        if (rbrt_gpu_render_aov(scene, &cam, aov_samples ? aov_samples : samples, seed, &ao, nullptr) != RBRT_OK) die(std::string("rbrt_gpu: ") + rbrt_last_error());
        if (denoise_splits) {
            if (rbrt_gpu_denoise_variance(width, height, hdr.data(), var.data(), &ao, nullptr, nullptr, rgb.data(), nullptr) != RBRT_OK)
                die(std::string("rbrt_gpu: ") + rbrt_last_error());
        } else if (denoise && rbrt_gpu_denoise(width, height, hdr.data(), &ao, nullptr, nullptr, rgb.data(), nullptr) != RBRT_OK)   // on the first device
            die(std::string("rbrt_gpu: ") + rbrt_last_error());
    }
    rbrt_gpu_scene_destroy(scene);
    printf("Saving rendered image to %s\n", target.c_str());                        // main.rs:84
    if (!save_image(target, rgb, width, height)) die("Unable to save target img to " + target + "! Maybe the directory does not exist?");   // main.rs:86-91
    if (!aov.empty()) {
        const struct { const char* name; const std::vector<float>& v; int ch; } planes[] = {
            {"depth", depth, 1}, {"normal", normal, 3}, {"albedo", albedo, 3}, {"coverage", coverage, 1}};
        for (const auto& p : planes) {
            const std::string path = aov + "." + p.name + ".pfm";
            printf("Saving %s AOV to %s\n", p.name, path.c_str());
            if (!save_pfm(path, p.v.data(), width, height, p.ch)) die("Unable to save AOV to " + path + "! Maybe the directory does not exist?");
        }
    }
    fprintf(stderr, "[rbrt_b200] %llu rays, %llu samples in %.1f ms on %u GPU%s (%.1f Mrays/s)\n", (unsigned long long)st.rays,
            (unsigned long long)st.paths, st.ms_device, gpus, gpus > 1 ? "s" : "", st.ms_device > 0 ? st.rays / st.ms_device / 1e3 : 0.0);
    return 0;
}
