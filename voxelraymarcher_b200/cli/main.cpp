// VoxelRaymarcher CLI over the C ABI of libvrm_b200.so -- the reference's process-level seam (SURVEY.md §8b (1)):
//   VoxelRaymarcher <scale:int> <hashtable|vcs> <original|longestaxis>        (main/Main.cu:176-229, SURVEY.md F1)
// Same positional arguments, defaults (anything but the exact strings selects VCS / Longest Axis), prints, fixed
// 1920x1080 frame and camera, `resources/scene.vox` input and `output.png` output as the reference.  Extras (all optional,
// after the positional arguments): --scene PATH --out PATH --width W --height H --dump-voxels PATH (write the loaded voxel list as text and exit;
// no device needed) --depth PATH (also write the frame's depth, vrm_hit_surface_views: world distance from the camera per pixel, +inf where
// the ray hit nothing, as a little-endian grayscale PFM).
//
// Scene file: the reference's text format, one `x,y,z,color` line per voxel (geometry/VoxelFile.cuh:9-35); files that
// start with the magic "VOX " are read as MagicaVoxel binaries instead (north star; the reference itself has no such
// reader, so only the text path has reference semantics to match).
#include "../../include/vrm_b200.h"

#include <cerrno>
#include <climits>
#include <cstdint>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <string>
#include <vector>

namespace
{

// ---- scene readers ---------------------------------------------------------------------------------------------
// The reference's text scene (geometry/VoxelFile.cuh:9-35): one voxel per line, fields separated by commas, EMPTY fields do
// not count ("1,,2" has two fields), a line needs more than three fields, the first four are x, y, z, colour.  Numbers are read
// the way std::stoi reads them there: leading white space, an optional sign, decimal digits, anything behind them ignored.  A
// field without digits or outside int's range ends the reference with an uncaught exception; here it is reported and the load fails.
bool parseStoi(const char* first, const char* last, int32_t& out)
{
	std::string field(first, last);  // NUL-terminated copy for strtol
	char* stop = nullptr;
	errno = 0;
	const long v = std::strtol(field.c_str(), &stop, 10);
	if (stop == field.c_str() || errno == ERANGE || v < INT32_MIN || v > INT32_MAX) return false;
	out = static_cast<int32_t>(v);
	return true;
}

bool readCsvScene(const std::vector<uint8_t>& bytes, std::vector<int32_t>& xyz, std::vector<uint32_t>& rgb)
{
	const char* p = reinterpret_cast<const char*>(bytes.data());
	const char* const fileEnd = p + bytes.size();
	size_t lineNo = 0;
	while (p < fileEnd)
	{
		const char* eol = static_cast<const char*>(memchr(p, '\n', size_t(fileEnd - p)));
		const char* lineEnd = eol ? eol : fileEnd;
		lineNo++;
		const char* fieldAt[4];
		const char* fieldEnd[4];
		size_t fields = 0;
		for (const char* q = p; q < lineEnd;)
		{
			if (*q == ',') { q++; continue; }
			const char* e = q;
			while (e < lineEnd && *e != ',') e++;
			if (fields < 4) { fieldAt[fields] = q; fieldEnd[fields] = e; }
			fields++;
			q = e;
		}
		if (fields > 3)
		{
			int32_t v[4];
			for (int i = 0; i < 4; i++)
				if (!parseStoi(fieldAt[i], fieldEnd[i], v[i])) { std::cout << "ERROR: scene file line " << lineNo << ": field " << i + 1 << " is not an integer" << std::endl; return false; }
			xyz.push_back(v[0]); xyz.push_back(v[1]); xyz.push_back(v[2]);
			rgb.push_back(static_cast<uint32_t>(v[3]));
		}
		p = eol ? eol + 1 : fileEnd;
	}
	return true;
}

uint32_t rd32(const std::vector<uint8_t>& b, size_t o) { return b[o] | (b[o + 1] << 8) | (b[o + 2] << 16) | (uint32_t(b[o + 3]) << 24); }

// MagicaVoxel .vox (version 150/200): MAIN > (SIZE, XYZI)*, optional RGBA palette, optional scene graph (nTRN transform, nGRP
// group, nSHP shape nodes).  MagicaVoxel is z-up; the raymarcher is y-up, so (x, y, z)_vox -> (x, z, y).
//  * No scene graph (old files, single models): every model sits at the origin with its own coordinates.
//  * Scene graph: a model instance is placed by the transforms on the path from the root to its shape node -- frame 0's
//    translation `_t` and rotation `_r` (a signed permutation matrix packed in one byte) -- applied about the model's centre
//    floor(size / 2), voxel centres rotated, as MagicaVoxel does; a model referenced by several shape nodes appears once per node.
struct VoxModel { uint32_t size[3] = {0, 0, 0}; std::vector<uint8_t> xyzi; };
struct VoxXform { int r[3][3]; int64_t t[3]; };
struct VoxNode { int kind = 0; int child = -1; std::vector<int> children; std::vector<int> models; VoxXform x; };  // kind 1 nTRN, 2 nGRP, 3 nSHP

struct VoxReader
{
	const std::vector<uint8_t>& b;
	size_t pos, end;
	bool ok = true;
	VoxReader(const std::vector<uint8_t>& bytes, size_t from, size_t to) : b(bytes), pos(from), end(to) {}
	uint32_t u32() { if (pos + 4 > end) { ok = false; pos = end; return 0; } const uint32_t v = rd32(b, pos); pos += 4; return v; }
	std::string str() { const uint32_t n = u32(); if (!ok || pos + n > end) { ok = false; pos = end; return {}; } std::string s(reinterpret_cast<const char*>(b.data() + pos), n); pos += n; return s; }
	void dict(std::vector<std::pair<std::string, std::string>>& out) { const uint32_t n = u32(); for (uint32_t i = 0; ok && i < n; i++) { std::string k = str(), v = str(); out.emplace_back(k, v); } }
};

VoxXform voxIdentity() { VoxXform x; for (int i = 0; i < 3; i++) { for (int j = 0; j < 3; j++) x.r[i][j] = i == j; x.t[i] = 0; } return x; }

VoxXform voxCompose(const VoxXform& parent, const VoxXform& child)  // parent o child
{
	VoxXform o;
	for (int i = 0; i < 3; i++)
	{
		for (int j = 0; j < 3; j++) { o.r[i][j] = 0; for (int k = 0; k < 3; k++) o.r[i][j] += parent.r[i][k] * child.r[k][j]; }
		o.t[i] = parent.t[i];
		for (int k = 0; k < 3; k++) o.t[i] += parent.r[i][k] * child.t[k];
	}
	return o;
}

void voxRotation(uint8_t packed, int r[3][3])
{
	// bits 0-1 / 2-3: column of the non-zero entry of rows 0 / 1 (row 2 takes the remaining column); bits 4, 5, 6: the rows' signs
	const int c0 = packed & 3, c1 = (packed >> 2) & 3;
	int c2 = 3 - c0 - c1;
	if (c0 > 2 || c1 > 2 || c0 == c1 || c2 < 0 || c2 > 2) { for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) r[i][j] = i == j; return; }
	for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) r[i][j] = 0;
	r[0][c0] = (packed & 16) ? -1 : 1; r[1][c1] = (packed & 32) ? -1 : 1; r[2][c2] = (packed & 64) ? -1 : 1;
}

bool readMagicaVoxel(const std::vector<uint8_t>& b, std::vector<int32_t>& xyz, std::vector<uint32_t>& rgb)
{
	if (b.size() < 20 || memcmp(b.data(), "VOX ", 4) != 0 || memcmp(b.data() + 8, "MAIN", 4) != 0) return false;
	std::vector<uint32_t> palette(256);
	for (int i = 0; i < 256; i++) palette[i] = 0x010101u * uint32_t(i);  // grey ramp unless an RGBA chunk follows
	std::vector<VoxModel> models;
	std::vector<VoxNode> nodes;
	uint32_t pendingSize[3] = {0, 0, 0};
	size_t pos = 20;
	while (pos + 12 <= b.size())
	{
		const char* id = reinterpret_cast<const char*>(b.data() + pos);
		const uint32_t n = rd32(b, pos + 4);
		const size_t body = pos + 12;
		if (body + n > b.size()) break;
		if (memcmp(id, "SIZE", 4) == 0 && n >= 12) { for (int i = 0; i < 3; i++) pendingSize[i] = rd32(b, body + 4 * size_t(i)); }
		else if (memcmp(id, "XYZI", 4) == 0 && n >= 4)
		{
			VoxModel m;
			for (int i = 0; i < 3; i++) m.size[i] = pendingSize[i];
			const uint32_t count = rd32(b, body);
			const size_t have = (n - 4) / 4;
			m.xyzi.assign(b.begin() + long(body + 4), b.begin() + long(body + 4 + 4 * std::min<size_t>(count, have)));
			models.push_back(std::move(m));
		}
		else if (memcmp(id, "RGBA", 4) == 0 && n >= 1024)
		{
			for (int i = 0; i < 255; i++)  // palette entry i is stored at index i+1
			{
				const uint8_t* c = b.data() + body + 4 * size_t(i);
				palette[i + 1] = (uint32_t(c[0]) << 16) | (uint32_t(c[1]) << 8) | c[2];
			}
		}
		else if (memcmp(id, "nTRN", 4) == 0 || memcmp(id, "nGRP", 4) == 0 || memcmp(id, "nSHP", 4) == 0)
		{
			VoxReader r(b, body, body + n);
			const uint32_t nodeId = r.u32();
			std::vector<std::pair<std::string, std::string>> attrs;
			r.dict(attrs);
			VoxNode node;
			node.x = voxIdentity();
			if (id[1] == 'T')
			{
				node.kind = 1;
				node.child = int(r.u32());
				r.u32(); r.u32();  // reserved id, layer id
				const uint32_t frames = r.u32();
				for (uint32_t f = 0; r.ok && f < frames; f++)
				{
					std::vector<std::pair<std::string, std::string>> frame;
					r.dict(frame);
					if (f != 0) continue;  // animation frames other than the first are ignored
					for (const auto& kv : frame)
					{
						if (kv.first == "_t") { long long tx = 0, ty = 0, tz = 0; if (sscanf(kv.second.c_str(), "%lld %lld %lld", &tx, &ty, &tz) == 3) { node.x.t[0] = tx; node.x.t[1] = ty; node.x.t[2] = tz; } }
						else if (kv.first == "_r") voxRotation(uint8_t(std::strtoul(kv.second.c_str(), nullptr, 10)), node.x.r);
					}
				}
			}
			else if (id[1] == 'G')
			{
				node.kind = 2;
				const uint32_t kids = r.u32();
				for (uint32_t k = 0; r.ok && k < kids; k++) node.children.push_back(int(r.u32()));
			}
			else
			{
				node.kind = 3;
				const uint32_t count = r.u32();
				for (uint32_t k = 0; r.ok && k < count; k++)
				{
					node.models.push_back(int(r.u32()));
					std::vector<std::pair<std::string, std::string>> modelAttrs;
					r.dict(modelAttrs);
				}
			}
			if (r.ok && nodeId < (1u << 20))
			{
				if (nodes.size() <= nodeId) nodes.resize(nodeId + 1);
				nodes[nodeId] = node;
			}
		}
		pos = body + n;  // children of MAIN follow in line (the chunk's child size is the size of MAIN's children, not skipped)
	}
	auto emit = [&](const VoxModel& m, const VoxXform* x) {
		for (size_t i = 0; i + 4 <= m.xyzi.size(); i += 4)
		{
			const uint8_t* v = m.xyzi.data() + i;
			int64_t w[3] = {v[0], v[1], v[2]};
			if (x)
			{
				// voxel centre relative to the model's centre, in half voxels (exact), rotated, halved with floor, translated
				const int64_t c2[3] = {2 * int64_t(v[0]) + 1 - int64_t(m.size[0]), 2 * int64_t(v[1]) + 1 - int64_t(m.size[1]), 2 * int64_t(v[2]) + 1 - int64_t(m.size[2])};
				for (int a = 0; a < 3; a++)
				{
					const int64_t r2 = x->r[a][0] * c2[0] + x->r[a][1] * c2[1] + x->r[a][2] * c2[2];
					w[a] = (r2 >= 0 ? r2 / 2 : -((-r2 + 1) / 2)) + x->t[a];
				}
			}
			xyz.push_back(int32_t(w[0])); xyz.push_back(int32_t(w[2])); xyz.push_back(int32_t(w[1]));  // z-up -> y-up
			rgb.push_back(palette[v[3]]);
		}
	};
	bool graph = false;
	for (const VoxNode& nd : nodes) graph = graph || nd.kind == 3;
	if (!graph || nodes.empty() || nodes[0].kind == 0)
	{
		for (const VoxModel& m : models) emit(m, nullptr);
		return true;
	}
	// depth-first walk from node 0 (explicit stack; a malformed file cannot recurse without bound: at most nodes.size() levels)
	struct Item { int node; VoxXform x; size_t depth; };
	std::vector<Item> stack;
	stack.push_back({0, voxIdentity(), 0});
	while (!stack.empty())
	{
		const Item it = stack.back();
		stack.pop_back();
		if (it.node < 0 || size_t(it.node) >= nodes.size() || it.depth > nodes.size()) continue;
		const VoxNode& nd = nodes[size_t(it.node)];
		if (nd.kind == 1) stack.push_back({nd.child, voxCompose(it.x, nd.x), it.depth + 1});
		else if (nd.kind == 2) { for (size_t k = nd.children.size(); k-- > 0;) stack.push_back({nd.children[k], it.x, it.depth + 1}); }
		else if (nd.kind == 3) { for (int mi : nd.models) if (mi >= 0 && size_t(mi) < models.size()) emit(models[size_t(mi)], &it.x); }
	}
	return true;
}

// ---- PNG writer (8-bit RGB, stored deflate blocks; stands in for stbi_write_png, images/ImageWriter.cpp:8-16) ------------
uint32_t crcTable[256];
void initCrc()
{
	for (uint32_t n = 0; n < 256; n++)
	{
		uint32_t c = n;
		for (int k = 0; k < 8; k++) c = (c & 1) ? 0xEDB88320u ^ (c >> 1) : c >> 1;
		crcTable[n] = c;
	}
}
uint32_t crc32(const uint8_t* p, size_t n, uint32_t c = 0xFFFFFFFFu)
{
	for (size_t i = 0; i < n; i++) c = crcTable[(c ^ p[i]) & 0xFF] ^ (c >> 8);
	return c;
}
void put32(std::vector<uint8_t>& v, uint32_t x) { v.push_back(x >> 24); v.push_back(x >> 16); v.push_back(x >> 8); v.push_back(x); }
void chunk(std::vector<uint8_t>& out, const char* type, const std::vector<uint8_t>& data)
{
	put32(out, uint32_t(data.size()));
	size_t at = out.size();
	out.insert(out.end(), type, type + 4);
	out.insert(out.end(), data.begin(), data.end());
	put32(out, crc32(out.data() + at, out.size() - at) ^ 0xFFFFFFFFu);
}
bool writePng(const std::string& path, const uint8_t* rgb, uint32_t w, uint32_t h)
{
	initCrc();
	std::vector<uint8_t> raw;
	raw.reserve(size_t(h) * (size_t(w) * 3 + 1));
	for (uint32_t y = 0; y < h; y++)
	{
		raw.push_back(0);  // filter: none
		raw.insert(raw.end(), rgb + size_t(y) * w * 3, rgb + size_t(y + 1) * w * 3);
	}
	std::vector<uint8_t> z = {0x78, 0x01};
	uint32_t a = 1, b = 0;
	for (size_t off = 0; off < raw.size() || off == 0; off += 65535)
	{
		size_t n = std::min<size_t>(65535, raw.size() - off);
		bool last = off + n >= raw.size();
		z.push_back(last ? 1 : 0);
		z.push_back(n & 0xFF); z.push_back(n >> 8); z.push_back(~n & 0xFF); z.push_back((~n >> 8) & 0xFF);
		z.insert(z.end(), raw.begin() + off, raw.begin() + off + n);
		for (size_t i = 0; i < n; i++) { a = (a + raw[off + i]) % 65521; b = (b + a) % 65521; }
		if (last) break;
	}
	put32(z, (b << 16) | a);
	std::vector<uint8_t> out = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
	std::vector<uint8_t> ihdr;
	put32(ihdr, w); put32(ihdr, h);
	ihdr.push_back(8); ihdr.push_back(2); ihdr.push_back(0); ihdr.push_back(0); ihdr.push_back(0);
	chunk(out, "IHDR", ihdr);
	chunk(out, "IDAT", z);
	chunk(out, "IEND", {});
	std::ofstream f(path, std::ios::binary);
	f.write(reinterpret_cast<const char*>(out.data()), std::streamsize(out.size()));
	return bool(f);
}

// Grayscale PFM ("Pf", scale -1 = little-endian floats); PFM stores the bottom row first, the frame has row 0 at the top.
bool writePfm(const std::string& path, const float* depth, uint32_t w, uint32_t h)
{
	std::ofstream f(path, std::ios::binary);
	f << "Pf\n" << w << ' ' << h << "\n-1.0\n";
	for (uint32_t y = h; y-- > 0;)
		for (uint32_t x = 0; x < w; x++)
		{
			uint32_t bits;
			memcpy(&bits, depth + size_t(y) * w + x, 4);
			const char le[4] = {char(bits), char(bits >> 8), char(bits >> 16), char(bits >> 24)};
			f.write(le, 4);
		}
	return bool(f);
}

}  // namespace

int main(int argc, char* argv[])
{
	if (argc <= 1)  // Main.cu:181-185
	{
		std::cout << "You need to provide a voxel scale" << std::endl;
		return 1;
	}
	int32_t scale = std::stoi(argv[1]);
	int storage = VRM_STORAGE_VCS, algorithm = VRM_ALGO_LONGEST_AXIS;
	if (argc > 2 && std::strcmp(argv[2], "hashtable") == 0) { std::cout << "Storage Type: Cuckoo Hash Table" << std::endl; storage = VRM_STORAGE_HASHTABLE; }  // Main.cu:45-55
	else std::cout << "Storage Type: Voxel Cluster Storage" << std::endl;
	if (argc > 3 && std::strcmp(argv[3], "original") == 0) { std::cout << "Raymarching Algorithm: Original" << std::endl; algorithm = VRM_ALGO_ORIGINAL; }  // Main.cu:58-68
	else std::cout << "Raymarching Algorithm: Longest Axis" << std::endl;
	std::string scenePath = "resources/scene.vox", outPath = "output.png", depthPath;  // Main.cu:99,170; VoxelFile.cuh:12
	uint32_t width = 1920, height = 1080;                                   // Main.cu:195-196
	for (int i = 4; i + 1 < argc; i += 2)
	{
		if (!std::strcmp(argv[i], "--scene")) scenePath = argv[i + 1];
		else if (!std::strcmp(argv[i], "--out")) outPath = argv[i + 1];
		else if (!std::strcmp(argv[i], "--width")) width = uint32_t(std::stoul(argv[i + 1]));
		else if (!std::strcmp(argv[i], "--height")) height = uint32_t(std::stoul(argv[i + 1]));
		else if (!std::strcmp(argv[i], "--depth")) depthPath = argv[i + 1];
	}

	std::string dumpPath;
	for (int i = 4; i + 1 < argc; i += 2) if (!std::strcmp(argv[i], "--dump-voxels")) dumpPath = argv[i + 1];

	// the scene file is read before the device is touched (a malformed file fails without one; --dump-voxels needs none)
	std::vector<int32_t> xyz;
	std::vector<uint32_t> rgb;
	{
		std::ifstream f(scenePath, std::ios::binary);
		std::vector<uint8_t> bytes((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
		bool loaded = true;
		if (bytes.size() >= 4 && memcmp(bytes.data(), "VOX ", 4) == 0) loaded = readMagicaVoxel(bytes, xyz, rgb);
		else loaded = readCsvScene(bytes, xyz, rgb);  // a missing file yields an empty scene, as in the reference
		if (!loaded) { std::cout << "ERROR: could not read " << scenePath << std::endl; return EXIT_FAILURE; }
	}
	if (!dumpPath.empty())
	{
		// the loaded voxel list in the reference's text format, in load order (tests; converting a MagicaVoxel file for the reference)
		std::ofstream out(dumpPath);
		for (size_t i = 0; i < rgb.size(); i++) out << xyz[3 * i] << ',' << xyz[3 * i + 1] << ',' << xyz[3 * i + 2] << ',' << rgb[i] << '\n';
		return out ? EXIT_SUCCESS : EXIT_FAILURE;
	}

	char name[256] = "";
	int devCount = vrm_device_count();  // pickCudaDevice, Main.cu:82-94
	printf("Device Count: %d\n", devCount);
	if (devCount) vrm_device_name(0, name, sizeof(name));
	printf("Device: %s\n", name);

	vrm_scene* scene = nullptr;
	int rc = vrm_scene_create(0, &scene);
	if (rc != VRM_OK) { std::cout << "ERROR: " << vrm_error_string(rc) << " (a CUDA device is required)" << std::endl; return EXIT_FAILURE; }

	rc = vrm_scene_add_voxels(scene, xyz.data(), rgb.data(), rgb.size());
	float buildMs = 0.0f;
	if (rc == VRM_OK) rc = vrm_scene_build(scene, storage, &buildMs);
	if (rc != VRM_OK) { std::cout << "ERROR: " << vrm_error_string(rc) << ": " << vrm_last_error(scene) << std::endl; return EXIT_FAILURE; }
	uint32_t diameter = 0, filled = 0;
	int32_t minCoord = 0;
	vrm_scene_info(scene, &diameter, &minCoord, &filled, nullptr, nullptr);
	std::cout << "There are : " << filled << "/" << diameter * diameter * diameter << " regions that are filled" << std::endl;  // VoxelSceneCPU.cuh:54
	std::cout << "Storage Structures Generated" << std::endl;                                                                  // VoxelSceneCPU.cuh:86

	float origin[3] = {6.0f, 2.0f, 6.0f}, lookAt[3] = {0.0f, 0.0f, -1.0f}, up[3] = {0.0f, 1.0f, 0.0f}, cam[VRM_CAMERA_FLOATS];  // Main.cu:199
	float aspect = static_cast<float>(width) / static_cast<float>(height);
	vrm_camera_make(origin, lookAt, up, 60.0f, aspect, cam);
	float translation[3] = {0.0f, 0.0f, 0.0f}, kernelMs = 0.0f;  // Main.cu:215
	std::vector<uint8_t> frame(size_t(width) * height * 3);
	std::vector<int32_t> hits(depthPath.empty() ? 0 : size_t(width) * height * 4);
	rc = vrm_render(scene, cam, translation, uint32_t(scale), algorithm, width, height, frame.data(), depthPath.empty() ? nullptr : hits.data(), &kernelMs);
	std::cout << (rc == VRM_OK ? "no error" : vrm_last_error(scene)) << std::endl;  // cudaGetErrorString(cudaPeekAtLastError()), Main.cu:154-155
	std::cout << "Execution Time for Ray Marching Algorithm is: " << static_cast<long long>(kernelMs * 1000.0f) << " microseconds" << std::endl;  // Main.cu:162
	if (rc == VRM_OK && !writePng(outPath, frame.data(), width, height)) std::cout << "ERROR: Failed to write image to: " << outPath << std::endl;  // ImageWriter.cpp:11-14
	if (rc == VRM_OK && !depthPath.empty())
	{
		std::vector<float> depth(size_t(width) * height);
		rc = vrm_hit_surface_views(scene, cam, 1, translation, uint32_t(scale), width, height, hits.data(), depth.data(), nullptr);
		if (rc != VRM_OK) std::cout << "ERROR: " << vrm_error_string(rc) << ": " << vrm_last_error(scene) << std::endl;
		else if (!writePfm(depthPath, depth.data(), width, height)) std::cout << "ERROR: Failed to write depth to: " << depthPath << std::endl;
	}
	vrm_scene_destroy(scene);
	return rc == VRM_OK ? EXIT_SUCCESS : EXIT_FAILURE;
}
