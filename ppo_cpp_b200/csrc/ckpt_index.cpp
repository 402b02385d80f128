// `<prefix>.index` of the TensorFlow Saver-V2 bundle that PPO2::save writes (reference ppo2/ppo2.hpp:107-131 runs the graph's
// `save/control_dependency` op; TensorFlow 1.14's BundleWriter produces `<prefix>.index` + `<prefix>.data-00000-of-00001`).
// Without the index neither the reference (ppo2.hpp:169-189, `save/restore_all`) nor TensorFlow can read our checkpoints back.
//
// The index is a LevelDB-format table (TensorFlow's lib/io/table_builder: block restart interval 16, no compression):
//   data block   key ""            -> BundleHeaderProto  { num_shards = 1, version { producer = 1 } }   (little endian = default)
//                key <tensor name> -> BundleEntryProto   { dtype = DT_FLOAT, shape, offset, size, crc32c (masked, of the tensor bytes) }
//                keys ascending and prefix-compressed against their predecessor; ONE restart point (16 entries = one interval)
//   meta-index   empty block
//   index block  one entry: shortest separator after the last key ("n" for "model/...") -> handle (offset, size) of the data block
//   footer       handles of the meta-index and index blocks, zero padding to 40 bytes, magic 0xdb4775248b80fb57
// every block is followed by a 5-byte trailer: compression type 0 + masked CRC-32C of (block bytes + type byte).
// Pinned byte for byte on the checkpoint the reference ships (resources/ppo_cl/*.pkl.71.index, 498 bytes) by tests/test_abi_cpu.py.
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "meta_parser.h"

namespace ppo {
namespace {

uint32_t crc32c(const uint8_t* p, size_t n) {  // Castagnoli polynomial, reflected (0x82F63B78), as LevelDB / TensorFlow
    static uint32_t table[256];
    static bool init = false;
    if (!init) {
        for (uint32_t i = 0; i < 256; ++i) {
            uint32_t c = i;
            for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ 0x82F63B78u : c >> 1;
            table[i] = c;
        }
        init = true;
    }
    uint32_t c = 0xFFFFFFFFu;
    for (size_t i = 0; i < n; ++i) c = table[(c ^ p[i]) & 0xFFu] ^ (c >> 8);
    return c ^ 0xFFFFFFFFu;
}
uint32_t mask_crc(uint32_t c) { return ((c >> 15) | (c << 17)) + 0xa282ead8u; }

void put_varint(std::string& s, uint64_t v) {
    while (v >= 0x80u) {
        s.push_back((char)(v | 0x80u));
        v >>= 7;
    }
    s.push_back((char)v);
}
void put_fixed32(std::string& s, uint32_t v) {
    for (int i = 0; i < 4; ++i) s.push_back((char)((v >> (8 * i)) & 0xFFu));
}

// one table block: entries (shared | unshared | value length as varints, key suffix, value), restart offsets, restart count
struct Block {
    std::string buf, last;
    int n = 0;
    std::vector<uint32_t> restarts{0};
    void add(const std::string& key, const std::string& value) {
        size_t shared = 0;
        if (n % 16 == 0 && n > 0) restarts.push_back((uint32_t)buf.size());
        else if (n > 0)
            while (shared < last.size() && shared < key.size() && last[shared] == key[shared]) ++shared;
        put_varint(buf, shared);
        put_varint(buf, key.size() - shared);
        put_varint(buf, value.size());
        buf.append(key, shared, std::string::npos);
        buf.append(value);
        last = key;
        ++n;
    }
    std::string finish() const {
        std::string out = buf;
        for (uint32_t r : restarts) put_fixed32(out, r);
        put_fixed32(out, (uint32_t)restarts.size());
        return out;
    }
};

// appends block + trailer to the file image, returns the block's handle (offset, size without the trailer) as two varints
std::string emit(std::string& file, const std::string& block) {
    std::string handle;
    put_varint(handle, file.size());
    put_varint(handle, block.size());
    std::string with_type = block;
    with_type.push_back('\0');  // kNoCompression
    file.append(with_type);
    put_fixed32(file, mask_crc(crc32c(reinterpret_cast<const uint8_t*>(with_type.data()), with_type.size())));
    return handle;
}

// leveldb BytewiseComparator::FindShortSuccessor: the first byte that can be incremented, incremented, the rest dropped
std::string short_successor(const std::string& key) {
    for (size_t i = 0; i < key.size(); ++i)
        if ((uint8_t)key[i] != 0xFFu) {
            std::string s = key.substr(0, i + 1);
            s[i] = (char)((uint8_t)s[i] + 1);
            return s;
        }
    return key;
}

}  // namespace

// Tensors in ascending name order; `data` is the payload of the .data file in the same order (sizes follow from the shapes).
std::string bundle_index_image(const std::vector<std::string>& names, const std::vector<std::vector<int64_t>>& shapes, const float* data) {
    Block db;
    {
        std::string header;  // BundleHeaderProto
        header.push_back((char)0x08); put_varint(header, 1);          // num_shards = 1
        header.push_back((char)0x1a); put_varint(header, 2);          // version { producer = 1 }
        header.push_back((char)0x08); put_varint(header, 1);
        db.add("", header);
    }
    uint64_t offset = 0;
    for (size_t i = 0; i < names.size(); ++i) {
        uint64_t count = 1;
        std::string shape;  // TensorShapeProto: repeated Dim dim = 2 { int64 size = 1 }
        for (int64_t dsz : shapes[i]) {
            std::string dim;
            dim.push_back((char)0x08); put_varint(dim, (uint64_t)dsz);
            shape.push_back((char)0x12); put_varint(shape, dim.size()); shape.append(dim);
            count *= (uint64_t)dsz;
        }
        const uint64_t bytes = count * sizeof(float);
        std::string e;  // BundleEntryProto (zero-valued fields are not written: shard_id always, offset of the first tensor)
        e.push_back((char)0x08); put_varint(e, 1);  // dtype = DT_FLOAT
        e.push_back((char)0x12); put_varint(e, shape.size()); e.append(shape);
        if (offset != 0) { e.push_back((char)0x20); put_varint(e, offset); }
        e.push_back((char)0x28); put_varint(e, bytes);
        e.push_back((char)0x35);
        put_fixed32(e, mask_crc(crc32c(reinterpret_cast<const uint8_t*>(data) + offset, bytes)));
        db.add(names[i], e);
        offset += bytes;
    }
    std::string file;
    const std::string data_handle = emit(file, db.finish());
    const std::string meta_handle = emit(file, Block().finish());
    Block ib;
    ib.add(short_successor(db.last), data_handle);
    const std::string index_handle = emit(file, ib.finish());
    std::string footer = meta_handle + index_handle;
    footer.resize(40, '\0');
    const uint64_t magic = 0xdb4775248b80fb57ull;
    put_fixed32(footer, (uint32_t)(magic & 0xFFFFFFFFu));
    put_fixed32(footer, (uint32_t)(magic >> 32));
    return file + footer;
}

// The 15 model tensors of an MLP [h1, h2] policy in checkpoint (ascending name) order with their TF shapes; 14 without
// model/pi/logstd for a categorical head (Discrete action space).
void model_bundle_layout(int obs_dim, int act_dim, int h1, int h2, bool discrete, std::vector<std::string>& names,
                         std::vector<std::vector<int64_t>>& shapes) {
    const int64_t O = obs_dim, A = act_dim, H1 = h1, H2 = h2;
    names = {"model/pi/b", "model/pi/logstd", "model/pi/w", "model/pi_fc0/b", "model/pi_fc0/w", "model/pi_fc1/b", "model/pi_fc1/w", "model/q/b",
             "model/q/w", "model/vf/b", "model/vf/w", "model/vf_fc0/b", "model/vf_fc0/w", "model/vf_fc1/b", "model/vf_fc1/w"};
    shapes = {{A}, {1, A}, {H2, A}, {H1}, {O, H1}, {H2}, {H1, H2}, {A}, {H2, A}, {1}, {H2, 1}, {H1}, {O, H1}, {H2}, {H1, H2}};
    if (discrete) {
        names.erase(names.begin() + 1);
        shapes.erase(shapes.begin() + 1);
    }
}

int write_index(const char* prefix, int obs_dim, int act_dim, int hidden1, int hidden2, bool discrete, const float* data, size_t n_floats) {
    if (!prefix || !data || obs_dim < 1 || act_dim < 1 || hidden1 < 1 || hidden2 < 1) return -1;  // PPO_ERR_INVALID
    std::vector<std::string> names;
    std::vector<std::vector<int64_t>> shapes;
    model_bundle_layout(obs_dim, act_dim, hidden1, hidden2, discrete, names, shapes);
    size_t total = 0;
    for (const auto& s : shapes) {
        size_t c = 1;
        for (int64_t d : s) c *= (size_t)d;
        total += c;
    }
    if (total != n_floats) return -1;
    const std::string image = ppo::bundle_index_image(names, shapes, data);
    const std::string path = std::string(prefix) + ".index";
    FILE* f = fopen(path.c_str(), "wb");
    if (!f) return -3;  // PPO_ERR_IO
    const size_t put = fwrite(image.data(), 1, image.size(), f);
    fclose(f);
    return put == image.size() ? 0 : -3;
}

}  // namespace ppo

extern "C" int ppo_checkpoint_write_index(const char* prefix, int obs_dim, int act_dim, int hidden1, int hidden2, const float* data, size_t n_floats) {
    return ppo::write_index(prefix, obs_dim, act_dim, hidden1, hidden2, false, data, n_floats);
}
extern "C" int ppo_checkpoint_write_index_ex(const char* prefix, int action_space, int obs_dim, int act_dim, int hidden1, int hidden2,
                                             const float* data, size_t n_floats) {
    if (action_space != 0 && action_space != 1) return -1;  // PPO_ERR_INVALID
    return ppo::write_index(prefix, obs_dim, act_dim, hidden1, hidden2, action_space == 1, data, n_floats);
}
