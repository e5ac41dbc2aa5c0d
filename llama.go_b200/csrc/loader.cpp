// loader.cpp — ggjt v1 model files straight into HBM (SURVEY.md §8f-3).
//
// Same file format and acceptance rules as the reference loader (pkg/llama/llama.go:712-976,
// written by scripts/convert-pth-to-ggml.py): magic 0x67676a74, version 1, 7 hyper-parameters,
// vocab records, then tensor records {n_dims, name_len, dtype, ne[n_dims], name, pad to 32, data}
// until EOF; F32 and F16 only (F16 widened to FP32 on the device, llama.go:938-941); unknown tensor
// names abort (llama.go:906-910).  Differences in mechanism, not in result: the file is memory-mapped
// and every tensor goes host -> HBM through two pinned staging buffers on a copy stream (the
// reference reads F16 tensors with one 2-byte Read per element); with LB_TYPE_Q8_0 the MulMat
// matrices are block-quantised on the device as they arrive; with LB_TYPE_F16 they keep F16 data byte
// for byte (streamed straight into place) and F32 data is rounded to nearest even on the device.
#include <fcntl.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <memory>

#include "llama.hpp"

namespace lb {
namespace llama {

namespace {
struct Mapped {
    const uint8_t *p = nullptr;
    size_t n = 0;
    int fd = -1;
    ~Mapped() {
        if (p) munmap(const_cast<uint8_t *>(p), n);
        if (fd >= 0) close(fd);
    }
};
struct Reader {
    const uint8_t *p;
    size_t n, off = 0;
    bool has(size_t k) const { return off + k <= n; }
    uint32_t u32() {
        LB_CHECK(has(4), "Invalid model file: truncated");
        uint32_t v;
        memcpy(&v, p + off, 4);
        off += 4;
        return v;
    }
};
}  // namespace

LoadedModel load_ggjt(const std::string &path, int device, uint32_t layer_begin, uint32_t layer_end_or_0, int weight_type) {
    Mapped mf;
    mf.fd = open(path.c_str(), O_RDONLY);
    LB_CHECK(mf.fd >= 0, "Failed to load model '" + path + "'");
    struct stat st;
    LB_CHECK(fstat(mf.fd, &st) == 0 && st.st_size > 36, "Invalid model file '" + path + "'");
    mf.n = (size_t)st.st_size;
    void *mp = mmap(nullptr, mf.n, PROT_READ, MAP_PRIVATE, mf.fd, 0);
    LB_CHECK(mp != MAP_FAILED, "mmap failed for '" + path + "'");
    mf.p = static_cast<const uint8_t *>(mp);
    madvise(mp, mf.n, MADV_SEQUENTIAL);

    Reader r{mf.p, mf.n};
    const uint32_t magic = r.u32();
    LB_CHECK(magic != 0x67676d6cu && magic != 0x67676d66u, "Invalid model file '" + path + "'! Too old, regenerate!");  // llama.go:724
    LB_CHECK(magic == 0x67676a74u, "Invalid model file '" + path + "'! Wrong MAGIC in header");                         // llama.go:729
    LB_CHECK(r.u32() == 1u, "Invalid model file '" + path + "'! Unsupported version");                                  // llama.go:736
    HParams hp;
    hp.vocab = r.u32(); hp.dim = r.u32(); hp.mult = r.u32(); hp.heads = r.u32(); hp.layers = r.u32();
    (void)r.u32();  // rot (obsolete)
    (void)r.u32();  // ftype
    LoadedModel out;
    out.vocab.reserve(hp.vocab);
    for (uint32_t i = 0; i < hp.vocab; i++) {  // llama.go:799-811
        const uint32_t len = r.u32();
        LB_CHECK(r.has((size_t)len + 4), "Invalid model file: truncated vocab");
        out.vocab.emplace_back(reinterpret_cast<const char *>(r.p + r.off), len);
        r.off += len;
        float score;
        memcpy(&score, r.p + r.off, 4);
        r.off += 4;
        out.scores.push_back(score);
    }
    const uint32_t layer_end = layer_end_or_0 ? layer_end_or_0 : hp.layers;
    out.model.reset(new Model(hp, device, layer_begin, layer_end, weight_type));
    Model &m = *out.model;
    LB_CUDA(cudaSetDevice(device));

    // two pinned staging buffers + a copy stream: host page-in of chunk i+1 overlaps the H2D of chunk i
    constexpr size_t CHUNK = 64u << 20;
    void *pin[2] = {nullptr, nullptr};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    cudaStream_t cs = nullptr;
    void *dev_tmp = nullptr;
    size_t dev_tmp_bytes = 0;
    auto cleanup = [&]() {
        for (int i = 0; i < 2; i++) {
            if (pin[i]) cudaFreeHost(pin[i]);
            if (ev[i]) cudaEventDestroy(ev[i]);
        }
        if (cs) cudaStreamDestroy(cs);
        if (dev_tmp) cudaFree(dev_tmp);
    };
    try {
        LB_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            LB_CUDA(cudaMallocHost(&pin[i], CHUNK));
            LB_CUDA(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
        }
        int slot = 0;
        while (r.has(12)) {
            const uint32_t n_dims = r.u32();
            if (n_dims < 1 || n_dims > 2) break;  // llama.go:890-893
            const uint32_t name_len = r.u32();
            const uint32_t dtype = r.u32();
            uint64_t nelem = 1;
            for (uint32_t i = 0; i < n_dims; i++) nelem *= r.u32();
            LB_CHECK(r.has(name_len), "Invalid model file: truncated tensor name");
            const std::string name(reinterpret_cast<const char *>(r.p + r.off), name_len);
            r.off += name_len;
            r.off = (r.off + 31) & ~(size_t)31;  // data is 32-byte aligned in the file, llama.go:926-933
            LB_CHECK(Model::known_name(hp, name), "Unknown tensor '" + name + "' in model file");  // llama.go:906-910
            LB_CHECK(dtype == 0 || dtype == 1, "Tensor data type is not supported yet!");          // llama.go:956-958
            const size_t esz = dtype == 0 ? 4 : 2;
            const size_t nbytes = (size_t)nelem * esz;
            LB_CHECK(r.has(nbytes), "Failed to read BIG chunk from model!");                        // llama.go:951-955
            const uint8_t *src = r.p + r.off;
            r.off += nbytes;
            auto it = m.tensors.find(name);
            if (it == m.tensors.end()) continue;  // another pipeline stage's tensor
            const Model::Entry &e = it->second;
            LB_CHECK(e.nelem == nelem, "tensor '" + name + "' has the wrong size");
            // stored as it is in the file (FP32 into FP32, F16 into an F16 matrix): stream straight into place
            const bool direct = e.h ? dtype == 1 : (dtype == 0 && !e.q8.q);
            if (!direct && dev_tmp_bytes < nbytes + nelem * 4) {
                if (dev_tmp) { LB_CUDA(cudaStreamSynchronize(cs)); cudaFree(dev_tmp); dev_tmp = nullptr; }
                dev_tmp_bytes = nbytes + nelem * 4;
                LB_CUDA(cudaMalloc(&dev_tmp, dev_tmp_bytes));
            }
            uint8_t *raw_dst = !direct ? static_cast<uint8_t *>(dev_tmp) : e.h ? reinterpret_cast<uint8_t *>(e.h) : reinterpret_cast<uint8_t *>(e.ptr);
            for (size_t o = 0; o < nbytes; o += CHUNK) {
                const size_t c = nbytes - o < CHUNK ? nbytes - o : CHUNK;
                LB_CUDA(cudaEventSynchronize(ev[slot]));  // staging buffer free again
                memcpy(pin[slot], src + o, c);
                LB_CUDA(cudaMemcpyAsync(raw_dst + o, pin[slot], c, cudaMemcpyHostToDevice, cs));
                LB_CUDA(cudaEventRecord(ev[slot], cs));
                slot ^= 1;
            }
            if (!direct && e.h) {
                m.round_to_f16(static_cast<const float *>(dev_tmp), e.h, nelem, name, cs);   // synchronises cs: dev_tmp is reused
            } else if (!direct) {
                float *f32 = e.q8.q ? reinterpret_cast<float *>(static_cast<uint8_t *>(dev_tmp) + nbytes) : e.ptr;
                const float *quant_src = f32;
                if (dtype == 1) k::f16_to_f32(static_cast<const uint16_t *>(dev_tmp), f32, nelem, cs);
                else quant_src = static_cast<const float *>(dev_tmp);
                if (e.q8.q) k::quantize_q8(quant_src, e.q8.q, e.q8.d, (uint32_t)(nelem / e.cols), e.cols, cs);
                LB_CUDA(cudaStreamSynchronize(cs));  // dev_tmp is reused by the next tensor
            }
            out.tensors_loaded++;
        }
        LB_CUDA(cudaStreamSynchronize(cs));
    } catch (...) {
        cleanup();
        throw;
    }
    cleanup();
    return out;
}

}  // namespace llama
}  // namespace lb
