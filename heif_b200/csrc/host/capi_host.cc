// C ABI for the host-side parse layer (no CUDA in this translation unit).
#include <cstring>
#include <string>

#include "capi_common.h"
#include "heic_decoder.h"

namespace heic {
thread_local std::string g_last_error;
void set_last_error(const std::string& s) { g_last_error = s; }
}  // namespace heic

using namespace heic;

struct heic_b200_file {
  std::unique_ptr<HeicFile> f;
};

extern "C" {

int32_t heic_b200_abi_version(void) { return HEIC_B200_ABI_VERSION; }
const char* heic_b200_last_error(void) { return g_last_error.c_str(); }

int64_t heic_b200_remove_emulation_prevention(const uint8_t* data, size_t len, uint8_t* out,
                                              uint32_t* epb_pos, size_t epb_cap, size_t* n_epb) {
  return guard([&]() -> int64_t {
    if ((!data && len) || (!out && len)) bail(HEIC_E_INVALID_ARG, "null buffer");
    std::vector<uint32_t> epb;
    std::vector<uint8_t> v = RbspReader::remove_emulation_prevention(data, len, &epb);
    if (!v.empty()) std::memcpy(out, v.data(), v.size());
    if (n_epb) *n_epb = epb.size();
    if (epb_pos)
      for (size_t i = 0; i < epb.size() && i < epb_cap; ++i) epb_pos[i] = epb[i];
    return static_cast<int64_t>(v.size());
  });
}

static int64_t read_golomb(const uint8_t* data, size_t len, size_t* bit_pos, bool is_signed, void* out) {
  return guard([&]() -> int64_t {
    if (!data || !bit_pos || !out) bail(HEIC_E_INVALID_ARG, "null argument");
    RbspReader r(data, len);
    if (*bit_pos > len * 8) bail(HEIC_E_INVALID_ARG, "bit position beyond the buffer");
    r.read_bits(0);
    for (size_t i = 0; i < *bit_pos; ++i) r.read_bit();
    if (is_signed) *static_cast<int32_t*>(out) = r.read_se();
    else *static_cast<uint32_t*>(out) = r.read_ue();
    *bit_pos = r.byte_position() * 8 + r.bit_position();
    return 0;
  });
}
int32_t heic_b200_rbsp_read_ue(const uint8_t* data, size_t len, size_t* bit_pos, uint32_t* out) {
  return static_cast<int32_t>(read_golomb(data, len, bit_pos, false, out));
}
int32_t heic_b200_rbsp_read_se(const uint8_t* data, size_t len, size_t* bit_pos, int32_t* out) {
  return static_cast<int32_t>(read_golomb(data, len, bit_pos, true, out));
}

int32_t heic_b200_parse_sps(const uint8_t* rbsp, size_t len, heic_sps* out) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!rbsp || !out) bail(HEIC_E_INVALID_ARG, "null argument");
    *out = sequence_parameter_set_rbsp(rbsp, len);
    return 0;
  }));
}

int32_t heic_b200_parse_pps(const uint8_t* rbsp, size_t len, heic_pps* out) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!rbsp || !out) bail(HEIC_E_INVALID_ARG, "null argument");
    *out = picture_parameter_set_rbsp(rbsp, len);
    return 0;
  }));
}

int32_t heic_b200_parse_slice_header(const uint8_t* rbsp, size_t len, uint32_t nal_unit_type,
                                     const heic_sps* sps, const heic_pps* pps, const uint32_t* epb_pos,
                                     size_t n_epb, heic_slice_header* out) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!rbsp || !sps || !pps || !out || (n_epb && !epb_pos)) bail(HEIC_E_INVALID_ARG, "null argument");
    *out = slice_segment_header(rbsp, len, nal_unit_type, *sps, *pps, epb_pos, n_epb);
    return 0;
  }));
}

int32_t heic_b200_parse_slice_header_raw(const uint8_t* nal_payload, size_t len, uint32_t nal_unit_type, const heic_sps* sps,
                                         const heic_pps* pps, heic_slice_header* out) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!nal_payload || !sps || !pps || !out) bail(HEIC_E_INVALID_ARG, "null argument");
    *out = slice_segment_header_raw(nal_payload, len, nal_unit_type, *sps, *pps);
    return 0;
  }));
}

int32_t heic_b200_file_open(const uint8_t* data, size_t len, heic_b200_file** out) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!data || !out) bail(HEIC_E_INVALID_ARG, "null argument");
    auto h = std::make_unique<heic_b200_file>();
    h->f = HeicDecoder::open(data, len);
    *out = h.release();
    return 0;
  }));
}

void heic_b200_file_close(heic_b200_file* f) { delete f; }

const heic_image_desc* heic_b200_file_primary_image(const heic_b200_file* f) {
  return f ? &f->f->primary.desc : nullptr;
}
uint32_t heic_b200_file_aux_image_count(const heic_b200_file* f) {
  return f ? static_cast<uint32_t>(f->f->aux.size()) : 0;
}
const heic_image_desc* heic_b200_file_aux_image(const heic_b200_file* f, uint32_t i) {
  return (f && i < f->f->aux.size()) ? &f->f->aux[i]->desc : nullptr;
}
const heic_image_desc* heic_b200_file_primary_image_raw(const heic_b200_file* f) {
  return f ? &f->f->primary.desc_raw : nullptr;
}
const heic_image_desc* heic_b200_file_aux_image_raw(const heic_b200_file* f, uint32_t i) {
  return (f && i < f->f->aux.size()) ? &f->f->aux[i]->desc_raw : nullptr;
}
static const ImageStorage* image_of(const heic_b200_file* f, int32_t image) {
  if (!f) return nullptr;
  if (image < 0) return &f->f->primary;
  return static_cast<size_t>(image) < f->f->aux.size() ? f->f->aux[image].get() : nullptr;
}
int32_t heic_b200_file_parameter_set_nal(const heic_b200_file* f, int32_t image, uint32_t nal_unit_type,
                                         const uint8_t** data, size_t* len) {
  const ImageStorage* img = image_of(f, image);
  if (!img || !data || !len) {
    set_last_error("invalid argument");
    return HEIC_E_INVALID_ARG;
  }
  const std::vector<uint8_t>* v = nal_unit_type == 32 ? &img->vps_nal : nal_unit_type == 33 ? &img->sps_nal
                                  : nal_unit_type == 34 ? &img->pps_nal : nullptr;
  if (!v || v->empty()) {
    set_last_error("no such parameter set");
    return HEIC_E_INVALID_ARG;
  }
  *data = v->data();
  *len = v->size();
  return 0;
}
int32_t heic_b200_file_tile_nal(const heic_b200_file* f, int32_t image, uint32_t tile, const uint8_t** data, size_t* len) {
  const ImageStorage* img = image_of(f, image);
  if (!img || !data || !len || tile >= img->nal.size()) {
    set_last_error("invalid argument");
    return HEIC_E_INVALID_ARG;
  }
  *data = img->nal[tile].data();
  *len = img->nal[tile].size();
  return 0;
}
int32_t heic_b200_file_info(const heic_b200_file* f, heic_file_info* out) {
  if (!f || !out) {
    set_last_error("null argument");
    return HEIC_E_INVALID_ARG;
  }
  *out = f->f->info;
  return 0;
}
int32_t heic_b200_file_image_transform(const heic_b200_file* f, int32_t image, heic_image_transform* out) {
  const ImageStorage* img = image_of(f, image);
  if (!img || !out) {
    set_last_error("invalid argument");
    return HEIC_E_INVALID_ARG;
  }
  *out = img->transform;
  return 0;
}

}  // extern "C"
