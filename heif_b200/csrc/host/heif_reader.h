// HeifReader — ISOBMFF / HEIF container parse on the host.
// Same role and entry points as the reference's src/heif/reader.rs (HeifReader::{new, read,
// get_item_data}) and the accessors of src/heif/grammar.rs (Heif::{primary_item_id,
// item_info_by_item_id, hevc_configuration_record}); differences are listed where they occur.
#pragma once
#include <cstdint>
#include <string>
#include <utility>
#include <vector>

#include "rbsp_reader.h"

namespace heic {

constexpr uint32_t fourcc(const char (&s)[5]) {
  return (uint32_t(uint8_t(s[0])) << 24) | (uint32_t(uint8_t(s[1])) << 16) | (uint32_t(uint8_t(s[2])) << 8) |
         uint32_t(uint8_t(s[3]));
}
std::string fourcc_str(uint32_t v);

struct ItemInfoEntry {  // grammar.rs:184-193 (infe v2/v3)
  uint32_t item_id = 0;
  uint32_t item_protection_index = 0;
  uint32_t item_type = 0;
  bool hidden = false;
  std::string item_name, content_type;
};

struct SingleItemReferenceBox {  // grammar.rs:203-208
  uint32_t reference_type = 0;
  uint32_t from_item_id = 0;
  std::vector<uint32_t> to_item_ids;
};

struct RawNalUnit {
  std::vector<uint8_t> data;
};
struct NalArray {  // hevc/grammar.rs:329-343
  uint8_t type_byte = 0;
  std::vector<RawNalUnit> nal_units;
  bool array_completeness() const { return type_byte & 0x80; }
  uint32_t nal_unit_type() const { return type_byte & 0x3f; }
};
struct HEVCDecoderConfigurationRecord {  // hevc/grammar.rs:157-222
  uint8_t configuration_version = 0, general_profile_byte = 0;
  uint32_t general_profile_compatibility_flags = 0;
  uint64_t general_constraint_indicator_flags = 0;
  uint8_t general_level_idc = 0;
  uint16_t min_spatial_segmentation = 0;
  uint8_t parallelism_byte = 0, chroma_format_byte = 0, bit_depth_luma_byte = 0, bit_depth_chroma_byte = 0;
  uint16_t avg_frame_rate = 0;
  uint8_t frame_rate_byte = 0;
  std::vector<NalArray> arrays;
  uint8_t general_profile_idc() const { return general_profile_byte & 0x1f; }
  uint8_t chroma_format_idc() const { return chroma_format_byte & 3; }
  uint8_t bit_depth_luma_minus8() const { return bit_depth_luma_byte & 7; }
  uint8_t bit_depth_chroma_minus8() const { return bit_depth_chroma_byte & 7; }
  uint8_t length_size_minus_one() const { return frame_rate_byte & 3; }
};

// One child of ipco.  Unlike the reference (reader.rs:460-463 drops unknown children so ipma
// indices drift, SURVEY Appendix B #7) every child keeps its slot.
struct ItemProperty {
  uint32_t kind = 0;
  size_t payload_offset = 0, payload_size = 0;  // box payload in the file
  // parsed forms (valid according to kind)
  uint32_t ispe_width = 0, ispe_height = 0;     // 'ispe'
  uint32_t irot_angle = 0;                      // 'irot' (ccw quarter turns)
  uint32_t imir_axis = 0;                       // 'imir'
  // 'clap' (ISO/IEC 14496-12 12.1.4): cleanApertureWidthN/D, cleanApertureHeightN/D, horizOffN/D, vertOffN/D
  uint32_t clap_width_n = 0, clap_width_d = 0, clap_height_n = 0, clap_height_d = 0;
  int32_t clap_horiz_off_n = 0, clap_vert_off_n = 0;
  uint32_t clap_horiz_off_d = 0, clap_vert_off_d = 0;
  std::vector<uint8_t> pixi_bits;               // 'pixi'
  uint32_t colr_type = 0;                       // 'colr': 'nclx' / 'prof' / 'rICC'
  uint32_t nclx_primaries = 2, nclx_transfer = 2, nclx_matrix = 2, nclx_full_range = 0;
  std::string aux_type;                         // 'auxC'
  HEVCDecoderConfigurationRecord hvcc;          // 'hvcC'
};

struct ItemPropertyAssociation {
  uint32_t item_id = 0;
  std::vector<std::pair<bool, uint32_t>> entries;  // (essential, 1-based property index)
};

struct ItemLocationBoxReference {  // grammar.rs:312-319
  uint32_t item_id = 0;
  uint32_t construction_method = 0;
  uint32_t data_reference_index = 0;
  uint64_t base_offset = 0;
  std::vector<std::pair<uint64_t, uint64_t>> extents;  // (offset, length)
};

struct GridDescriptor {  // HEIF 6.6.2.3 — the reference never parses it (idat is skipped, reader.rs:139-142)
  uint32_t rows = 0, cols = 0, output_width = 0, output_height = 0;
};

struct Heif {
  uint32_t major_brand = 0, minor_version = 0;
  std::vector<uint32_t> compatible_brands;
  std::string handler_kind;
  uint32_t primary_item = 0;
  bool has_primary_item = false;
  std::vector<ItemInfoEntry> item_info_entries;
  std::vector<SingleItemReferenceBox> item_references;
  std::vector<ItemProperty> properties;
  std::vector<ItemPropertyAssociation> associations;
  std::vector<ItemLocationBoxReference> item_location;
  size_t idat_offset = 0, idat_size = 0;

  uint32_t primary_item_id() const { return primary_item; }
  const ItemInfoEntry* item_info_by_item_id(uint32_t id) const;
  // grammar.rs:38-49 returns the FIRST hvcC in ipco whatever item it belongs to (Appendix B #6).
  const HEVCDecoderConfigurationRecord* hevc_configuration_record() const;
  // The hvcC (or any property kind) actually associated with an item through ipma.
  const ItemProperty* property_of(uint32_t item_id, uint32_t kind) const;
  // Every property of an item, in the order its ipma entries list them.
  std::vector<const ItemProperty*> properties_of(uint32_t item_id) const;
  std::vector<uint32_t> references_from(uint32_t from_item_id, uint32_t reference_type) const;
  std::vector<uint32_t> references_to(uint32_t to_item_id, uint32_t reference_type) const;
};

// imir axis_type -> orientation bits of heic_image_transform: axis 0 mirrors top <-> bottom (6 = half turn, then
// left <-> right), axis 1 mirrors left <-> right (4).  This follows libheif's reading and the later editions of
// ISO/IEC 23008-12; the 2017 wording ("vertical axis" for 0) can be read the other way round, in which case only this
// table changes.
constexpr uint32_t kImirOrientation[2] = {6, 4};

// The transformative properties (clap, irot, imir) of an image of canvas_w x canvas_h, applied in the given order,
// reduced to heic_image_transform's normal form.  Other property kinds are skipped.  Throws HEIC_E_BITSTREAM for a clap
// with a zero denominator, an empty clean aperture, or one that does not lie inside the image it applies to.
heic_image_transform compose_transform(uint32_t canvas_w, uint32_t canvas_h, const std::vector<const ItemProperty*>& props);

class HeifReader {
 public:
  HeifReader(const uint8_t* data, size_t len) : data_(data), len_(len) {}
  Heif read();
  // reader.rs:33-57.  construction_method 0 (file offset) and 1 (idat) are supported and multiple
  // extents are concatenated — both are todo!() in the reference (reader.rs:42,47).
  std::vector<uint8_t> get_item_data(const Heif& heif, uint32_t item_id) const;
  GridDescriptor read_grid_descriptor(const Heif& heif, uint32_t item_id) const;

 private:
  struct BoxHeader {
    uint32_t kind;
    size_t start, payload, end;
  };
  BoxHeader read_box_header(size_t pos, size_t limit) const;
  uint64_t be(size_t pos, unsigned nbytes, size_t limit) const;
  void read_meta(Heif& h, const BoxHeader& box) const;
  void read_iinf(Heif& h, const BoxHeader& box) const;
  void read_iref(Heif& h, const BoxHeader& box) const;
  void read_iprp(Heif& h, const BoxHeader& box) const;
  void read_iloc(Heif& h, const BoxHeader& box) const;
  void read_hvcc(ItemProperty& p, const BoxHeader& box) const;
  const uint8_t* data_;
  size_t len_;
};

}  // namespace heic
