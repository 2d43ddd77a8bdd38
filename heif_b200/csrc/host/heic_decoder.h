// HeicDecoder — host orchestration: container -> parameter sets -> per-tile slice headers ->
// plain-data image descriptors for the GPU path.  Mirrors HeicDecoder::decode's item walk
// (reference src/heic/decoder.rs:12-112); the tile loop at decoder.rs:114-119 is what the
// CUDA pipeline replaces.
#pragma once
#include <memory>
#include <vector>

#include "heif_reader.h"
#include "hevc_parse.h"

namespace heic {

struct ImageStorage {
  heic_image_desc desc;
  std::vector<heic_tile_desc> tiles;
  heic_image_desc desc_raw;                // the same image with raw tile payloads (heic_tile_desc::escaped = 1)
  std::vector<heic_tile_desc> tiles_raw;
  std::vector<std::vector<uint8_t>> rbsp;  // un-escaped slice RBSP per tile (owned)
  std::vector<std::vector<uint8_t>> nal;   // escaped VCL NAL unit per tile incl. 2-byte header
  std::vector<uint8_t> vps_nal, sps_nal, pps_nal;  // escaped parameter-set NAL units from hvcC
  heic_image_transform transform;                  // the item's clap / irot / imir in normal form
  uint32_t item_id = 0;
};

struct HeicFile {
  Heif heif;
  ImageStorage primary;
  std::vector<std::unique_ptr<ImageStorage>> aux;
  heic_file_info info;
};

// decoder.rs:135-143 — hvcC NAL: 2-byte header + escaped payload, no length prefix.
std::vector<uint8_t> read_hvcc_nal_unit(const std::vector<uint8_t>& raw, uint16_t* header);
// decoder.rs:146-164 — item data: length-prefixed NAL units; exactly one VCL NAL per item.
// Returns the un-escaped RBSP of that NAL; epb receives removed-byte positions.
std::vector<uint8_t> read_item_nal_unit(const std::vector<uint8_t>& item, unsigned length_size,
                                        uint16_t* header, std::vector<uint32_t>* epb,
                                        std::vector<uint8_t>* raw_nal = nullptr);

class HeicDecoder {
 public:
  // Parse everything up to (and including) the slice-segment headers.
  static std::unique_ptr<HeicFile> open(const uint8_t* data, size_t len);

 private:
  static void build_image(const HeifReader& reader, const Heif& heif, uint32_t item_id, ImageStorage& out);
};

}  // namespace heic
