#include "heic_decoder.h"

#include <cstring>

namespace heic {

std::vector<uint8_t> read_hvcc_nal_unit(const std::vector<uint8_t>& raw, uint16_t* header) {
  if (raw.size() < 2) bail(HEIC_E_BITSTREAM, "nal unit is too short");
  if (header) *header = static_cast<uint16_t>((raw[0] << 8) | raw[1]);
  return RbspReader::remove_emulation_prevention(raw.data() + 2, raw.size() - 2);
}

std::vector<uint8_t> read_item_nal_unit(const std::vector<uint8_t>& item, unsigned length_size,
                                        uint16_t* header, std::vector<uint32_t>* epb,
                                        std::vector<uint8_t>* raw_nal) {
  // The reference demands that the 4-byte length covers the whole item (decoder.rs:146-164).
  // Encoders may prepend SEI/AUD NAL units, so we walk all length-prefixed units and require
  // exactly one VCL unit (nal_unit_type < 32).
  size_t pos = 0;
  const uint8_t* vcl = nullptr;
  size_t vcl_len = 0;
  while (pos < item.size()) {
    if (pos + length_size > item.size())
      bail(HEIC_E_BITSTREAM, "nal unit is too short (need length prefix + 2 header bytes)");
    size_t n = 0;
    for (unsigned i = 0; i < length_size; ++i) n = (n << 8) | item[pos + i];
    pos += length_size;
    if (n < 2 || n > item.size() - pos)
      bail(HEIC_E_BITSTREAM, "tile item NAL length prefix says " + std::to_string(n) + " bytes, but item has " +
                                 std::to_string(item.size() - pos) + " bytes of NAL data");
    unsigned type = (item[pos] >> 1) & 0x3f;
    if (type < 32) {
      if (vcl) bail(HEIC_E_UNSUPPORTED, "tile item should contain exactly one VCL NAL unit");
      vcl = item.data() + pos;
      vcl_len = n;
    }
    pos += n;
  }
  if (!vcl) bail(HEIC_E_BITSTREAM, "tile item contains no VCL NAL unit");
  if (header) *header = static_cast<uint16_t>((vcl[0] << 8) | vcl[1]);
  if (raw_nal) raw_nal->assign(vcl, vcl + vcl_len);
  return RbspReader::remove_emulation_prevention(vcl + 2, vcl_len - 2, epb);
}

static const RawNalUnit& first_nal_of_type(const HEVCDecoderConfigurationRecord& c, uint32_t type, const char* what) {
  for (auto& a : c.arrays)
    if (a.nal_unit_type() == type) {
      if (a.nal_units.empty()) bail(HEIC_E_BITSTREAM, std::string(what) + " array is empty");
      return a.nal_units.front();
    }
  bail(HEIC_E_BITSTREAM, std::string("no ") + what + " in hvcC");
}

void HeicDecoder::build_image(const HeifReader& reader, const Heif& heif, uint32_t item_id, ImageStorage& out) {
  const ItemInfoEntry* info = heif.item_info_by_item_id(item_id);
  if (!info) bail(HEIC_E_BITSTREAM, "item " + std::to_string(item_id) + " not found in item_info");
  out.item_id = item_id;
  std::memset(&out.desc, 0, sizeof out.desc);

  std::vector<uint32_t> tile_ids;
  GridDescriptor grid;
  if (info->item_type == fourcc("grid")) {
    // decoder.rs:88-94 takes the first iref whose from_item_id matches, whatever its type
    // (Appendix B #13); we require 'dimg'.
    tile_ids = heif.references_from(item_id, fourcc("dimg"));
    if (tile_ids.empty()) bail(HEIC_E_BITSTREAM, "grid " + std::to_string(item_id) + " has no tile references");
    grid = reader.read_grid_descriptor(heif, item_id);
    if (uint64_t{grid.rows} * grid.cols != tile_ids.size())
      bail(HEIC_E_BITSTREAM, "grid rows*cols does not match the number of dimg references");
  } else if (info->item_type == fourcc("hvc1")) {
    tile_ids.push_back(item_id);
    grid.rows = grid.cols = 1;
  } else {
    bail(HEIC_E_UNSUPPORTED, "unsupported primary item type: " + fourcc_str(info->item_type));
  }

  const ItemProperty* hvcc_prop = heif.property_of(tile_ids.front(), fourcc("hvcC"));
  if (!hvcc_prop) bail(HEIC_E_BITSTREAM, "missing HEVC decoder configuration");
  const HEVCDecoderConfigurationRecord& cfg = hvcc_prop->hvcc;
  for (uint32_t id : tile_ids) {
    const ItemInfoEntry* ti = heif.item_info_by_item_id(id);
    if (!ti || ti->item_type != fourcc("hvc1")) bail(HEIC_E_UNSUPPORTED, "grid tile is not an hvc1 item");
    if (heif.property_of(id, fourcc("hvcC")) != hvcc_prop)
      bail(HEIC_E_UNSUPPORTED, "grid tiles with different hvcC configurations");
  }

  {
    for (auto& a : cfg.arrays)
      if (a.nal_unit_type() == 32 && !a.nal_units.empty()) out.vps_nal = a.nal_units.front().data;
    out.sps_nal = first_nal_of_type(cfg, 33, "SPS").data;
    out.pps_nal = first_nal_of_type(cfg, 34, "PPS").data;
    std::vector<uint8_t> sps_rbsp = read_hvcc_nal_unit(first_nal_of_type(cfg, 33, "SPS").data, nullptr);
    out.desc.sps = sequence_parameter_set_rbsp(sps_rbsp.data(), sps_rbsp.size());
    std::vector<uint8_t> pps_rbsp = read_hvcc_nal_unit(first_nal_of_type(cfg, 34, "PPS").data, nullptr);
    out.desc.pps = picture_parameter_set_rbsp(pps_rbsp.data(), pps_rbsp.size());
  }
  {
    // HEIF 6.5.5: a 'colr' property of type nclx on the item overrides the colour description of the bitstream's VUI
    const ItemProperty* colr = heif.property_of(item_id, fourcc("colr"));
    if (colr && colr->colr_type == fourcc("nclx")) {
      out.desc.sps.vui_parameters_present_flag = 1;
      out.desc.sps.video_full_range_flag = colr->nclx_full_range;
      out.desc.sps.matrix_coeffs = colr->nclx_matrix;
      out.desc.sps.colour_primaries = colr->nclx_primaries;
      out.desc.sps.transfer_characteristics = colr->nclx_transfer;
    }
  }
  const heic_sps& sps = out.desc.sps;

  out.rbsp.resize(tile_ids.size());
  out.nal.resize(tile_ids.size());
  out.tiles.resize(tile_ids.size());
  out.tiles_raw.resize(tile_ids.size());
  for (size_t t = 0; t < tile_ids.size(); ++t) {
    std::vector<uint8_t> item = reader.get_item_data(heif, tile_ids[t]);
    uint16_t header = 0;
    std::vector<uint32_t> epb;
    out.rbsp[t] = read_item_nal_unit(item, cfg.length_size_minus_one() + 1u, &header, &epb, &out.nal[t]);
    heic_tile_desc& td = out.tiles[t];
    std::memset(&td, 0, sizeof td);
    td.nal_unit_type = (header >> 9) & 0x3f;
    td.rbsp = out.rbsp[t].data();
    td.rbsp_len = static_cast<uint32_t>(out.rbsp[t].size());
    td.header = slice_segment_header(td.rbsp, td.rbsp_len, td.nal_unit_type, sps, out.desc.pps, epb.data(), epb.size());
    // the same tile as it lies in mdat: raw payload after the 2-byte NAL header, offsets in raw byte counts
    heic_tile_desc& tr = out.tiles_raw[t];
    std::memset(&tr, 0, sizeof tr);
    tr.nal_unit_type = td.nal_unit_type;
    tr.escaped = 1;
    tr.rbsp = out.nal[t].data() + 2;
    tr.rbsp_len = static_cast<uint32_t>(out.nal[t].size() - 2);
    tr.header = slice_segment_header_raw(tr.rbsp, tr.rbsp_len, tr.nal_unit_type, sps, out.desc.pps);
  }

  uint32_t sub_w = (sps.chroma_format_idc == 1 || sps.chroma_format_idc == 2) ? 2 : 1;
  uint32_t sub_h = sps.chroma_format_idc == 1 ? 2 : 1;
  uint32_t tile_w = sps.pic_width_in_luma_samples - sub_w * (sps.conf_win_left_offset + sps.conf_win_right_offset);
  uint32_t tile_h = sps.pic_height_in_luma_samples - sub_h * (sps.conf_win_top_offset + sps.conf_win_bottom_offset);
  out.desc.grid_rows = grid.rows;
  out.desc.grid_cols = grid.cols;
  if (info->item_type == fourcc("grid")) {
    out.desc.output_width = grid.output_width;
    out.desc.output_height = grid.output_height;
    if (uint64_t{tile_w} * grid.cols < grid.output_width || uint64_t{tile_h} * grid.rows < grid.output_height)
      bail(HEIC_E_BITSTREAM, "grid tiles do not cover the output canvas");
  } else {
    out.desc.output_width = tile_w;
    out.desc.output_height = tile_h;
  }
  const ItemProperty* irot = heif.property_of(item_id, fourcc("irot"));
  out.desc.rotation_ccw_quarter_turns = irot ? irot->irot_angle : 0;
  out.transform = compose_transform(out.desc.output_width, out.desc.output_height, heif.properties_of(item_id));
  out.desc.n_tiles = static_cast<uint32_t>(tile_ids.size());
  out.desc.tiles = out.tiles.data();
  out.desc_raw = out.desc;
  out.desc_raw.tiles = out.tiles_raw.data();
}

std::unique_ptr<HeicFile> HeicDecoder::open(const uint8_t* data, size_t len) {
  auto f = std::make_unique<HeicFile>();
  HeifReader reader(data, len);
  f->heif = reader.read();
  const Heif& heif = f->heif;
  uint32_t primary = heif.primary_item_id();
  build_image(reader, heif, primary, f->primary);
  for (uint32_t aux_id : heif.references_to(primary, fourcc("auxl"))) {
    auto img = std::make_unique<ImageStorage>();
    try {
      build_image(reader, heif, aux_id, *img);
    } catch (const Error&) {
      continue;  // an undecodable auxiliary image does not make the primary image undecodable
    }
    f->aux.push_back(std::move(img));
  }

  // tests/libheif_comparison.rs:41-111 — the metadata the reference's integration test pins.
  heic_file_info& fi = f->info;
  std::memset(&fi, 0, sizeof fi);
  fi.primary_item_id = primary;
  const ItemProperty* ispe = heif.property_of(primary, fourcc("ispe"));
  fi.ispe_width = ispe ? ispe->ispe_width : f->primary.desc.output_width;
  fi.ispe_height = ispe ? ispe->ispe_height : f->primary.desc.output_height;
  fi.rotation_ccw_quarter_turns = f->primary.desc.rotation_ccw_quarter_turns;
  const heic_image_transform& xf = f->primary.transform;
  bool swap = xf.orientation & 1;
  fi.rotated_width = swap ? xf.crop_h : xf.crop_w;
  fi.rotated_height = swap ? xf.crop_w : xf.crop_h;
  fi.luma_bits = f->primary.desc.sps.bit_depth_luma_minus8 + 8;
  fi.chroma_bits = f->primary.desc.sps.bit_depth_chroma_minus8 + 8;
  fi.thumbnail_count = static_cast<uint32_t>(heif.references_to(primary, fourcc("thmb")).size());
  fi.item_count = static_cast<uint32_t>(heif.item_info_entries.size());
  fi.is_grid = f->primary.desc.n_tiles > 1 || heif.item_info_by_item_id(primary)->item_type == fourcc("grid");
  return f;
}

}  // namespace heic
