// ISOBMFF / HEIF box walk.  Structure follows ISO/IEC 14496-12 and 23008-12; behaviour is checked
// against the reference's src/heif/reader.rs on halfmoonbay.heic (SURVEY Appendix A).
#include "heif_reader.h"

#include <algorithm>
#include <cstring>

namespace heic {

std::string fourcc_str(uint32_t v) {
  char s[5] = {char(v >> 24), char(v >> 16), char(v >> 8), char(v), 0};
  return s;
}

const ItemInfoEntry* Heif::item_info_by_item_id(uint32_t id) const {
  for (auto& e : item_info_entries)
    if (e.item_id == id) return &e;
  return nullptr;
}

const HEVCDecoderConfigurationRecord* Heif::hevc_configuration_record() const {
  for (auto& p : properties)
    if (p.kind == fourcc("hvcC")) return &p.hvcc;
  return nullptr;
}

const ItemProperty* Heif::property_of(uint32_t item_id, uint32_t kind) const {
  for (auto& a : associations) {
    if (a.item_id != item_id) continue;
    for (auto& e : a.entries) {
      if (e.second == 0 || e.second > properties.size()) continue;
      const ItemProperty& p = properties[e.second - 1];
      if (p.kind == kind) return &p;
    }
  }
  return nullptr;
}

std::vector<const ItemProperty*> Heif::properties_of(uint32_t item_id) const {
  std::vector<const ItemProperty*> out;
  for (auto& a : associations) {
    if (a.item_id != item_id) continue;
    for (auto& e : a.entries)
      if (e.second != 0 && e.second <= properties.size()) out.push_back(&properties[e.second - 1]);
  }
  return out;
}

namespace {

// floor(n / d) for d > 0
__int128 floor_div(__int128 n, __int128 d) { return n >= 0 ? n / d : -((-n + d - 1) / d); }

// Pixel (x, y) of a w x h block whose image after orientation o (see heic_image_transform) has pixel (ox, oy) there.
// Forward: 1: (y, w - 1 - x)  2: (w - 1 - x, h - 1 - y)  3: (h - 1 - y, x), then ox -> width - 1 - ox when o & 4.
void unorient(uint32_t o, int64_t w, int64_t h, int64_t ox, int64_t oy, int64_t& x, int64_t& y) {
  if (o & 4) ox = ((o & 1) ? h : w) - 1 - ox;
  switch (o & 3) {
    case 0: x = ox, y = oy; break;
    case 1: y = ox, x = w - 1 - oy; break;
    case 2: x = w - 1 - ox, y = h - 1 - oy; break;
    default: y = h - 1 - ox, x = oy; break;
  }
}

}  // namespace

heic_image_transform compose_transform(uint32_t canvas_w, uint32_t canvas_h, const std::vector<const ItemProperty*>& props) {
  heic_image_transform t{0, 0, canvas_w, canvas_h, 0};
  for (const ItemProperty* p : props) {
    uint32_t rot = t.orientation & 3, mir = t.orientation >> 2;
    if (p->kind == fourcc("irot")) {
      // a turn after a mirror is the mirror after the opposite turn
      rot = mir ? (rot - p->irot_angle) & 3 : (rot + p->irot_angle) & 3;
      t.orientation = rot | (mir << 2);
    } else if (p->kind == fourcc("imir")) {
      // left <-> right toggles the mirror; top <-> bottom is a half turn and then left <-> right
      const uint32_t m = kImirOrientation[p->imir_axis & 1];
      rot = mir ? (rot - (m & 3)) & 3 : (rot + (m & 3)) & 3;
      t.orientation = rot | ((mir ^ 1u) << 2);
    } else if (p->kind == fourcc("clap")) {
      const int64_t W = (t.orientation & 1) ? t.crop_h : t.crop_w, H = (t.orientation & 1) ? t.crop_w : t.crop_h;
      if (!p->clap_width_d || !p->clap_height_d || !p->clap_horiz_off_d || !p->clap_vert_off_d)
        bail(HEIC_E_BITSTREAM, "clap with a zero denominator");
      // Exact rationals: left = horizOff + (W - cleanW) / 2, rounded down; the width rounded to the nearest integer (halves
      // up).  The rounding of non-integral values is this library's choice; it has not been compared with libheif's.
      const __int128 wn = p->clap_width_n, wd = p->clap_width_d, hn = p->clap_height_n, hd = p->clap_height_d;
      const __int128 xn = p->clap_horiz_off_n, xd = p->clap_horiz_off_d, yn = p->clap_vert_off_n, yd = p->clap_vert_off_d;
      const __int128 cw = floor_div(2 * wn + wd, 2 * wd), ch = floor_div(2 * hn + hd, 2 * hd);
      const __int128 left = floor_div(2 * xn * wd + ((__int128)W * wd - wn) * xd, 2 * xd * wd);
      const __int128 top = floor_div(2 * yn * hd + ((__int128)H * hd - hn) * yd, 2 * yd * hd);
      if (cw <= 0 || ch <= 0 || left < 0 || top < 0 || left + cw > W || top + ch > H)
        bail(HEIC_E_BITSTREAM, "clap clean aperture is empty or not inside the image");
      // the rectangle's corners back in crop coordinates
      int64_t x0, y0, x1, y1;
      unorient(t.orientation, t.crop_w, t.crop_h, (int64_t)left, (int64_t)top, x0, y0);
      unorient(t.orientation, t.crop_w, t.crop_h, (int64_t)(left + cw - 1), (int64_t)(top + ch - 1), x1, y1);
      t.crop_x += (uint32_t)std::min(x0, x1);
      t.crop_y += (uint32_t)std::min(y0, y1);
      t.crop_w = (uint32_t)(std::max(x0, x1) - std::min(x0, x1) + 1);
      t.crop_h = (uint32_t)(std::max(y0, y1) - std::min(y0, y1) + 1);
    }
  }
  return t;
}

std::vector<uint32_t> Heif::references_from(uint32_t from, uint32_t type) const {
  std::vector<uint32_t> out;
  for (auto& r : item_references)
    if (r.from_item_id == from && r.reference_type == type) out.insert(out.end(), r.to_item_ids.begin(), r.to_item_ids.end());
  return out;
}

std::vector<uint32_t> Heif::references_to(uint32_t to, uint32_t type) const {
  std::vector<uint32_t> out;
  for (auto& r : item_references)
    if (r.reference_type == type && std::find(r.to_item_ids.begin(), r.to_item_ids.end(), to) != r.to_item_ids.end())
      out.push_back(r.from_item_id);
  return out;
}

uint64_t HeifReader::be(size_t pos, unsigned nbytes, size_t limit) const {
  if (pos + nbytes > limit || pos + nbytes > len_) bail(HEIC_E_BITSTREAM, "box field beyond end of box");
  uint64_t v = 0;
  for (unsigned i = 0; i < nbytes; ++i) v = (v << 8) | data_[pos + i];
  return v;
}

HeifReader::BoxHeader HeifReader::read_box_header(size_t pos, size_t limit) const {
  BoxHeader b;
  b.start = pos;
  uint64_t size = be(pos, 4, limit);
  b.kind = static_cast<uint32_t>(be(pos + 4, 4, limit));
  size_t hdr = 8;
  if (size == 1) {
    size = be(pos + 8, 8, limit);
    hdr = 16;
  } else if (size == 0) {
    size = limit - pos;  // box extends to the end of its container
  }
  if (b.kind == fourcc("uuid")) hdr += 16;
  if (size < hdr || size > limit - pos) bail(HEIC_E_BITSTREAM, "box '" + fourcc_str(b.kind) + "' has an invalid size");
  b.payload = pos + hdr;
  b.end = pos + static_cast<size_t>(size);
  return b;
}

// reader.rs:59-83: ftyp first, then top-level boxes; only meta is interpreted.
Heif HeifReader::read() {
  Heif h;
  size_t pos = 0;
  BoxHeader ftyp = read_box_header(pos, len_);
  if (ftyp.kind != fourcc("ftyp")) bail(HEIC_E_BITSTREAM, "file does not start with an ftyp box");
  h.major_brand = static_cast<uint32_t>(be(ftyp.payload, 4, ftyp.end));
  h.minor_version = static_cast<uint32_t>(be(ftyp.payload + 4, 4, ftyp.end));
  for (size_t p = ftyp.payload + 8; p + 4 <= ftyp.end; p += 4) h.compatible_brands.push_back(static_cast<uint32_t>(be(p, 4, ftyp.end)));
  pos = ftyp.end;
  bool have_meta = false;
  while (pos < len_) {
    BoxHeader b = read_box_header(pos, len_);
    if (b.kind == fourcc("meta") && !have_meta) {
      read_meta(h, b);
      have_meta = true;
    }
    pos = b.end;
  }
  if (!have_meta) bail(HEIC_E_BITSTREAM, "missing required meta box");
  if (!h.has_primary_item) bail(HEIC_E_BITSTREAM, "missing required pitm box");
  if (h.item_info_entries.empty()) bail(HEIC_E_BITSTREAM, "missing required iinf box");
  if (h.item_location.empty()) bail(HEIC_E_BITSTREAM, "missing required iloc box");
  return h;
}

// reader.rs:100-156.  The reference requires hdlr to be the first child; we accept any order.
void HeifReader::read_meta(Heif& h, const BoxHeader& box) const {
  uint32_t vf = static_cast<uint32_t>(be(box.payload, 4, box.end));
  if ((vf >> 24) != 0) bail(HEIC_E_UNSUPPORTED, "meta box version != 0");
  size_t pos = box.payload + 4;
  while (pos < box.end) {
    BoxHeader b = read_box_header(pos, box.end);
    switch (b.kind) {
      case fourcc("hdlr"): {
        // FullBox, pre_defined(4), handler_type(4)
        uint32_t kind = static_cast<uint32_t>(be(b.payload + 8, 4, b.end));
        h.handler_kind = fourcc_str(kind);
        break;
      }
      case fourcc("pitm"): {
        uint32_t v = static_cast<uint32_t>(be(b.payload, 4, b.end)) >> 24;
        h.primary_item = static_cast<uint32_t>(be(b.payload + 4, v == 0 ? 2 : 4, b.end));
        h.has_primary_item = true;
        break;
      }
      case fourcc("iinf"): read_iinf(h, b); break;
      case fourcc("iref"): read_iref(h, b); break;
      case fourcc("iprp"): read_iprp(h, b); break;
      case fourcc("iloc"): read_iloc(h, b); break;
      case fourcc("idat"):
        h.idat_offset = b.payload;
        h.idat_size = b.end - b.payload;
        break;
      default: break;  // dinf etc.: not needed to locate or decode items
    }
    pos = b.end;
  }
}

static std::string read_cstr(const uint8_t* data, size_t& pos, size_t end) {
  size_t s = pos;
  while (pos < end && data[pos] != 0) ++pos;
  std::string out(reinterpret_cast<const char*>(data + s), pos - s);
  if (pos < end) ++pos;  // consume the NUL (the reference keeps it in the remainder, Appendix B #8)
  return out;
}

// reader.rs:282-374
void HeifReader::read_iinf(Heif& h, const BoxHeader& box) const {
  uint32_t v = static_cast<uint32_t>(be(box.payload, 4, box.end)) >> 24;
  size_t pos = box.payload + 4;
  uint32_t count = static_cast<uint32_t>(be(pos, v == 0 ? 2 : 4, box.end));
  pos += v == 0 ? 2 : 4;
  for (uint32_t i = 0; i < count && pos < box.end; ++i) {
    BoxHeader b = read_box_header(pos, box.end);
    pos = b.end;
    if (b.kind != fourcc("infe")) continue;
    uint32_t vf = static_cast<uint32_t>(be(b.payload, 4, b.end));
    uint32_t ver = vf >> 24;
    if (ver < 2) bail(HEIC_E_UNSUPPORTED, "infe version < 2");
    ItemInfoEntry e;
    e.hidden = vf & 1;
    size_t p = b.payload + 4;
    e.item_id = static_cast<uint32_t>(be(p, ver == 2 ? 2 : 4, b.end));
    p += ver == 2 ? 2 : 4;
    e.item_protection_index = static_cast<uint32_t>(be(p, 2, b.end));
    p += 2;
    e.item_type = static_cast<uint32_t>(be(p, 4, b.end));
    p += 4;
    e.item_name = read_cstr(data_, p, b.end);
    if (e.item_type == fourcc("mime")) e.content_type = read_cstr(data_, p, b.end);
    h.item_info_entries.push_back(std::move(e));
  }
}

// reader.rs:376-422
void HeifReader::read_iref(Heif& h, const BoxHeader& box) const {
  uint32_t v = static_cast<uint32_t>(be(box.payload, 4, box.end)) >> 24;
  unsigned idsz = v == 0 ? 2 : 4;
  size_t pos = box.payload + 4;
  while (pos < box.end) {
    BoxHeader b = read_box_header(pos, box.end);
    SingleItemReferenceBox r;
    r.reference_type = b.kind;
    size_t p = b.payload;
    r.from_item_id = static_cast<uint32_t>(be(p, idsz, b.end));
    p += idsz;
    uint32_t n = static_cast<uint32_t>(be(p, 2, b.end));
    p += 2;
    for (uint32_t i = 0; i < n; ++i, p += idsz) r.to_item_ids.push_back(static_cast<uint32_t>(be(p, idsz, b.end)));
    h.item_references.push_back(std::move(r));
    pos = b.end;
  }
}

// reader.rs:570-630
void HeifReader::read_hvcc(ItemProperty& prop, const BoxHeader& b) const {
  HEVCDecoderConfigurationRecord& c = prop.hvcc;
  size_t p = b.payload;
  c.configuration_version = static_cast<uint8_t>(be(p, 1, b.end));
  if (c.configuration_version != 1) bail(HEIC_E_UNSUPPORTED, "unsupported hvcC version");
  c.general_profile_byte = static_cast<uint8_t>(be(p + 1, 1, b.end));
  c.general_profile_compatibility_flags = static_cast<uint32_t>(be(p + 2, 4, b.end));
  c.general_constraint_indicator_flags = be(p + 6, 6, b.end);
  c.general_level_idc = static_cast<uint8_t>(be(p + 12, 1, b.end));
  c.min_spatial_segmentation = static_cast<uint16_t>(be(p + 13, 2, b.end));
  c.parallelism_byte = static_cast<uint8_t>(be(p + 15, 1, b.end));
  c.chroma_format_byte = static_cast<uint8_t>(be(p + 16, 1, b.end));
  c.bit_depth_luma_byte = static_cast<uint8_t>(be(p + 17, 1, b.end));
  c.bit_depth_chroma_byte = static_cast<uint8_t>(be(p + 18, 1, b.end));
  c.avg_frame_rate = static_cast<uint16_t>(be(p + 19, 2, b.end));
  c.frame_rate_byte = static_cast<uint8_t>(be(p + 21, 1, b.end));
  uint32_t n_arrays = static_cast<uint32_t>(be(p + 22, 1, b.end));
  p += 23;
  for (uint32_t a = 0; a < n_arrays; ++a) {
    NalArray arr;
    arr.type_byte = static_cast<uint8_t>(be(p, 1, b.end));
    uint32_t n = static_cast<uint32_t>(be(p + 1, 2, b.end));
    p += 3;
    for (uint32_t i = 0; i < n; ++i) {
      uint32_t l = static_cast<uint32_t>(be(p, 2, b.end));
      p += 2;
      if (p + l > b.end) bail(HEIC_E_BITSTREAM, "hvcC NAL unit beyond end of box");
      RawNalUnit nal;
      nal.data.assign(data_ + p, data_ + p + l);
      arr.nal_units.push_back(std::move(nal));
      p += l;
    }
    c.arrays.push_back(std::move(arr));
  }
}

// reader.rs:424-568
void HeifReader::read_iprp(Heif& h, const BoxHeader& box) const {
  size_t pos = box.payload;
  while (pos < box.end) {
    BoxHeader b = read_box_header(pos, box.end);
    if (b.kind == fourcc("ipco")) {
      size_t p = b.payload;
      while (p < b.end) {
        BoxHeader c = read_box_header(p, b.end);
        ItemProperty prop;
        prop.kind = c.kind;
        prop.payload_offset = c.payload;
        prop.payload_size = c.end - c.payload;
        switch (c.kind) {
          case fourcc("ispe"):
            prop.ispe_width = static_cast<uint32_t>(be(c.payload + 4, 4, c.end));
            prop.ispe_height = static_cast<uint32_t>(be(c.payload + 8, 4, c.end));
            break;
          case fourcc("irot"): prop.irot_angle = static_cast<uint32_t>(be(c.payload, 1, c.end)) & 3; break;
          case fourcc("imir"): prop.imir_axis = static_cast<uint32_t>(be(c.payload, 1, c.end)) & 1; break;
          case fourcc("clap"):
            prop.clap_width_n = static_cast<uint32_t>(be(c.payload, 4, c.end));
            prop.clap_width_d = static_cast<uint32_t>(be(c.payload + 4, 4, c.end));
            prop.clap_height_n = static_cast<uint32_t>(be(c.payload + 8, 4, c.end));
            prop.clap_height_d = static_cast<uint32_t>(be(c.payload + 12, 4, c.end));
            prop.clap_horiz_off_n = static_cast<int32_t>(static_cast<uint32_t>(be(c.payload + 16, 4, c.end)));
            prop.clap_horiz_off_d = static_cast<uint32_t>(be(c.payload + 20, 4, c.end));
            prop.clap_vert_off_n = static_cast<int32_t>(static_cast<uint32_t>(be(c.payload + 24, 4, c.end)));
            prop.clap_vert_off_d = static_cast<uint32_t>(be(c.payload + 28, 4, c.end));
            break;
          case fourcc("pixi"): {
            uint32_t n = static_cast<uint32_t>(be(c.payload + 4, 1, c.end));
            for (uint32_t i = 0; i < n; ++i) prop.pixi_bits.push_back(static_cast<uint8_t>(be(c.payload + 5 + i, 1, c.end)));
            break;
          }
          case fourcc("colr"):
            prop.colr_type = static_cast<uint32_t>(be(c.payload, 4, c.end));
            if (prop.colr_type == fourcc("nclx")) {
              prop.nclx_primaries = static_cast<uint32_t>(be(c.payload + 4, 2, c.end));
              prop.nclx_transfer = static_cast<uint32_t>(be(c.payload + 6, 2, c.end));
              prop.nclx_matrix = static_cast<uint32_t>(be(c.payload + 8, 2, c.end));
              prop.nclx_full_range = static_cast<uint32_t>(be(c.payload + 10, 1, c.end)) >> 7;
            }
            break;
          case fourcc("auxC"): {
            size_t q = c.payload + 4;
            prop.aux_type = read_cstr(data_, q, c.end);
            break;
          }
          case fourcc("hvcC"): read_hvcc(prop, c); break;
          default: break;
        }
        h.properties.push_back(std::move(prop));
        p = c.end;
      }
    } else if (b.kind == fourcc("ipma")) {
      uint32_t vf = static_cast<uint32_t>(be(b.payload, 4, b.end));
      uint32_t ver = vf >> 24;
      bool wide = vf & 1;
      size_t p = b.payload + 4;
      uint32_t n = static_cast<uint32_t>(be(p, 4, b.end));
      p += 4;
      for (uint32_t i = 0; i < n; ++i) {
        ItemPropertyAssociation a;
        a.item_id = static_cast<uint32_t>(be(p, ver < 1 ? 2 : 4, b.end));
        p += ver < 1 ? 2 : 4;
        uint32_t cnt = static_cast<uint32_t>(be(p, 1, b.end));
        p += 1;
        for (uint32_t k = 0; k < cnt; ++k) {
          if (wide) {
            uint32_t v = static_cast<uint32_t>(be(p, 2, b.end));
            p += 2;
            a.entries.emplace_back((v & 0x8000) != 0, v & 0x7fff);
          } else {
            uint32_t v = static_cast<uint32_t>(be(p, 1, b.end));
            p += 1;
            a.entries.emplace_back((v & 0x80) != 0, v & 0x7f);
          }
        }
        h.associations.push_back(std::move(a));
      }
    }
    pos = b.end;
  }
}

// reader.rs:632-704
void HeifReader::read_iloc(Heif& h, const BoxHeader& box) const {
  uint32_t ver = static_cast<uint32_t>(be(box.payload, 4, box.end)) >> 24;
  if (ver > 2) bail(HEIC_E_UNSUPPORTED, "unsupported iloc version");
  size_t p = box.payload + 4;
  uint32_t b1 = static_cast<uint32_t>(be(p, 1, box.end)), b2 = static_cast<uint32_t>(be(p + 1, 1, box.end));
  p += 2;
  unsigned offset_size = b1 >> 4, length_size = b1 & 15, base_offset_size = b2 >> 4, index_size = b2 & 15;
  auto ok = [](unsigned s) { return s == 0 || s == 4 || s == 8; };
  if (!ok(offset_size) || !ok(length_size) || !ok(base_offset_size) || !ok(index_size))
    bail(HEIC_E_BITSTREAM, "iloc field size not in {0,4,8}");
  uint32_t count = static_cast<uint32_t>(be(p, ver < 2 ? 2 : 4, box.end));
  p += ver < 2 ? 2 : 4;
  for (uint32_t i = 0; i < count; ++i) {
    ItemLocationBoxReference r;
    r.item_id = static_cast<uint32_t>(be(p, ver < 2 ? 2 : 4, box.end));
    p += ver < 2 ? 2 : 4;
    if (ver >= 1) {
      r.construction_method = static_cast<uint32_t>(be(p, 2, box.end)) & 15;
      p += 2;
    }
    r.data_reference_index = static_cast<uint32_t>(be(p, 2, box.end));
    p += 2;
    r.base_offset = base_offset_size ? be(p, base_offset_size, box.end) : 0;
    p += base_offset_size;
    uint32_t n_ext = static_cast<uint32_t>(be(p, 2, box.end));
    p += 2;
    for (uint32_t k = 0; k < n_ext; ++k) {
      if (ver >= 1 && index_size) p += index_size;
      uint64_t off = offset_size ? be(p, offset_size, box.end) : 0;
      p += offset_size;
      uint64_t ln = length_size ? be(p, length_size, box.end) : 0;
      p += length_size;
      r.extents.emplace_back(off, ln);
    }
    h.item_location.push_back(std::move(r));
  }
}

std::vector<uint8_t> HeifReader::get_item_data(const Heif& heif, uint32_t item_id) const {
  const ItemLocationBoxReference* ref = nullptr;
  for (auto& r : heif.item_location)
    if (r.item_id == item_id) ref = &r;
  if (!ref) bail(HEIC_E_BITSTREAM, "item " + std::to_string(item_id) + " not found in iloc");
  if (ref->data_reference_index != 0) bail(HEIC_E_UNSUPPORTED, "item data in an external file");
  size_t base, limit;
  if (ref->construction_method == 0) {
    base = 0;
    limit = len_;
  } else if (ref->construction_method == 1) {
    base = heif.idat_offset;
    limit = heif.idat_offset + heif.idat_size;
  } else {
    bail(HEIC_E_UNSUPPORTED, "iloc construction_method " + std::to_string(ref->construction_method));
  }
  std::vector<uint8_t> out;
  for (auto& e : ref->extents) {
    uint64_t start = base + ref->base_offset + e.first;
    uint64_t length = e.second ? e.second : (limit > start ? limit - start : 0);  // 0 = to end
    if (start > limit || length > limit - start) bail(HEIC_E_BITSTREAM, "item " + std::to_string(item_id) + " data out of bounds");
    out.insert(out.end(), data_ + start, data_ + start + length);
  }
  return out;
}

GridDescriptor HeifReader::read_grid_descriptor(const Heif& heif, uint32_t item_id) const {
  std::vector<uint8_t> d = get_item_data(heif, item_id);
  if (d.size() < 8 || d[0] != 0) bail(HEIC_E_BITSTREAM, "bad grid descriptor");
  GridDescriptor g;
  bool wide = d[1] & 1;
  g.rows = d[2] + 1u;
  g.cols = d[3] + 1u;
  if (wide) {
    if (d.size() < 12) bail(HEIC_E_BITSTREAM, "bad grid descriptor");
    g.output_width = (uint32_t(d[4]) << 24) | (d[5] << 16) | (d[6] << 8) | d[7];
    g.output_height = (uint32_t(d[8]) << 24) | (d[9] << 16) | (d[10] << 8) | d[11];
  } else {
    g.output_width = (d[4] << 8) | d[5];
    g.output_height = (d[6] << 8) | d[7];
  }
  return g;
}

}  // namespace heic
