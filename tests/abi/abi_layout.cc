// Prints the binary layout of the plugin ABI, one "name value" line per size, member offset and constant, in the same
// order for two header sets: by default include/b200_heif_plugin_abi.h (and the constants the library assumes), with
// -DREFERENCE_HEADERS the reference's own headers (libheif/api/libheif/heif_plugin.h, heif_error.h, heif_library.h).
// tests/golden/abi_layout.txt is the output for the reference headers; tests/test_plugin.py compares the two.
#include <cstddef>
#include <cstdint>
#include <cstdio>

#ifdef REFERENCE_HEADERS
#include <libheif/heif.h>
#include <libheif/heif_plugin.h>
typedef heif_error Error;
typedef heif_decoder_plugin Decoder;
typedef heif_encoder_plugin Encoder;
typedef heif_encoder_parameter EncoderParameter;
typedef heif_decoder_plugin_options DecoderOptions;
typedef heif_security_limits SecurityLimits;
typedef heif_plugin_info PluginInfo;
typedef heif_color_profile_nclx Nclx;
static const long kConstants[] = {
    heif_error_Decoder_plugin_error, heif_error_Encoder_plugin_error, heif_error_Unsupported_feature, heif_error_Memory_allocation_error,
    heif_error_Usage_error, heif_suberror_Security_limit_exceeded, heif_suberror_Unsupported_codec, heif_suberror_End_of_data,
    heif_suberror_Unsupported_bit_depth, heif_compression_HEVC, heif_colorspace_YCbCr, heif_colorspace_monochrome, heif_channel_Y,
    heif_channel_Cb, heif_channel_Cr, heif_chroma_420, heif_plugin_type_decoder, heif_plugin_type_encoder, (long)LIBHEIF_MAKE_VERSION(1, 21, 0)};
#else
#include "../../include/b200_heif_plugin_abi.h"
typedef b200h_error Error;
typedef b200h_decoder_plugin Decoder;
typedef b200h_encoder_plugin Encoder;
typedef b200h_encoder_parameter EncoderParameter;
typedef b200h_decoder_options DecoderOptions;
typedef b200h_security_limits SecurityLimits;
typedef b200h_plugin_info PluginInfo;
// the leading members of heif_color_profile_nclx the library reads
struct Nclx { uint8_t version; int color_primaries; int transfer_characteristics; int matrix_coefficients; uint8_t full_range_flag; };
// heif_chroma_420, the plugin types (b200h_plugin_info) and LIBHEIF_MAKE_VERSION(1, 21, 0) as the library uses them
static const long kConstants[] = {
    B200H_ERR_DECODER_PLUGIN, B200H_ERR_ENCODER_PLUGIN, B200H_ERR_UNSUPPORTED_FEATURE, B200H_ERR_MEMORY, B200H_ERR_USAGE,
    B200H_SUBERR_SECURITY_LIMIT, B200H_SUBERR_UNSUPPORTED_CODEC, B200H_SUBERR_END_OF_DATA, B200H_SUBERR_UNSUPPORTED_BIT_DEPTH,
    B200H_COMPRESSION_HEVC, B200H_COLORSPACE_YCBCR, B200H_COLORSPACE_MONOCHROME, B200H_CHANNEL_Y, B200H_CHANNEL_CB, B200H_CHANNEL_CR,
    1, 1, 0, (1L << 24) | (21L << 16)};
#endif

static const char* kConstantNames[] = {
    "error.decoder_plugin", "error.encoder_plugin", "error.unsupported_feature", "error.memory", "error.usage",
    "suberror.security_limit", "suberror.unsupported_codec", "suberror.end_of_data", "suberror.unsupported_bit_depth",
    "compression.hevc", "colorspace.ycbcr", "colorspace.monochrome", "channel.y", "channel.cb", "channel.cr",
    "chroma.420", "plugin_type.decoder", "plugin_type.encoder", "version(1,21,0)"};
static_assert(sizeof(kConstantNames) / sizeof(kConstantNames[0]) == sizeof(kConstants) / sizeof(kConstants[0]), "one name per constant");

#define SIZE(T) std::printf("sizeof %s %zu\n", #T, sizeof(T))
#define OFF(T, m) std::printf("offsetof %s.%s %zu\n", #T, #m, offsetof(T, m))

int main() {
  SIZE(Error); OFF(Error, message);
  SIZE(Decoder);
  OFF(Decoder, plugin_api_version); OFF(Decoder, get_plugin_name); OFF(Decoder, does_support_format); OFF(Decoder, new_decoder);
  OFF(Decoder, push_data); OFF(Decoder, decode_image); OFF(Decoder, set_strict_decoding); OFF(Decoder, id_name);
  OFF(Decoder, decode_next_image); OFF(Decoder, minimum_required_libheif_version); OFF(Decoder, does_support_format2);
  OFF(Decoder, new_decoder2); OFF(Decoder, push_data2); OFF(Decoder, flush_data); OFF(Decoder, decode_next_image2);
  SIZE(Encoder);
  OFF(Encoder, compression_format); OFF(Encoder, id_name); OFF(Encoder, priority); OFF(Encoder, supports_lossless_compression);
  OFF(Encoder, new_encoder); OFF(Encoder, list_parameters); OFF(Encoder, get_parameter_string); OFF(Encoder, query_input_colorspace);
  OFF(Encoder, encode_image); OFF(Encoder, get_compressed_data); OFF(Encoder, query_input_colorspace2); OFF(Encoder, query_encoded_size);
  OFF(Encoder, minimum_required_libheif_version); OFF(Encoder, start_sequence_encoding); OFF(Encoder, get_compressed_data2);
  OFF(Encoder, does_indicate_keyframes);
  SIZE(EncoderParameter); OFF(EncoderParameter, has_default);
  SIZE(DecoderOptions); OFF(DecoderOptions, limits);
  OFF(SecurityLimits, max_image_size_pixels);
  SIZE(PluginInfo);
  OFF(Nclx, matrix_coefficients); OFF(Nclx, full_range_flag);
  for (size_t i = 0; i < sizeof(kConstants) / sizeof(kConstants[0]); i++) std::printf("constant %s %ld\n", kConstantNames[i], kConstants[i]);
  return 0;
}
