// rtrb_png.h — device PNG encoder (rtrb_png.cu) as the C ABI in rtrb_api.cu drives it.
//
// Pipeline (all on one stream, no host synchronisation):
//   png_filter_kernel   one CTA per row: the five PNG filters, keeps the smallest sum of |signed byte|
//   png_deflate_kernel  one CTA per RTRB_PNG_SEGMENT_BYTES of the filtered stream: LZ77 + one stored / fixed /
//                       dynamic Huffman block, sync flush, chunk CRC-32 and Adler-32 partial
//   png_assemble_kernel prefix sum over the segment sizes, signature, IHDR, zlib header, Adler-32 trailer, IEND
//   png_place_kernel    every segment's IDAT chunk at its offset
//   png_publish_kernel  (pipelined frames) the finished file into mapped host memory by device stores
#ifndef RTRB_PNG_H
#define RTRB_PNG_H

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/rtrb_b200.h"
#include "rtrb_devbuf.h"

// PNG framing around the segments: signature 8, IHDR chunk 25, IDAT with the 2-byte zlib header 14, IDAT with the
// 4-byte Adler-32 trailer 16, IEND 12.  Each segment is one IDAT chunk (12 bytes of length, type and CRC).
#define RTRB_PNG_FIXED_BYTES (8 + 25 + 14 + 16 + 12)
#define RTRB_PNG_CHUNK_BYTES 12
// Worst case of one segment of n input bytes: a stored block (5 header bytes) plus the 5-byte empty stored block
// of the sync flush.  The encoder never emits more, because it keeps the smallest of the three block types.
#define RTRB_PNG_SEGMENT_WORST(n) ((size_t)(n) + 10)

// Bytes of the filtered stream: one filter-type byte per row in front of the row's RGB8 pixels.
inline size_t rtrb_png_filtered_bytes(int width, int height) { return (size_t)height * ((size_t)width * 3 + 1); }
inline size_t rtrb_png_segments(int width, int height) {
  return (rtrb_png_filtered_bytes(width, height) + RTRB_PNG_SEGMENT_BYTES - 1) / RTRB_PNG_SEGMENT_BYTES;
}
inline size_t rtrb_png_bound(int width, int height) {
  const size_t n = rtrb_png_filtered_bytes(width, height), segs = rtrb_png_segments(width, height);
  return RTRB_PNG_FIXED_BYTES + segs * (RTRB_PNG_CHUNK_BYTES + RTRB_PNG_SEGMENT_WORST(0)) + n;
}

// Device scratch of one renderer; grows with the largest frame encoded so far and is released with the renderer.
struct RtrbPngScratch {
  DevBuf<uint8_t> filtered;             // the filtered stream
  DevBuf<uint32_t> tokens;              // LZ77 tokens, RTRB_PNG_SEGMENT_BYTES slots per segment
  DevBuf<uint8_t> seg_out;              // each segment's deflate bytes, RTRB_PNG_SEGMENT_WORST(segment) apart
  DevBuf<uint32_t> seg_meta;            // per segment: bytes, chunk CRC-32, Adler-32 of its input
  DevBuf<unsigned long long> seg_off;   // per segment: offset of its IDAT chunk in the file
  DevBuf<uint8_t> file;                 // the finished PNG file
  DevBuf<unsigned long long> total;     // its byte count
};

// Queues the encoder for a width x height image at `src` (RTRB_FMT_RGB8 / RGBA8 / PNG_RGB8) on `stream`.  The file
// lands in s.file and its size in s.total; with host_mapped / count_mapped (device aliases of mapped host memory)
// it is also stored there.  Adds the number of kernel launches to *launches.
cudaError_t rtrb_png_encode(RtrbPngScratch& s, const uint8_t* src, int width, int height, int pixel_format,
                            cudaStream_t stream, uint8_t* host_mapped, unsigned long long* count_mapped,
                            unsigned long long* launches);

#endif  // RTRB_PNG_H
