// rtrb_png.h — device PNG encoder (rtrb_png.cu) as the C ABI in rtrb_api.cu drives it.
//
// Pipeline (all on one stream, no host synchronisation):
//   png_filter_kernel   one CTA per row: the five PNG filters, keeps the smallest sum of |signed byte|
//   png_deflate_kernel  one CTA per RTRB_PNG_SEGMENT_BYTES of the filtered stream: LZ77 + one stored / fixed /
//                       dynamic Huffman block, sync flush, chunk CRC-32 and Adler-32 partial
//   png_assemble_kernel prefix sum over the segment sizes, signature, IHDR, zlib header, Adler-32 trailer, IEND
//   png_place_kernel    every segment's IDAT chunk at its offset
//   png_publish_kernel  (pipelined frames) the finished file into mapped host memory by device stores
//
// APNG frames (rtrb_apng_encode, DESIGN.md 15) put apng_diff_kernel in front: it keeps the frame as compact RGB8 and
// finds the bounding box of the pixels whose RGB changed since the previous frame.  The crop's filter and deflate
// (png_filter_kernel<true>, png_deflate_kernel<true>) and apng_place_kernel read its size from device memory and run
// on grids sized for the whole frame, so the host never waits for the rectangle; apng_assemble_kernel writes the fcTL
// chunk and the framing around the segments.
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

// One APNG frame: fcTL (12 + 26 bytes), then the PNG chunks of the stream, each fdAT chunk 4 bytes longer than an
// IDAT chunk for its sequence number.  The whole canvas is the largest crop.
inline size_t rtrb_apng_frame_bound(int width, int height) {
  const size_t n = rtrb_png_filtered_bytes(width, height), segs = rtrb_png_segments(width, height);
  return (12 + 26) + (14 + 4) + (16 + 4) + segs * (RTRB_PNG_CHUNK_BYTES + 4 + RTRB_PNG_SEGMENT_WORST(0)) + n;
}

// Device scratch of one renderer; grows with the largest frame encoded so far and is released with the renderer.
struct RtrbPngScratch {
  DevBuf<uint8_t> filtered;             // the filtered stream
  DevBuf<uint32_t> tokens;              // LZ77 tokens, RTRB_PNG_SEGMENT_BYTES slots per segment
  DevBuf<uint8_t> seg_out;              // each segment's deflate bytes, RTRB_PNG_SEGMENT_WORST(segment) apart
  DevBuf<uint32_t> seg_meta;            // per segment: bytes, chunk CRC-32 (of its fdAT chunk in an APNG crop),
                                        // Adler-32 of its input
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

// Device words of one animation.  box and ctas_done are apng_diff_kernel's running reduction and are reset by its last
// CTA; the rectangle and the sizes describe the frame being encoded.
struct RtrbApngState {
  int box[4];                // changed pixels so far: min x, min y, max x, max y (max x < 0: none)
  unsigned int ctas_done;    // CTAs of apng_diff_kernel that have merged their box
  int x0, y0, w, h;          // the frame's rectangle
  unsigned int nseg;         // segments of its filtered stream
  unsigned long long n_in;   // bytes of its filtered stream, h * (3 w + 1)
  unsigned int seq;          // sequence number of its fcTL chunk
  unsigned int next_seq;     // sequence number of the next frame's fcTL chunk
};

// Queues one APNG frame of a width x height animation: `src` (pixel_format) is compared with `prev` (the previous
// frame, compact RGB8; not read for the first frame) and stored compactly into `cur`, and the frame's fcTL and data
// chunks land in s.file, their byte count in s.total (and with host_mapped / count_mapped also there, as
// rtrb_png_encode).  `st` must start as { {INT_MAX, INT_MAX, -1, -1}, 0, ... 0 }.  Adds the kernel launches to *launches.
cudaError_t rtrb_apng_encode(RtrbPngScratch& s, RtrbApngState* st, const uint8_t* prev, uint8_t* cur, const uint8_t* src,
                             int width, int height, int pixel_format, bool first, int delay_num, int delay_den,
                             cudaStream_t stream, uint8_t* host_mapped, unsigned long long* count_mapped,
                             unsigned long long* launches);

#endif  // RTRB_PNG_H
