# Stub declarations + loader for the CUDA tracing core shim, same convention as the reference's
# lib/fast_4d_matrix/fast_4d_matrix.rb (stubs first, then `require_relative '../<name>'` at :38).
module Rtrb
  class Renderer
    # method stubs
    def initialize(world); raise NotImplementedError; end
    def update(world); raise NotImplementedError; end
    def render(camera, seed = 1, precision = 1); raise NotImplementedError; end
    def render_png(camera, seed = 1, precision = 1); raise NotImplementedError; end
    def render_progressive(camera, schedule, seed = 1); raise NotImplementedError; end
    def render_progressive_png(camera, schedule, seed = 1); raise NotImplementedError; end
    def stats; raise NotImplementedError; end
    def trace_rays(packed_rays, trace_depth, mc, seed = 1); raise NotImplementedError; end
    def intersect_rays(packed_rays); raise NotImplementedError; end
  end
end

require_relative '../rtrb_b200'

# Frame-level drop-in for the reference's pixel loops.  `Camera#render_cuda(file_path)` replaces
# render_sync(file_path) (src/camera.rb:101-110) / render_fork(file_path, n) (:41-68): one call
# returns the finished 8-bit rows, which go through the existing canvas + save_image (:36-39).
module Alex
  class Camera
    # Edits of @world's objects and lights since the last frame reach this one (Renderer#update re-bakes them in place).
    def render_cuda(file_path, seed = 1)
      rtrb_renderer
      rgb = @rtrb.render(self, seed)           # H*W*3 bytes (RGB8), row = y, column = x
      @height.times do |y|
        @width.times do |x|
          r, g, b = rgb.getbyte((y * @width + x) * 3), rgb.getbyte((y * @width + x) * 3 + 1), rgb.getbyte((y * @width + x) * 3 + 2)
          # same canvas coordinates render_sync uses: render_at returns [x, H-1-y] (camera.rb:98,105)
          @canvas.point(x, @height - 1 - y, PNG::Color.new(r, g, b))
        end
      end
      save_image(file_path)
    end

    # save_image's file without the canvas: the GPU renders and encodes the PNG (8-bit RGB), only the file crosses PCIe
    def render_cuda_png(file_path, seed = 1)
      rtrb_renderer
      File.binwrite(file_path, @rtrb.render_png(self, seed))
    end

    # render_cuda_png in passes: the file is rewritten after every pass of `schedule` (increasing sample counts ending
    # at pre_sample_times; default 1, 2, 4, ... then pre_sample_times), each a preview of the samples traced so far
    def render_cuda_progressive(file_path, schedule = nil)
      rtrb_renderer
      schedule ||= progressive_schedule(@pre_sample_times)
      @rtrb.render_progressive_png(self, schedule) { |png, _samples_done| File.binwrite(file_path, png) }
    end

    private

    def progressive_schedule(pre)
      out = []
      e = 1
      while e < pre
        out << e
        e *= 2
      end
      out << pre
    end

    def rtrb_renderer
      if @rtrb
        @rtrb.update(@world)
      else
        @rtrb = Rtrb::Renderer.new(@world)
      end
    end
  end
end
