const std = @import("std");
const util = @import("util.zig");
const config = @import("config");

const Point3 = @import("vec.zig").Point3;
const Vec = @import("vec.zig").Vec;
// [...]
        self.scene.deinit();
    }

    pub fn render(self: Camera) !void {
        // Setup Image/PPM
        var ppm = PPM.init(self.alloc, self.image.width, self.image.height);
        defer ppm.deinit();

        for (0..ppm.height) |j| {
            std.log.info("\rScanlines remaining: {d} ", .{ppm.height - j});
            for (0..ppm.width) |i| {
                var pixelColor = black;
                // Anti-aliasing sampling
                for (0..self.samplesPerPixel) |_| {
                    const ray = self.getRay(i, j);
                    pixelColor += self.rayColor(ray);
                }
                const avgColor = Color.fromVec(Vec.mulScalar(pixelColor, self.pixelSamplesScale));
                ppm.pixels[i + j * ppm.width] = avgColor;
            }
        }
        std.log.info("\rDone.\n", .{});

        // Save the file
        try ppm.saveBinary("images/" ++ config.fileName);
    }

    /// Non-recursive method for attenuating and bouncing the ray
