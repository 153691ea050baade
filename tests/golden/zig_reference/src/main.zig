    try camera.render();
}

// Since we are passing in a seed for the test options, we have a deterministic 
// image being built.  We will compare the expected and actual image since the
// result will be the same every time.
test "main" {
    try std.testing.expect(config.imgWidth == 400);
    try std.testing.expect(config.samplesPerPixel == 10);
// [...]
    const actual = try std.fs.cwd().readFileAlloc(std.testing.allocator, "images/" ++ config.fileName, 5e5);
    defer std.testing.allocator.free(actual);

    try std.testing.expectEqualStrings(expected, actual);
}
