    const samplesPerPixel = b.option(usize, "samplesPerPixel", "samples per pixel to use") orelse 500;
    const fileName = b.option([]const u8, "fileName", "name of the file to save") orelse "chapter14.ppm";
    const seed = b.option(u64, "seed", "an optional random seed to use for determistic results") orelse null;
    
    const buildOptions = b.addOptions();
    buildOptions.addOption(usize, "imgWidth", imgWidth);
    buildOptions.addOption(usize, "samplesPerPixel", samplesPerPixel);
    buildOptions.addOption([]const u8, "fileName", fileName);
    buildOptions.addOption(?u64, "seed", seed);

    const exe = b.addExecutable(.{
        .name = "raytracing-with-zig",
// [...]
    });

    exe.root_module.addOptions("config", buildOptions);

    b.installArtifact(exe);

// [...]
    testOptions.addOption(usize, "samplesPerPixel", 10);
    testOptions.addOption([]const u8, "fileName", fileName);
    testOptions.addOption(?u64, "seed", 0xdeadbeef);

    exe_unit_tests.root_module.addOptions("config", testOptions);

    const run_exe_unit_tests = b.addRunArtifact(exe_unit_tests);

